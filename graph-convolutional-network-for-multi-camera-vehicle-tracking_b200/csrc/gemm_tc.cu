// tcgen05 3xTF32 "NT" GEMM for sm_100a:  C[M,N] = A[M,K] * B[N,K]^T (+ bias[N]),  fp32 in / fp32 out.
//
// fp32 accuracy on the tensor cores: every operand is pre-split into two TF32-representable planes
//   x = hi + lo,  hi = rna_tf32(x),  lo = rna_tf32(x - hi)
// and each k-slice issues three MMAs:  main += hi*hi ;  corr += lo*hi + hi*lo   (the dropped lo*lo term is ~2^-22
// relative).  The tensor core adds into its fp32 accumulator with truncation, a bias that grows with the number of
// accumulation steps and with |accumulator| (measured: mean error toward zero, linear in K).  Keeping the small
// correction products in their own TMEM accumulator, and (BN=128) alternating two main accumulators over the k-slices,
// cuts that bias 3x / 6x; the epilogue sums the accumulators in fp32 round-to-nearest.  Used for the Gram matrix of the edge features
// (inference.py:453-456) and the node-encoder Linear layers (models/mpn.py:117, models/mlp.py:14).
//
// Kernel anatomy (one 128 x BN output tile per CTA, 192 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor.2d of the four operand tiles (A_hi, A_lo, B_hi, B_lo), SWIZZLE_128B,
//               into a STAGES-deep shared-memory ring guarded by full/empty mbarriers
//   warp 1      TMEM allocation + MMA issuer: one lane issues tcgen05.mma.cta_group::1.kind::tf32 (M=128, N=BN, K=8),
//               tcgen05.commit releases ring slots and finally signals the accumulator
//   warps 2..5  epilogue: tcgen05.ld 32x32b of the fp32 accumulator (one TMEM lane = one output row per thread),
//               bias add, vectorised global stores with edge masking
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include <cmath>

#include "common.cuh"
#include "kernels.h"
#include "tcgen05.cuh"

namespace mpn {

constexpr int TC_BM = 128;
constexpr int TC_BK = 32;                    // 32 fp32 = 128 bytes = one SWIZZLE_128B row
constexpr int TC_UMMA_K = 8;                 // kind::tf32: 32 bytes of K per instruction
constexpr int TC_THREADS = 192;
// F16 variant ("3xFP16"): the operand planes are fp16 (x*s = hi + lo, s a power of two that puts max|x| at 2^14; 11 + 11
// significant bits = the 22 bits of the TF32 pair), a 128-byte row holds 64 elements and one instruction covers K = 16:
// the same three products at twice the tensor-pipe rate and half the operand bytes.  Byte geometry of the stages, of the
// descriptors and of the k-advance is identical to the TF32 variant.  The epilogue multiplies by *out_scale (= s_a^-1 s_b^-1).
constexpr int TC_BK_F16 = 64;

// K-major, SWIZZLE_128B shared-memory matrix descriptor (8-row x 128-byte atoms, 1024 bytes apart)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);          // start address            bits [0,14)
  d |= (uint64_t)1 << 16;                           // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                 // stride byte offset: next 8-row group
  d |= (uint64_t)1 << 46;                           // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                           // layout type: SWIZZLE_128B
  return d;
}

template <int BN>
struct TcCfg {
  static constexpr int STAGES = (BN == 256) ? 2 : 3;
  static constexpr int A_BYTES = TC_BM * TC_BK * 4;           // one plane of A per stage (16 KB)
  static constexpr int B_BYTES = BN * TC_BK * 4;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
  static constexpr int N_MAIN = (BN == 256) ? 1 : 2;          // main accumulators (alternating k-slices)
  static constexpr int TMEM_COLS = 512;                        // main(s) + correction accumulator, power of two
  static constexpr int CORR_COL = N_MAIN * BN;
  static constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
  static constexpr uint32_t IDESC_F16 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);   // a/b format 0 = F16
};

// SYM: C = A A^T (A == B, M == N): only tiles on or above the diagonal are computed, the epilogue also writes the mirror.
// run_flag (optional, device): the grid returns at once when *run_flag == 0.
template <int BN, bool SYM, bool F16>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_nt_3xtf32_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                      const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                      const float* __restrict__ bias, float* __restrict__ C, int M, int N, int K,
                      const int* __restrict__ graph_nptr, const long long* __restrict__ g_off,
                      const float* __restrict__ out_scale, const int* __restrict__ run_flag) {
  pdl_wait();
  if (run_flag != nullptr && *run_flag == 0) return;
  constexpr int BK = F16 ? TC_BK_F16 : TC_BK;            // elements of K per stage (128 bytes either way)
  using Cfg = TcCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + Cfg::STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + Cfg::STAGES;
  uint64_t* tmem_full_bar = empty_bar + Cfg::STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int m0 = blockIdx.y * TC_BM, n0 = blockIdx.x * BN;     // output-local tile origin
  int tm0 = m0, tn0 = n0;                                // TMA row coordinates of the A / B tiles
  const int num_kb = (K + BK - 1) / BK;
  if (SYM && n0 + BN <= m0) return;                      // strictly below the diagonal: produced by the mirror store
  if (graph_nptr != nullptr) {
    // block-diagonal Gram (batched graphs): blockIdx.z = graph; its rows [base, base+ng) form an ng x ng block of C
    const int base = graph_nptr[blockIdx.z];
    const int ng = graph_nptr[blockIdx.z + 1] - base;
    if (m0 >= ng || n0 >= ng) return;
    tm0 = base + m0;
    tn0 = base + n0;
    M = N = ng;
    C += g_off[blockIdx.z];
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // TMEM: BN fp32 accumulator columns (power of two >= 32)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(Cfg::TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_hi));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_lo));
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* st = smem + stage * Cfg::STAGE_BYTES;
        mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
        const int k0 = kb * BK;
        tma_load_2d(&map_a_hi, &full_bar[stage], st, k0, tm0);
        tma_load_2d(&map_a_lo, &full_bar[stage], st + Cfg::A_BYTES, k0, tm0);
        tma_load_2d(&map_b_hi, &full_bar[stage], st + 2 * Cfg::A_BYTES, k0, tn0);
        tma_load_2d(&map_b_lo, &full_bar[stage], st + 2 * Cfg::A_BYTES + Cfg::B_BYTES, k0, tn0);
        if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sbase = smem_u32(smem + stage * Cfg::STAGE_BYTES);
        const uint64_t a_hi = make_smem_desc(sbase), a_lo = make_smem_desc(sbase + Cfg::A_BYTES);
        const uint64_t b_hi = make_smem_desc(sbase + 2 * Cfg::A_BYTES), b_lo = make_smem_desc(sbase + 2 * Cfg::A_BYTES + Cfg::B_BYTES);
#pragma unroll
        for (int kk = 0; kk < TC_BK / TC_UMMA_K; ++kk) {
          const uint64_t adv = (uint64_t)((kk * TC_UMMA_K * 4) >> 4);        // 32 bytes of K per instruction (8 tf32 / 16 fp16)
          const int slice = kb * (TC_BK / TC_UMMA_K) + kk;
          const int which = (Cfg::N_MAIN == 2) ? (slice & 1) : 0;
          if (F16) {
            umma_f16(tmem_base + which * BN, a_hi + adv, b_hi + adv, Cfg::IDESC_F16, slice >= Cfg::N_MAIN);
            umma_f16(tmem_base + Cfg::CORR_COL, a_lo + adv, b_hi + adv, Cfg::IDESC_F16, slice != 0);
            umma_f16(tmem_base + Cfg::CORR_COL, a_hi + adv, b_lo + adv, Cfg::IDESC_F16, 1);
          } else {
            umma_tf32(tmem_base + which * BN, a_hi + adv, b_hi + adv, Cfg::IDESC, slice >= Cfg::N_MAIN);
            umma_tf32(tmem_base + Cfg::CORR_COL, a_lo + adv, b_hi + adv, Cfg::IDESC, slice != 0);
            umma_tf32(tmem_base + Cfg::CORR_COL, a_hi + adv, b_lo + adv, Cfg::IDESC, 1);
          }
        }
        umma_commit(&empty_bar[stage]);                                         // slot free once these MMAs retire
        if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
      }
      umma_commit(tmem_full_bar);                                               // accumulator complete
    }
  } else {
    // ===== epilogue (warps 2..5): TMEM lane quarter = warp % 4 =====
    mbar_wait(tmem_full_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int q = warp & 3;
    const int row = m0 + q * 32 + lane;
    const bool vec_ok = ((N & 3) == 0) && ((((uintptr_t)C) & 15) == 0);
    const float oscale = (F16 && out_scale) ? *out_scale : 1.f;       // power of two: exact
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (n0 + c0 >= N) break;                                                  // warp-uniform
      float v[32], w[32];
      const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
      tmem_ld32(tq, v);
      if (Cfg::N_MAIN == 2) {
        tmem_ld32(tq + BN, w);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += w[j];
      }
      tmem_ld32(tq + Cfg::CORR_COL, w);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = F16 ? (v[j] + w[j]) * oscale : v[j] + w[j];
      if (row < M) {
        float* out = C + (size_t)row * N + n0 + c0;
        if (vec_ok && n0 + c0 + 32 <= N) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 o = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            if (bias) {
              const float4 b = *reinterpret_cast<const float4*>(bias + n0 + c0 + j);
              o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
            }
            *reinterpret_cast<float4*>(out + j) = o;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (n0 + c0 + j < N) out[j] = v[j] + (bias ? bias[n0 + c0 + j] : 0.f);
        }
      }
      if (SYM && row < M) {                               // mirror: C[col][row]; lanes hold consecutive rows -> coalesced
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int col = n0 + c0 + j;
          if (col < N && col >= m0 + TC_BM) C[(size_t)col * N + row] = v[j];
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS));
  }
}

// x -> (hi, lo) TF32 planes.  Optional fused input transform f(x)[m,k] = relu(x*scale[k] + shift[k]): the BatchNorm+ReLU of
// the previous encoder layer (models/mlp.py:14-19), so the activation is never re-written in fp32.
template <typename T>
__global__ void __launch_bounds__(256) split_tf32_kernel(const T* __restrict__ x, long long n4, int K, const float* __restrict__ scale,
                                                         const float* __restrict__ shift, const int* __restrict__ row_gid,
                                                         float4* __restrict__ hi, float4* __restrict__ lo) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = ld4(x, i);
    float in[4] = {v.x, v.y, v.z, v.w};
    if (scale != nullptr) {
      const int k = (int)((i * 4) % K);                 // K % 4 == 0: the four lanes stay inside one row
      const size_t o = (row_gid ? (size_t)row_gid[(i * 4) / K] * K : 0) + k;          // per-graph BatchNorm (batched graphs)
      const float4 sc = *reinterpret_cast<const float4*>(scale + o), sh = *reinterpret_cast<const float4*>(shift + o);
      in[0] = fmaxf(fmaf(in[0], sc.x, sh.x), 0.f);
      in[1] = fmaxf(fmaf(in[1], sc.y, sh.y), 0.f);
      in[2] = fmaxf(fmaf(in[2], sc.z, sh.z), 0.f);
      in[3] = fmaxf(fmaf(in[3], sc.w, sh.w), 0.f);
    }
    float h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t hb, lb;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(in[j]));
      h[j] = __uint_as_float(hb);
      const float r = in[j] - h[j];
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(r));
      l[j] = __uint_as_float(lb);
    }
    hi[i] = make_float4(h[0], h[1], h[2], h[3]);
    lo[i] = make_float4(l[0], l[1], l[2], l[3]);
  }
}

// x*s -> (hi, lo) fp16 planes, s = 2^(14 - ceil(log2(amax))) read from the device (amax = max |x|, float bits, made by the
// producer of x); also publishes out_scale = s^-2 for the epilogue of a Gram GEMM (both operands share the planes).
__device__ __forceinline__ float f16_scale_of(float amax) {
  if (!(amax > 0.f) || !isfinite(amax)) return 1.f;
  int e;
  frexpf(amax, &e);                                     // amax = m * 2^e, m in [0.5, 1)  ->  amax * 2^(14-e) in [2^13, 2^14)
  return ldexpf(1.f, 14 - e);
}
__global__ void __launch_bounds__(256) split_f16_kernel(const float4* __restrict__ x, long long n4, const float* __restrict__ amax,
                                                        uint2* __restrict__ hi, uint2* __restrict__ lo, float* __restrict__ out_scale,
                                                        const int* __restrict__ run_flag) {
  pdl_wait();
  if (run_flag != nullptr && *run_flag == 0) return;
  const float s = f16_scale_of(*amax);
  if (out_scale && blockIdx.x == 0 && threadIdx.x == 0) *out_scale = (1.f / s) * (1.f / s);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = x[i];
    const float in[4] = {v.x * s, v.y * s, v.z * s, v.w * s};
    __half h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      h[j] = __float2half_rn(in[j]);
      l[j] = __float2half_rn(in[j] - __half2float(h[j]));
    }
    uint2 ph, pl;
    ph.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
    ph.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
    pl.x = (uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16);
    pl.y = (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16);
    hi[i] = ph;
    lo[i] = pl;
  }
}

// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

int make_tma_map_2d(CUtensorMap* map, const void* base, int rows, int K, int box_rows, bool f16) {
  EncodeTiledFn enc = get_encode_fn();
  MPN_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * (f16 ? sizeof(__half) : sizeof(float))};
  cuuint32_t box[2] = {(cuuint32_t)(f16 ? TC_BK_F16 : TC_BK), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MPN_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%d K=%d)", (int)r, rows, K);
  return MPN_OK;
}

int split_tf32(const float* x, long long n, float* hi, float* lo, cudaStream_t st) {
  MPN_REQUIRE(x && hi && lo && n > 0 && (n % 4) == 0, "split_tf32: bad arguments (n must be a positive multiple of 4)");
  MPN_REQUIRE((((uintptr_t)x | (uintptr_t)hi | (uintptr_t)lo) & 15) == 0, "split_tf32: pointers must be 16-byte aligned");
  mpn::launch(split_tf32_kernel<float>, (int)min((long long)kNumSMs * 8, (n / 4 + 255) / 256), 256, 0, st, x, n / 4, 4, nullptr, nullptr, nullptr, (float4*)hi, (float4*)lo);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

bool gemm_tc_supported(int M, int N, int K) { return M >= 1 && N >= 64 && K >= 64 && (K % 4) == 0; }

size_t gemm_tc_workspace_bytes(int M, int N, int K) {
  if (!gemm_tc_supported(M, N, K)) return 0;
  const size_t plane_a = (((size_t)M * K * sizeof(float)) + 255) & ~(size_t)255;
  const size_t plane_b = (((size_t)N * K * sizeof(float)) + 255) & ~(size_t)255;
  return 2 * plane_a + 2 * plane_b + 1024;
}

template <int BN, bool SYM, bool F16 = false>
static int launch_tc(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl, const float* bias,
                     float* C, int M, int N, int K, cudaStream_t st, const int* graph_nptr = nullptr, const long long* g_off = nullptr,
                     int n_graphs = 1, int max_ng = 0, const float* out_scale = nullptr, const int* run_flag = nullptr) {
  static bool configured = false;
  if (!configured) {
    MPN_CUDA_OK(cudaFuncSetAttribute(gemm_nt_3xtf32_kernel<BN, SYM, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<BN>::SMEM_BYTES));
    configured = true;
  }
  dim3 grid(div_up(N, BN), div_up(M, TC_BM));
  if (graph_nptr) grid = dim3(div_up(max_ng, BN), div_up(max_ng, TC_BM), n_graphs);
  mpn::launch(gemm_nt_3xtf32_kernel<BN, SYM, F16>, grid, TC_THREADS, TcCfg<BN>::SMEM_BYTES, st, ah, al, bh, bl, bias, C, M, N, K, graph_nptr, g_off, out_scale, run_flag);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int gemm_nt_tc(const void* A, const float* B, const float* bias, float* C, int M, int N, int K, void* ws, size_t ws_bytes,
               cudaStream_t st, const float* a_scale, const float* a_shift, const float* b_hi_cached, const float* b_lo_cached,
               const int* row_gid, int a_kind) {
  MPN_REQUIRE(gemm_tc_supported(M, N, K), "tcgen05 GEMM: unsupported shape %d x %d x %d", M, N, K);
  MPN_REQUIRE(ws && ws_bytes >= gemm_tc_workspace_bytes(M, N, K), "tcgen05 GEMM: workspace too small");
  MPN_REQUIRE((((uintptr_t)B) & 15) == 0 && x_vec4_aligned(A, a_kind), "tcgen05 GEMM: operands must be aligned to four elements");
  char* w = (char*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
  const size_t plane_b = (((size_t)N * K * sizeof(float)) + 255) & ~(size_t)255;
  const size_t plane_a = (((size_t)M * K * sizeof(float)) + 255) & ~(size_t)255;
  float* b_hi = (float*)w;
  float* b_lo = (float*)(w + plane_b);
  float *a_hi, *a_lo;
  const int split_grid = kNumSMs * 8;
  if (b_hi_cached && b_lo_cached) {                  // weights: planes made once by mpn_split_tf32
    b_hi = (float*)b_hi_cached;
    b_lo = (float*)b_lo_cached;
  } else {
    mpn::launch(split_tf32_kernel<float>, split_grid, 256, 0, st, B, (long long)N * K / 4, K, nullptr, nullptr, nullptr, (float4*)b_hi, (float4*)b_lo);
    MPN_LAUNCH_OK();
  }
  const float* Af = (const float*)A;
  if (a_kind == MPN_X_F32 && a_scale == nullptr && Af >= B && Af + (size_t)M * K <= B + (size_t)N * K) {   // A is a row block of B (Gram matrix): share the planes
    a_hi = b_hi + (Af - B);
    a_lo = b_lo + (Af - B);
  } else {
    a_hi = (float*)(w + 2 * plane_b);
    a_lo = (float*)(w + 2 * plane_b + plane_a);
    MPN_TRY(with_x_type(a_kind, [&](auto at) {
      mpn::launch(split_tf32_kernel<x_elem_t<decltype(at)>>, split_grid, 256, 0, st, (decltype(at))A, (long long)M * K / 4, K, a_scale, a_shift, row_gid,
                  (float4*)a_hi, (float4*)a_lo);
      MPN_LAUNCH_OK();
      return MPN_OK;
    }));
  }
  CUtensorMap ah, al, bh, bl;
  static int forced_bn = -1;                         // diagnostics: MPN_TC_BN=128|256 overrides the tile width
  if (forced_bn < 0) {
    const char* e = getenv("MPN_TC_BN");
    forced_bn = e ? atoi(e) : 0;
  }
  // 128-wide tiles measured both faster (3 stages, more tiles per wave) and more accurate (three accumulators) than 256
  const int BN = (forced_bn == 128 || forced_bn == 256) ? forced_bn : 128;
  MPN_TRY(make_tma_map_2d(&ah, a_hi, M, K, TC_BM, false));
  MPN_TRY(make_tma_map_2d(&al, a_lo, M, K, TC_BM, false));
  MPN_TRY(make_tma_map_2d(&bh, b_hi, N, K, BN, false));
  MPN_TRY(make_tma_map_2d(&bl, b_lo, N, K, BN, false));
  const bool sym = (Af == B) && (M == N) && bias == nullptr;    // Gram matrix: half the tiles
  if (BN == 256) return launch_tc<256, false>(ah, al, bh, bl, bias, C, M, N, K, st);
  if (sym) return launch_tc<128, true>(ah, al, bh, bl, bias, C, M, N, K, st);
  return launch_tc<128, false>(ah, al, bh, bl, bias, C, M, N, K, st);
}

// fp16 operand planes with the fused input transform f(x)[m,k] = relu(x*scale[k] + shift[k]) of the previous encoder layer.
// The plane scale comes from *amax_dev (float bits, device) when given, else from amax_host; out_scale = 1 / (s_a * b_scale).
template <typename T>
__global__ void __launch_bounds__(256) split_f16_bn_kernel(const T* __restrict__ x, long long n4, int K, const float* __restrict__ scale,
                                                           const float* __restrict__ shift, const int* __restrict__ row_gid,
                                                           const float* __restrict__ amax_dev, float amax_host, float b_scale,
                                                           uint2* __restrict__ hi, uint2* __restrict__ lo, float* __restrict__ out_scale) {
  pdl_wait();
  const float s = f16_scale_of(amax_dev ? *amax_dev : amax_host);
  if (out_scale && blockIdx.x == 0 && threadIdx.x == 0) *out_scale = (1.f / s) * (1.f / b_scale);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = ld4(x, i);
    float in[4] = {v.x, v.y, v.z, v.w};
    if (scale != nullptr) {
      const int k = (int)((i * 4) % K);
      const size_t o = (row_gid ? (size_t)row_gid[(i * 4) / K] * K : 0) + k;
      const float4 sc = *reinterpret_cast<const float4*>(scale + o), sh = *reinterpret_cast<const float4*>(shift + o);
      in[0] = fmaxf(fmaf(in[0], sc.x, sh.x), 0.f);
      in[1] = fmaxf(fmaf(in[1], sc.y, sh.y), 0.f);
      in[2] = fmaxf(fmaf(in[2], sc.z, sh.z), 0.f);
      in[3] = fmaxf(fmaf(in[3], sc.w, sh.w), 0.f);
    }
    __half h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float t = fminf(in[j] * s, 65000.f);        // (the activation bound is mathematical: the clamp never binds)
      h[j] = __float2half_rn(t);
      l[j] = __float2half_rn(t - __half2float(h[j]));
    }
    uint2 ph, pl;
    ph.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
    ph.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
    pl.x = (uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16);
    pl.y = (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16);
    hi[i] = ph;
    lo[i] = pl;
  }
}
template <typename T>
__global__ void __launch_bounds__(256) absmax_kernel(const T* __restrict__ x, long long n4, unsigned int* __restrict__ amax_bits) {
  pdl_wait();
  float m = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = ld4(x, i);
    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(amax_bits, __float_as_uint(m));
}

float f16_plane_scale_host(float amax) {
  if (!(amax > 0.f) || !std::isfinite(amax)) return 1.f;
  int e;
  frexpf(amax, &e);
  return ldexpf(1.f, 14 - e);
}

// weights -> cached fp16 planes (host-known amax); returns the power-of-two scale that was applied
int split_f16_host_scale(const float* x, long long n, float amax, void* hi, void* lo, float* scale_out, cudaStream_t st) {
  MPN_REQUIRE(x && hi && lo && n > 0 && (n % 4) == 0, "split_f16: bad arguments (n must be a positive multiple of 4)");
  MPN_REQUIRE((((uintptr_t)x | (uintptr_t)hi | (uintptr_t)lo) & 15) == 0, "split_f16: pointers must be 16-byte aligned");
  mpn::launch(split_f16_bn_kernel<float>, (int)min((long long)kNumSMs * 8, (n / 4 + 255) / 256), 256, 0, st, x, n / 4, 4, nullptr, nullptr, nullptr,
                                                                                           nullptr, amax, 1.f, (uint2*)hi, (uint2*)lo, nullptr);
  MPN_LAUNCH_OK();
  if (scale_out) *scale_out = f16_plane_scale_host(amax);
  return MPN_OK;
}

// C = f(A) B^T + bias on 3xFP16 planes: A split here (fused BatchNorm+ReLU of the previous layer), B planes cached.
// a_amax_dev == nullptr && a_amax_host <= 0: max |A| is measured first (one pass over A; layer 0).
int gemm_nt_tc_f16(const void* A, const float* bias, float* C, int M, int N, int K, void* ws, size_t ws_bytes, cudaStream_t st,
                   const float* a_scale, const float* a_shift, const int* row_gid, float a_amax_host, const void* b_hi16,
                   const void* b_lo16, float b_scale, int a_kind) {
  MPN_REQUIRE(gemm_tc_supported(M, N, K) && (K % 8) == 0, "tcgen05 fp16-plane GEMM: unsupported shape %d x %d x %d", M, N, K);
  MPN_REQUIRE(ws && ws_bytes >= gemm_tc_workspace_bytes(M, N, K), "tcgen05 GEMM: workspace too small");
  MPN_REQUIRE(b_hi16 && b_lo16 && b_scale > 0.f, "tcgen05 fp16-plane GEMM: missing weight planes");
  MPN_REQUIRE(x_vec4_aligned(A, a_kind), "tcgen05 fp16-plane GEMM: A must be aligned to four elements");
  char* w = (char*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
  const size_t plane = (((size_t)M * K * sizeof(__half)) + 255) & ~(size_t)255;
  __half* a_hi = (__half*)w;
  __half* a_lo = (__half*)(w + plane);
  float* out_scale = (float*)(w + 2 * plane);
  unsigned int* amax_bits = (unsigned int*)(w + 2 * plane + 256);
  const float* amax_dev = nullptr;
  if (!(a_amax_host > 0.f)) MPN_CUDA_OK(cudaMemsetAsync(amax_bits, 0, sizeof(unsigned int), st));
  MPN_TRY(with_x_type(a_kind, [&](auto at) {
    using T = x_elem_t<decltype(at)>;
    if (!(a_amax_host > 0.f)) {
      mpn::launch(absmax_kernel<T>, kNumSMs * 8, 256, 0, st, (const T*)A, (long long)M * K / 4, amax_bits);
      MPN_LAUNCH_OK();
      amax_dev = (const float*)amax_bits;
    }
    mpn::launch(split_f16_bn_kernel<T>, kNumSMs * 8, 256, 0, st, (const T*)A, (long long)M * K / 4, K, a_scale, a_shift, row_gid, amax_dev,
                a_amax_host, b_scale, (uint2*)a_hi, (uint2*)a_lo, out_scale);
    MPN_LAUNCH_OK();
    return MPN_OK;
  }));
  CUtensorMap ah, al, bh, bl;
  MPN_TRY(make_tma_map_2d(&ah, a_hi, M, K, TC_BM, true));
  MPN_TRY(make_tma_map_2d(&al, a_lo, M, K, TC_BM, true));
  MPN_TRY(make_tma_map_2d(&bh, b_hi16, N, K, 128, true));
  MPN_TRY(make_tma_map_2d(&bl, b_lo16, N, K, 128, true));
  return launch_tc<128, false, true>(ah, al, bh, bl, bias, C, M, N, K, st, nullptr, nullptr, 1, 0, out_scale);
}

static bool gram_f16_enabled() {
  static int opt = -1;                               // MPN_GRAM_F16=0 keeps the TF32 planes (diagnostics)
  if (opt < 0) { const char* e = getenv("MPN_GRAM_F16"); opt = e ? atoi(e) : 1; }
  return opt != 0;
}

// Gram block C[M,N] = A X^T where A is the row block of X starting at row a_row0 (X: [N,K], amax_dev = max |X| as float bits
// written by the producer of X).  fp16 planes (3xFP16) when K % 8 == 0, else the TF32 path.  Symmetric tiles when A == X.
int gram_nt_tc(const float* X, int a_row0, float* C, int M, int N, int K, const float* amax_dev, void* ws, size_t ws_bytes, cudaStream_t st,
               const int* run_flag) {
  const float* A = X + (size_t)a_row0 * K;
  if (!gram_f16_enabled() || amax_dev == nullptr || (K % 8) != 0) {
    MPN_REQUIRE(run_flag == nullptr, "tcgen05 Gram: the TF32 planes have no conditional launch");
    return gemm_nt_tc(A, X, nullptr, C, M, N, K, ws, ws_bytes, st);
  }
  MPN_REQUIRE(gemm_tc_supported(M, N, K), "tcgen05 Gram: unsupported shape %d x %d x %d", M, N, K);
  MPN_REQUIRE(ws && ws_bytes >= gemm_tc_workspace_bytes(M, N, K), "tcgen05 Gram: workspace too small");
  char* w = (char*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
  const size_t plane = (((size_t)N * K * sizeof(__half)) + 255) & ~(size_t)255;
  __half* hi = (__half*)w;
  __half* lo = (__half*)(w + plane);
  float* out_scale = (float*)(w + 2 * plane);
  mpn::launch(split_f16_kernel, kNumSMs * 8, 256, 0, st, (const float4*)X, (long long)N * K / 4, amax_dev, (uint2*)hi, (uint2*)lo, out_scale, run_flag);
  MPN_LAUNCH_OK();
  CUtensorMap ah, al, bh, bl;
  MPN_TRY(make_tma_map_2d(&ah, hi + (size_t)a_row0 * K, M, K, TC_BM, true));
  MPN_TRY(make_tma_map_2d(&al, lo + (size_t)a_row0 * K, M, K, TC_BM, true));
  MPN_TRY(make_tma_map_2d(&bh, hi, N, K, 128, true));
  MPN_TRY(make_tma_map_2d(&bl, lo, N, K, 128, true));
  if (a_row0 == 0 && M == N) return launch_tc<128, true, true>(ah, al, bh, bl, nullptr, C, M, N, K, st, nullptr, nullptr, 1, 0, out_scale, run_flag);
  return launch_tc<128, false, true>(ah, al, bh, bl, nullptr, C, M, N, K, st, nullptr, nullptr, 1, 0, out_scale, run_flag);
}

// Block-diagonal Gram matrix of a batch of graphs: for graph i with rows [nptr[i], nptr[i+1]) the ng x ng block
// X_i X_i^T is written (row-major, ld = ng) at Gbuf + g_off[i].  Symmetric tiles only.
int gram_blockdiag_tc(const float* X, int N, int K, const int* graph_nptr, const long long* g_off, int n_graphs, int max_ng,
                      float* Gbuf, void* ws, size_t ws_bytes, cudaStream_t st, const float* amax_dev) {
  MPN_REQUIRE(gemm_tc_supported(N, 64, K), "block-diagonal tcgen05 Gram: unsupported K=%d", K);
  MPN_REQUIRE(n_graphs >= 1 && n_graphs <= 65535, "block-diagonal Gram: at most 65535 graphs per launch");
  const size_t plane = (((size_t)N * K * sizeof(float)) + 255) & ~(size_t)255;
  MPN_REQUIRE(ws && ws_bytes >= 2 * plane + 256, "block-diagonal Gram: workspace too small");
  char* w = (char*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
  if (gram_f16_enabled() && amax_dev != nullptr && (K % 8) == 0) {     // 3xFP16 planes (see gram_nt_tc)
    const size_t plane16 = (((size_t)N * K * sizeof(__half)) + 255) & ~(size_t)255;
    __half *hi16 = (__half*)w, *lo16 = (__half*)(w + plane16);
    float* out_scale = (float*)(w + 2 * plane16);
    mpn::launch(split_f16_kernel, kNumSMs * 8, 256, 0, st, (const float4*)X, (long long)N * K / 4, amax_dev, (uint2*)hi16, (uint2*)lo16, out_scale, (const int*)nullptr);
    MPN_LAUNCH_OK();
    CUtensorMap mh16, ml16;
    MPN_TRY(make_tma_map_2d(&mh16, hi16, N, K, TC_BM, true));
    MPN_TRY(make_tma_map_2d(&ml16, lo16, N, K, TC_BM, true));
    return launch_tc<128, true, true>(mh16, ml16, mh16, ml16, nullptr, Gbuf, N, N, K, st, graph_nptr, g_off, n_graphs, max_ng, out_scale);
  }
  float *hi = (float*)w, *lo = (float*)(w + plane);
  mpn::launch(split_tf32_kernel<float>, kNumSMs * 8, 256, 0, st, X, (long long)N * K / 4, K, nullptr, nullptr, nullptr, (float4*)hi, (float4*)lo);
  MPN_LAUNCH_OK();
  CUtensorMap mh, ml;
  MPN_TRY(make_tma_map_2d(&mh, hi, N, K, TC_BM, false));
  MPN_TRY(make_tma_map_2d(&ml, lo, N, K, TC_BM, false));
  return launch_tc<128, true>(mh, ml, mh, ml, nullptr, Gbuf, N, N, K, st, graph_nptr, g_off, n_graphs, max_ng);
}

}  // namespace mpn
