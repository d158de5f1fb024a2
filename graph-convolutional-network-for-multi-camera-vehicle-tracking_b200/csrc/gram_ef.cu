// K1 for dense cross-camera graphs: the edge features (inference.py:453-456) formed in the epilogue of the Gram GEMM.
//
//   edge_attr[e] = [ ||x_r - x_c + 1e-6||_2 , 1 - cos(x_r, x_c) ]
//
// Every row of such a graph lists all nodes but one contiguous gap (the node's own camera, inference.py:407-413), so the edge id
// of the ordered pair (i, j) is closed-form:  e = rowptr[i] + j - (j past the gap ? gap length : 0).  The accumulator tile goes
// TMEM -> registers -> distance / cosine -> edge_attr; no Gram matrix in HBM, no gather pass, and the five moment sums of the
// first encoder BatchNorm (sum a, b, aa, ab, bb over all edges; models/mlp.py:16 on encoder.edge_mlp.fc_layers.1) are taken on
// the way, which deletes one sweep over edge_attr from the forward.
//
// Kernel anatomy (persistent, one CTA per SM, 192 threads; tiles = the 128 x 128 blocks of the Gram matrix that hold edges, the
// upper triangle only when the row block is the whole graph):
//   warp 0      TMA producer: the four fp16 operand planes (A_hi, A_lo, B_hi, B_lo) of a k-block, SWIZZLE_128B, 3-stage ring;
//               it runs ahead into the next tile while the epilogue of the current one drains
//   warp 1      MMA issuer: tcgen05.mma.kind::f16 M=128 N=128 K=16, three products per k-slice (hi.hi | lo.hi + hi.lo) into two
//               alternating main accumulators and one correction accumulator (the tensor core truncates on accumulate: DESIGN.md)
//   warps 2..5  epilogue: thread = TMEM lane = row i.  Per 32-column chunk: three tcgen05.ld, then per column j
//                 g  = acc * 2^-(k_i + k_j)                      (per-row power-of-two plane scales: exact)
//                 d2 = |a'|^2 + |b'|^2 - 2 g  +- 2 eps (sum a' - sum b') + D eps^2        (centred rows a' = a - mean)
//                 cos = (g + mu.a' + mu.b' + |mu|^2) / (|a| |b|)
//               The mirrored entry (j -> i) of an off-diagonal tile is coalesced as it is (the lanes of a warp are consecutive
//               i = consecutive edges of row j); the direct entry (i -> j) goes through a padded shared-memory transpose so that
//               a warp writes 32 consecutive edges of one row.  Pairs whose d2 cancels (< 25 % of |a'|^2 + |b'|^2) are listed
//               and recomputed from the rows by edge_feature_refine (edge_features.cu), exactly as the reference sums them.
#include <cuda.h>
#include <cuda_fp16.h>

#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.h"
#include "tcgen05.cuh"

namespace mpn {

constexpr int GE_BM = 128, GE_BN = 128, GE_BK = 64;         // fp16: 64 elements = one 128-byte swizzle row
constexpr int GE_STAGES = 3;
constexpr int GE_PLANE_BYTES = GE_BM * GE_BK * 2;           // 16 KB
constexpr int GE_STAGE_BYTES = 4 * GE_PLANE_BYTES;          // 64 KB
constexpr int GE_EPI_WARPS = 8;                             // two per TMEM lane quarter (each takes half of the columns)
constexpr int GE_THREADS = 64 + 32 * GE_EPI_WARPS;
constexpr int GE_TMEM_COLS = 512;                           // two accumulator sets [hh | corr] (128 columns each), one per tile in flight
constexpr int GE_SUB = 8;                                   // columns per shared-memory transpose step
constexpr int GE_TPITCH = GE_SUB + 1;                       // float2 per row of the 32 x 8 transpose buffer (+1: conflict-free writes)
constexpr uint32_t GE_IDESC_N256 = (1u << 4) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(GE_BM >> 4) << 24);   // f16 x f16 -> f32
constexpr uint32_t GE_IDESC_N128 = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(GE_BM >> 4) << 24);

struct GeSmem {
  uint64_t full_bar[GE_STAGES], empty_bar[GE_STAGES], tmem_full_bar[2], tmem_empty_bar[2];
  uint32_t tmem_slot, pad;
  // per column j of the current tile: {|b'|^2, 2 eps sum b', mu.b' + |mu|^2/2, 1/|b|} and {2^-k_b (float bits), and the column's own
  // row of the graph for the mirrored entries: edge base before the gap, edge base after the gap, end of the gap} (base < 0: none)
  float4 cs_a[GE_BN];
  int4 cs_b[GE_BN];
  int4 rowinfo[GE_BM];                                       // rows of the tile: (edge base before the gap, after the gap, gap end, valid)
  // shared Gram (GeShare): edge_attr of the column's owner, and the rows [lo, hi) (global ids) whose pair with the column is this rank's
  float2* cs_ptr[GE_BN];
  int2 cs_lohi[GE_BN];
  float2 tbuf[GE_EPI_WARPS][32][GE_TPITCH];
};
constexpr int GE_SMEM_BYTES = GE_STAGES * GE_STAGE_BYTES + 1024 + (int)sizeof(GeSmem);
static_assert(GE_SMEM_BYTES <= 232448, "shared memory budget of one CTA");

__device__ __forceinline__ uint64_t ge_smem_desc(uint32_t saddr) {     // K-major, SWIZZLE_128B, 8-row atoms 1024 B apart
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ---- pre-pass 1: column means of x [n, D] in fp64.  grid (128-column tiles, row splits): a warp reads 512 contiguous bytes of a
// row per step; block partials go to part[split][col]; the last row split of a column tile to finish adds that tile's partials in
// a fixed order (one ticket counter per column tile).
constexpr int GE_CM_SPLITS = 37;                             // 16 column tiles x 37 row splits = 592 blocks at D = 2048
template <typename T>
__global__ void __launch_bounds__(256) ge_col_mean_kernel(const T* __restrict__ x, int n, int D, int rows_per_split,
                                                          double* __restrict__ part, unsigned int* __restrict__ ticket,
                                                          float* __restrict__ mu) {
  pdl_wait();
  __shared__ double red[8][128];
  __shared__ unsigned int s_ticket;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c4 = blockIdx.x * 32 + lane;                     // float4 column of this lane
  const int D4 = D >> 2;
  const int r0 = blockIdx.y * rows_per_split, r1 = min(r0 + rows_per_split, n);
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  if (c4 < D4) {
    const vec4_t<T>* p = reinterpret_cast<const vec4_t<T>*>(x) + c4;
    int r = r0 + warp;
    for (; r + 24 < r1; r += 32) {                           // four independent vector loads in flight per lane
      const float4 v0 = cvt4<T>(p[(size_t)r * D4]), v1 = cvt4<T>(p[(size_t)(r + 8) * D4]), v2 = cvt4<T>(p[(size_t)(r + 16) * D4]),
                   v3 = cvt4<T>(p[(size_t)(r + 24) * D4]);
      s[0] += ((double)v0.x + (double)v1.x) + ((double)v2.x + (double)v3.x);
      s[1] += ((double)v0.y + (double)v1.y) + ((double)v2.y + (double)v3.y);
      s[2] += ((double)v0.z + (double)v1.z) + ((double)v2.z + (double)v3.z);
      s[3] += ((double)v0.w + (double)v1.w) + ((double)v2.w + (double)v3.w);
    }
    for (; r < r1; r += 8) {
      const float4 v = cvt4<T>(p[(size_t)r * D4]);
      s[0] += v.x; s[1] += v.y; s[2] += v.z; s[3] += v.w;
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) red[warp][lane * 4 + j] = s[j];
  __syncthreads();
  if (threadIdx.x < 128) {
    const int col = blockIdx.x * 128 + threadIdx.x;
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    if (col < D) part[(size_t)blockIdx.y * D + col] = t;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(ticket + blockIdx.x, 1u);
  __syncthreads();
  if (s_ticket != gridDim.y - 1) return;                     // the last row split of this column tile adds the tile's partials
  __threadfence();
  {
    const int c = threadIdx.x & 127, hsel = threadIdx.x >> 7;  // two threads per column: even / odd splits, four loads in flight
    const int col = blockIdx.x * 128 + c;
    double t0 = 0.0, t1 = 0.0;
    if (col < D) {
      int i = hsel;
      for (; i + 2 < (int)gridDim.y; i += 4) {
        t0 += __ldcg(part + (size_t)i * D + col);
        t1 += __ldcg(part + (size_t)(i + 2) * D + col);
      }
      if (i < (int)gridDim.y) t0 += __ldcg(part + (size_t)i * D + col);
    }
    red[hsel][c] = t0 + t1;
    __syncthreads();
    if (hsel == 0 && col < D) mu[col] = (float)((red[0][c] + red[1][c]) / n);
  }
  if (threadIdx.x == 0) ticket[blockIdx.x] = 0u;
}

// ---- pre-pass 2: centred rows -> per-row scaled fp16 planes + node records, and the one-gap table of the graph's own rows.
// One warp per row (four fp32 terms, then fp64: the row statistics stay accurate to ~1e-7 relative, like the Gram entry they meet).  rec[r] = {|a'|^2, 2 eps sum a', mu.a' + |mu|^2/2, 1/|a|}, scale_inv[r] = 2^-k_r with max|a'| 2^k_r in
// [2^13, 2^14).  A row whose norm is too small for the reciprocal (the reference clamps |a||b| at 1e-8) poisons its |a'|^2 with
// NaN: every pair it takes part in then fails the cancellation test and is recomputed exactly.
// STAGE: the row is copied once into shared memory with cp.async (no registers held across the gap search and the statistics, so
// every warp of the grid is resident in one wave) and both passes read it from there; !STAGE (rows that do not fit): two passes
// over global memory.
// Gap table (rows of the graph block only): columns are strictly ascending within a row, so col[beg+k] - k is non-decreasing: 0
// before the gap, the gap length after it -> 32-ary search for the first k with col[beg+k] != k.  The row is "all columns but
// [k, k+gl)" iff the entry after the gap is k+gl and the last entry is n_cols-1; any other row raises *not_one_gap.
constexpr int GE_CS_WARPS = 4;
template <bool STAGE, typename T>
__global__ void __launch_bounds__(32 * GE_CS_WARPS) ge_center_split_kernel(const T* __restrict__ x, const float* __restrict__ mu, int n, int D,
                                                              uint2* __restrict__ hi, uint2* __restrict__ lo, float4* __restrict__ rec,
                                                              float* __restrict__ scale_inv, const mpn_graph g, int2* __restrict__ gap,
                                                              int* __restrict__ not_one_gap) {
  pdl_wait();
  extern __shared__ float4 cs_rows[];                        // STAGE: [GE_CS_WARPS][D * sizeof(T) / 16]
  constexpr bool KEEP_CENTRED = sizeof(T) == sizeof(float);  // fp32: the centred row replaces the staged one; 16-bit: re-centred
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int D4 = D >> 2;
  const float4* mu4 = reinterpret_cast<const float4*>(mu);
  const int D16 = D4 * (int)sizeof(T) / 4;                   // 16-byte chunks of a row
  float4* mine = cs_rows + (size_t)warp * D16;
  const T* srow = reinterpret_cast<const T*>(mine);
  for (int r = gwarp; r < n; r += nwarps) {
    const T* p = x + (size_t)r * D;
    if (STAGE) {                                             // the row's bytes are in flight while the gap search runs
      __syncwarp();
      for (int k = lane; k < D16; k += 32)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(mine + k)), "l"(reinterpret_cast<const float4*>(p) + k) : "memory");
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    const int lr = r - g.row_offset;
    if (lr >= 0 && lr < g.n_nodes) {                         // gap of local row lr (warp-uniform branch)
      const int beg = g.rowptr[lr], deg = g.rowptr[lr + 1] - beg;
      const int gl = g.n_cols - deg;
      int lo_k = 0, hi_k = deg;                              // first k in [lo_k, hi_k] with col[beg+k] != k (deg: the gap is at the end)
      while (hi_k - lo_k > 0) {
        const int span = hi_k - lo_k;
        const int step = (span + 31) / 32;
        const int k = lo_k + lane * step;                    // 32 probes across the interval
        const bool bad = k < hi_k ? (g.col[beg + k] != k) : true;
        const unsigned int bal = __ballot_sync(0xffffffffu, bad);
        const int first_bad = bal ? __ffs(bal) - 1 : 32;     // none: every probe is good, the answer lies behind the last one
        const int new_hi = min(lo_k + first_bad * step, hi_k);
        const int new_lo = first_bad == 0 ? lo_k : min(lo_k + (first_bad - 1) * step + 1, hi_k);
        if (step == 1) { lo_k = hi_k = new_hi; break; }
        lo_k = new_lo; hi_k = new_hi;
      }
      if (lane == 0) {
        gap[lr] = make_int2(lo_k, gl);
        const bool ok = gl >= 0 && (lo_k == deg || (g.col[beg + lo_k] == lo_k + gl && g.col[beg + deg - 1] == g.n_cols - 1));
        if (!ok) atomicOr(not_one_gap, 1);
      }
    }
    if (STAGE) {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncwarp();
    }
    double sq = 0.0, sx = 0.0, md = 0.0, mm = 0.0;
    float amax = 0.f;
    for (int k = lane; k < D4; k += 32) {
      const float4 v = ld4(STAGE ? srow : p, k);
      const float4 m = __ldg(mu4 + k);
      const float c[4] = {v.x - m.x, v.y - m.y, v.z - m.z, v.w - m.w};
      const float mv[4] = {m.x, m.y, m.z, m.w};
      if (STAGE && KEEP_CENTRED) mine[k] = make_float4(c[0], c[1], c[2], c[3]);
      float q = 0.f, s1 = 0.f, d1 = 0.f, m2 = 0.f;           // four terms in fp32, then one conversion each
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        amax = fmaxf(amax, fabsf(c[j]));
        q = fmaf(c[j], c[j], q); s1 += c[j]; d1 = fmaf(mv[j], c[j], d1); m2 = fmaf(mv[j], mv[j], m2);
      }
      sq += (double)q; sx += (double)s1; md += (double)d1; mm += (double)m2;
    }
    sq = warp_sum(sq); sx = warp_sum(sx); md = warp_sum(md); mm = warp_sum(mm);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    float s = 1.f;
    if (amax > 0.f && isfinite(amax)) {
      int e;
      frexpf(amax, &e);
      s = ldexpf(1.f, 14 - e);
    }
    if (lane == 0) {
      const double norm = sqrt(fmax(sq + 2.0 * md + mm, 0.0));
      const bool tiny = !(norm > 1e-3);
      rec[r] = make_float4(tiny ? __int_as_float(0x7fc00000) : (float)sq, (float)(2.0 * (double)PAIRWISE_EPS * sx),
                           (float)(md + 0.5 * mm), tiny ? 0.f : (float)(1.0 / norm));
      scale_inv[r] = 1.f / s;
    }
    uint2* oh = hi + (size_t)r * D4;
    uint2* ol = lo + (size_t)r * D4;
    for (int k = lane; k < D4; k += 32) {
      float c[4];
      if (STAGE && KEEP_CENTRED) {
        const float4 cv = mine[k];
        c[0] = cv.x * s; c[1] = cv.y * s; c[2] = cv.z * s; c[3] = cv.w * s;
      } else {                                               // the same fp32 difference as the staged one, scaled
        const float4 v = ld4(STAGE ? srow : p, k), m = __ldg(mu4 + k);
        c[0] = (v.x - m.x) * s; c[1] = (v.y - m.y) * s; c[2] = (v.z - m.z) * s; c[3] = (v.w - m.w) * s;
      }
      __half h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        h[j] = __float2half_rn(c[j]);
        l[j] = __float2half_rn(c[j] - __half2float(h[j]));
      }
      uint2 ph, pl;
      ph.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
      ph.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
      pl.x = (uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16);
      pl.y = (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16);
      oh[k] = ph;
      ol[k] = pl;
    }
  }
}


// ---- shared Gram: which rank computes a pair (kernels.h, GeShare) ----
__host__ __device__ __forceinline__ int ge_owner(const GeShare& sh, int c) {
  int s = 0;
  while (s + 1 < sh.world && c >= sh.blk[s + 1]) ++s;
  return s;
}
// rows [lo, hi) (global ids) of THIS rank that compute their pair with column c (owned by rank s); hi == 0: none
__host__ __device__ __forceinline__ int2 ge_row_range(const GeShare& sh, int s, int c) {
  const int R = sh.rank, W = sh.world;
  if (s == R) return make_int2(0, c);                                      // own block: r < c
  const int d = (s - R + W) % W;
  if (2 * d < W) return make_int2(0, 0x7fffffff);
  if (2 * d > W) return make_int2(0, 0);
  if (R < s) return (c < ((sh.blk[s] + sh.blk[s + 1]) >> 1)) ? make_int2(0, 0x7fffffff) : make_int2(0, 0);
  return make_int2((sh.blk[R] + sh.blk[R + 1]) >> 1, 0x7fffffff);
}

// one block: push (edge base, gap start, gap length, not_one_gap) of my rows into every rank's node table, raise my flag on every
// rank, wait for every rank's flag in my own memory, then *mode = 2 iff every rank reported dense cross-camera rows
__global__ void __launch_bounds__(1024) ge_share_exchange_kernel(const GeShare sh, const int* __restrict__ rowptr, const int2* __restrict__ gap,
                                                                 int M, const int* __restrict__ not_one_gap) {
  pdl_wait();
  const int bad = *not_one_gap;
  const int g0 = sh.blk[sh.rank];
  for (int r = threadIdx.x; r < M; r += blockDim.x) {
    const int2 gp = bad ? make_int2(0, 0) : gap[r];
    const int4 e = make_int4(rowptr[r], gp.x, gp.y, bad);
    for (int p = 0; p < sh.world; ++p) sh.tab[p][g0 + r] = e;
  }
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < sh.world) {
    st_release_sys(sh.flags[threadIdx.x] + 3 * MPN_MAX_PEERS + sh.rank, sh.seq);
    wait_flag(sh.flags[sh.rank] + 3 * MPN_MAX_PEERS + threadIdx.x, sh.seq);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int any_bad = 0;
    for (int p = 0; p < sh.world; ++p) {
      if (sh.blk[p + 1] <= sh.blk[p]) { any_bad = 1; continue; }          // a rank without rows: no shared mode
      int4 e;
      asm volatile("ld.volatile.global.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(e.x), "=r"(e.y), "=r"(e.z), "=r"(e.w) : "l"(sh.tab[sh.rank] + sh.blk[p]));
      any_bad |= e.w;
    }
    *sh.mode = any_bad ? 0 : 2;
  }
}

// ---- tile list: the 128 x 128 blocks that hold at least one edge, in a fixed order (one block, ordered compaction)
// sym: the row block is the whole graph -> blocks on or above the diagonal only (the epilogue writes both directions).
// A block is empty iff all of its rows belong to ONE camera whose node range covers all of its columns.
// shared (GeShare::mode == 2): the blocks that hold at least one pair this rank computes.
__global__ void __launch_bounds__(1024) ge_tile_list_kernel(const int2* __restrict__ gap, int M, int N, int row_global0, int sym,
                                                            int* __restrict__ tiles, int* __restrict__ n_tiles,
                                                            const int* __restrict__ not_one_gap, const GeShare sh) {
  pdl_wait();
  if (*not_one_gap != 0) { if (threadIdx.x == 0) *n_tiles = 0; return; }
  const bool shared = sh.mode != nullptr && *sh.mode == 2;
  __shared__ int warp_cnt[32];
  __shared__ int base;
  const int tm = (M + GE_BM - 1) / GE_BM, tn = (N + GE_BN - 1) / GE_BN;
  const int total = tm * tn;
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  for (int t0 = 0; t0 < total; t0 += blockDim.x) {
    const int t = t0 + threadIdx.x;
    bool keep = false;
    int ti = 0, tj = 0;
    if (t < total) {
      ti = t / tn; tj = t % tn;
      const int m0 = ti * GE_BM, n0 = tj * GE_BN;
      keep = !(sym && n0 + GE_BN <= m0 + row_global0);             // strictly below the diagonal: written by the mirror
      if (shared) {
        keep = false;
        const int r_lo = row_global0 + m0, r_hi = row_global0 + min(m0 + GE_BM, M);      // global rows [r_lo, r_hi)
        const int c_hi = min(n0 + GE_BN, N);
        for (int p = 0; p < sh.world && !keep; ++p) {
          const int a = max(n0, sh.blk[p]), b = min(c_hi, sh.blk[p + 1]);                 // this block's columns owned by rank p
          if (a >= b) continue;
          const int2 first = ge_row_range(sh, p, a), last = ge_row_range(sh, p, b - 1);   // the range is monotone in c within a block
          keep = (r_lo < first.y && r_hi > first.x) || (r_lo < last.y && r_hi > last.x);
        }
      }
      if (keep) {
        const int2 ga = gap[m0], gb = gap[min(m0 + GE_BM, M) - 1];
        const bool one_cam = ga.x == gb.x && ga.y == gb.y;
        if (one_cam && ga.x <= n0 && ga.x + ga.y >= min(n0 + GE_BN, N)) keep = false;
      }
    }
    const unsigned int bal = __ballot_sync(0xffffffffu, keep);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int off = base;
    for (int w = 0; w < warp; ++w) off += warp_cnt[w];
    if (keep) tiles[off + __popc(bal & ((1u << lane) - 1))] = (ti << 16) | tj;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += warp_cnt[w];
      base += s;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_tiles = base;
}

struct GeArgs {
  const float4* rec;          // [n_cols] node records, global node ids
  const float* scale_inv;     // [n_cols]
  const int* rowptr;          // [M+1] local rows
  const int2* gap;            // [M] local rows: (first column of the gap, length)
  const int* tiles;
  const int* n_tiles;
  const int* not_one_gap;
  float2* edge_attr;
  int* refine_list;
  int* refine_count;
  int balance;                // 1: blocks beyond ceil(T / rounds) take no tiles
  double* partials;           // [gridDim.x][MPN_SUMS_DOUBLES] moment partial rows (columns 0..4) or nullptr
  int M, N, K;                // rows of the block, columns (= nodes of the graph), feature width
  int row_global0;            // global node id of local row 0
  int sym;
  float d_eps2;               // D * eps^2
  GeShare sh;                 // SHARED kernel only
  const int4* node_tab;       // SHARED: this rank's copy of the node table [N]
};

template <bool SHARED>
__global__ void __launch_bounds__(GE_THREADS, 1)
gram_ef_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo, const GeArgs A) {
  pdl_wait();
  if (*A.not_one_gap != 0) return;
  if (A.sh.mode != nullptr && (*A.sh.mode == 2) != SHARED) return;       // sharded runs enqueue both variants: the exchange decides
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for the swizzled tiles, computed on the shared-space address so that the pointers keep their state space
  // (a round trip through uintptr_t makes every later access a generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  GeSmem& S = *reinterpret_cast<GeSmem*>(smem + GE_STAGES * GE_STAGE_BYTES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = *A.n_tiles;
  const int num_kb = (A.K + GE_BK - 1) / GE_BK;
  // Balanced rounds: T tiles take ceil(T / grid) rounds whatever happens, so only ceil(T / rounds) blocks work and the others leave
  // their SM to the kernels of the other stream (the node encoder runs beside this kernel): 448 tiles -> 112 blocks x 4 tiles.
  const int n_rounds = (n_tiles + (int)gridDim.x - 1) / (int)gridDim.x;
  const int t_stride = (A.balance && n_rounds > 0) ? (n_tiles + n_rounds - 1) / n_rounds : (int)gridDim.x;
  const int t_first = (int)blockIdx.x < t_stride ? (int)blockIdx.x : n_tiles;
  if (threadIdx.x == 0) {
    for (int s = 0; s < GE_STAGES; ++s) { mbar_init(&S.full_bar[s], 1); mbar_init(&S.empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&S.tmem_full_bar[a], 1); mbar_init(&S.tmem_empty_bar[a], 32 * GE_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(&S.tmem_slot, GE_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = S.tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_hi));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_lo));
      int stage = 0;
      uint32_t phase = 0;
      for (int t = t_first; t < n_tiles; t += t_stride) {
        const int tile = A.tiles[t];
        const int m0 = (tile >> 16) * GE_BM, n0 = (tile & 0xffff) * GE_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&S.empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * GE_STAGE_BYTES;
          mbar_expect_tx(&S.full_bar[stage], GE_STAGE_BYTES);
          const int k0 = kb * GE_BK;
          // stage layout: A_hi | A_lo | B_hi | B_lo (B_hi and B_lo adjacent: one N = 256 operand [b_hi ; b_lo])
          tma_load_2d(&map_a_hi, &S.full_bar[stage], st, k0, m0);
          tma_load_2d(&map_a_lo, &S.full_bar[stage], st + GE_PLANE_BYTES, k0, m0);
          tma_load_2d(&map_b_hi, &S.full_bar[stage], st + 2 * GE_PLANE_BYTES, k0, n0);
          tma_load_2d(&map_b_lo, &S.full_bar[stage], st + 3 * GE_PLANE_BYTES, k0, n0);
          if (++stage == GE_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    // per k-slice (16 fp16):  a_hi x [b_hi ; b_lo]^T  (N = 256)  ->  [hh_s | corr_s]      hi.hi and hi.lo in one instruction
    //                         a_lo x  b_hi^T          (N = 128)  ->        corr_s          lo.hi
    // Two accumulator sets [hh | corr] (2 x 256 TMEM columns) alternate from TILE to tile: while the epilogue warps drain set s
    // the issuer already fills set s ^ 1 with the next tile, so the tensor pipe does not wait for the epilogue.  The shared
    // A_hi / B_hi operands are read from shared memory twice instead of three times (the main loop is shared-memory bound).
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int t = t_first; t < n_tiles; t += t_stride, ++it) {
        const int as = it & 1;
        if (it >= 2) {                                    // the epilogue has read this set's previous tile (two tiles ago)
          mbar_wait(&S.tmem_empty_bar[as], (uint32_t)(((it >> 1) - 1) & 1));
          tc_fence_after();
        }
        const uint32_t set = tmem_base + (uint32_t)as * 256u;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&S.full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sbase = smem_u32(smem + stage * GE_STAGE_BYTES);
          const uint64_t a_hi = ge_smem_desc(sbase), a_lo = ge_smem_desc(sbase + GE_PLANE_BYTES);
          const uint64_t b_hi = ge_smem_desc(sbase + 2 * GE_PLANE_BYTES);     // rows 128..255 of the N = 256 operand are B_lo
#pragma unroll
          for (int kk = 0; kk < GE_BK / 16; ++kk) {
            const uint64_t adv = (uint64_t)((kk * 32) >> 4);          // 16 fp16 = 32 bytes of K per instruction
            umma_f16(set, a_hi + adv, b_hi + adv, GE_IDESC_N256, (kb | kk) != 0);
            umma_f16(set + 128u, a_lo + adv, b_hi + adv, GE_IDESC_N128, 1);
          }
          umma_commit(&S.empty_bar[stage]);
          if (++stage == GE_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&S.tmem_full_bar[as]);
      }
    }
  } else {
    // ===== epilogue (warps 2..9): TMEM lane quarter = warp & 3, column half = (warp - 2) >> 2; thread = one row of the tile =====
    const int ew = warp - 2;
    const int q = warp & 3, half = ew >> 2;
    const int et = threadIdx.x - 64;                      // 0..255 among the epilogue threads
    int it = 0;
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    float2 (*tb)[GE_TPITCH] = S.tbuf[ew];
    for (int t = t_first; t < n_tiles; t += t_stride, ++it) {
      const int as = it & 1;                                // accumulator set of this tile
      const int tile = A.tiles[t];
      const int m0 = (tile >> 16) * GE_BM, n0 = (tile & 0xffff) * GE_BN;
      const bool mirror = SHARED || (A.sym && n0 >= m0 + A.row_global0 + GE_BM);     // off-diagonal block of the whole graph
      // stage the per-column and per-row tables of this tile (the previous tile's epilogue has passed the named barrier below)
      if (et < GE_BN) {
        const int c = n0 + et;
        float4 ca = make_float4(0.f, 0.f, 0.f, 0.f);
        int4 cb = make_int4(0, -1, -1, 0);
        if (c < A.N) {
          ca = __ldg(A.rec + c);
          cb.x = __float_as_int(__ldg(A.scale_inv + c));
          const int lc = c - A.row_global0;                // the column as a row of this block (mirrored entries)
          if (SHARED) {
            const int owner = ge_owner(A.sh, c);
            const int2 range = ge_row_range(A.sh, owner, c);
            if (range.y > 0) {
              const int4 te = __ldg(A.node_tab + c);       // (edge base, gap start, gap length) of row c in its owner's shard
              cb.y = te.x; cb.z = te.x - te.z; cb.w = te.y + te.z;
            }
            S.cs_ptr[et] = A.sh.ea[owner];
            S.cs_lohi[et] = range;
          } else if (mirror && lc >= 0 && lc < A.M) {
            const int2 gp = __ldg(A.gap + lc);
            const int rp = __ldg(A.rowptr + lc);
            cb.y = rp; cb.z = rp - gp.y; cb.w = gp.x + gp.y;
          }
        } else if (SHARED) {
          S.cs_ptr[et] = A.edge_attr;
          S.cs_lohi[et] = make_int2(0, 0);
        }
        S.cs_a[et] = ca;
        S.cs_b[et] = cb;
      } else {
        const int r = m0 + et - GE_BN;
        int4 ri = make_int4(0, 0, 0, 0);
        if (r < A.M) {
          const int2 gp = __ldg(A.gap + r);
          const int rp = __ldg(A.rowptr + r);
          ri = make_int4(rp, rp - gp.y, gp.x + gp.y, 1);
        }
        S.rowinfo[et - GE_BN] = ri;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");       // tables visible to the epilogue warps
      const int row = m0 + q * 32 + lane;                  // local row of this thread
      const bool row_ok = row < A.M;
      float4 ra = make_float4(0.f, 0.f, 0.f, 0.f);
      float inv_a = 0.f;
      int gap0 = 0, gap1 = 0, rp_row = 0;
      if (row_ok) {
        ra = __ldg(A.rec + A.row_global0 + row);
        inv_a = __ldg(A.scale_inv + A.row_global0 + row);
        const int2 gp = __ldg(A.gap + row);
        rp_row = __ldg(A.rowptr + row);
        gap0 = gp.x; gap1 = gp.x + gp.y;
      }
      const float rn_a = ra.w, ma = ra.z, sa = ra.x, ea = ra.y;
      const int grow = A.row_global0 + row;                // global id of this thread's node (position in the mirrored rows)
      mbar_wait(&S.tmem_full_bar[as], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < 2; ++cc) {
        const int c0 = half * 64 + cc * 32;
        const int cbase = n0 + c0;
        if (cbase >= A.N) break;                            // warp-uniform
        // columns of this chunk that are edges of this thread's row: valid columns minus the row's gap, as a bit mask
        unsigned int cmask = 0u;
        if (row_ok) {
          const int nv = A.N - cbase;
          cmask = nv >= 32 ? 0xffffffffu : ((1u << nv) - 1u);
          const int lo = max(gap0 - cbase, 0), hi = min(gap1 - cbase, 32);
          if (hi > lo) cmask &= ~((hi >= 32 ? 0xffffffffu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u));
        }
        float v[32], w[32];
        const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 256 + c0);
        tmem_ld32_issue(tq, v);                             // hh
        tmem_ld32_issue(tq + 128u, w);                      // corr
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += w[j];
        float s_a = 0.f, s_b = 0.f, s_aa = 0.f, s_ab = 0.f, s_bb = 0.f;      // this chunk's sums in fp32 (<= 2 x 32 terms per lane)
        unsigned int flagged = 0u;                          // entries whose d2 cancels (rare): handled after the chunk
#pragma unroll
        for (int sub = 0; sub < 32 / GE_SUB; ++sub) {
#pragma unroll
          for (int jj = 0; jj < GE_SUB; ++jj) {
            const int j = sub * GE_SUB + jj;
            const float4 ca = S.cs_a[c0 + j];
            const int4 cb = S.cs_b[c0 + j];
            const float g = v[j] * (inv_a * __int_as_float(cb.x));
            const float tsum = sa + ca.x;
            const float u = fmaf(-2.f, g, tsum) + A.d_eps2;
            const float wv = ea - ca.y;
            const float d2d = u + wv, d2m = u - wv;
            bool cross = (cmask >> j) & 1u;
            if (SHARED) {                                   // pairs of this column that another rank computes are not mine
              const int2 range = S.cs_lohi[c0 + j];
              cross = cross && grow >= range.x && grow < range.y;
            }
            const bool cancel = !(fminf(d2d, d2m) >= REFINE_FRACTION * tsum);          // also true for NaN (degenerate rows)
            const float rs = rsqrt_approx(fmaxf(d2d, 1e-30f));
            const float dd = d2d * rs;
            const float dm = fmaf(-wv, rs, dd);             // sqrt(d2d - 2 w) to first order (w ~ 1e-6: the next term is ~1e-12)
            const float cosv = 1.0f - (g + ma + ca.z) * (rn_a * ca.w);
            const bool take = cross && !cancel;
            if (cross && cancel) flagged |= 1u << j;
            const float dds = take ? dd : 0.f, coss = take ? cosv : 0.f;
            if (mirror) {
              const float dms = take ? dm : 0.f;
              const float sd = dds + dms;
              s_a += sd; s_aa = fmaf(dds, dds, fmaf(dms, dms, s_aa)); s_b = fmaf(2.f, coss, s_b); s_bb = fmaf(2.f * coss, coss, s_bb);
              s_ab = fmaf(coss, sd, s_ab);
              if (cross && cb.y >= 0) {                     // (j -> i): consecutive lanes = consecutive edges of row j
                float2* dst = SHARED ? S.cs_ptr[c0 + j] : A.edge_attr;     // SHARED: the owner of row j, over NVLink if it is a peer
                dst[grow + (grow >= cb.w ? cb.z : cb.y)] = make_float2(dm, cosv);
              }
            } else {
              s_a += dds; s_aa = fmaf(dds, dds, s_aa); s_b += coss; s_bb = fmaf(coss, coss, s_bb); s_ab = fmaf(coss, dds, s_ab);
            }
            tb[lane][jj] = make_float2(cross ? dd : -1.f, cosv);
          }
          __syncwarp();
          // direct entries (i -> j) of 32 rows x 8 columns: 8 lanes per row, four rows per instruction
          {
            const int cj = lane & (GE_SUB - 1), rsel = lane >> 3;
            const int col = cbase + sub * GE_SUB + cj;
#pragma unroll
            for (int k = 0; k < 32; k += 4) {
              const int rr = k + rsel;
              const float2 o = tb[rr][cj];
              const int4 ri = S.rowinfo[q * 32 + rr];
              if (o.x >= 0.f) A.edge_attr[col + (col >= ri.z ? ri.y : ri.x)] = o;
            }
          }
          __syncwarp();
        }
        if (__any_sync(0xffffffffu, flagged != 0u)) {       // cold path: list the cancelled pairs for the exact recomputation
          while (flagged) {
            const int j = __ffs(flagged) - 1;
            flagged &= flagged - 1;
            const int col = cbase + j;
            const int4 cb = S.cs_b[c0 + j];
            const bool mir = !SHARED && mirror && cb.y >= 0;      // SHARED: edge_feature_refine writes both directions itself
            const int slot = atomicAdd(A.refine_count, mir ? 2 : 1);
            A.refine_list[slot] = col + (col >= gap1 ? rp_row - (gap1 - gap0) : rp_row);
            if (mir) A.refine_list[slot + 1] = grow + (grow >= cb.w ? cb.z : cb.y);
          }
        }
        acc[0] += (double)s_a; acc[1] += (double)s_b; acc[2] += (double)s_aa; acc[3] += (double)s_ab; acc[4] += (double)s_bb;
      }
      tc_fence_before();
      mbar_arrive(&S.tmem_empty_bar[as]);                   // this thread's tcgen05.ld of the tile have completed
      asm volatile("bar.sync 1, 256;" ::: "memory");       // everyone is done with cs / rowinfo before the next tile restages them
    }
    if (A.partials != nullptr) {
      // block partial row: fixed shuffle tree + fixed order over the eight warps (bit-reproducible for a fixed tile list)
      double* red = reinterpret_cast<double*>(&S.tbuf[0][0][0]);
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const double s = warp_sum(acc[k]);
        if (lane == 0) red[ew * 5 + k] = s;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (et < 5) {
        double s = 0.0;
        for (int wv = 0; wv < GE_EPI_WARPS; ++wv) s += red[wv * 5 + et];
        A.partials[(size_t)blockIdx.x * MPN_SUMS_DOUBLES + et] = s;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, GE_TMEM_COLS);
  }
}

int ge_workspace_layout(int n_cols, int M, int D, GeWorkspace* L, void* ws, size_t ws_bytes) {
  Arena a(ws, ws_bytes);
  const size_t plane = (size_t)n_cols * D;
  L->hi = a.take<uint16_t>(plane);
  L->lo = a.take<uint16_t>(plane);
  L->rec = a.take<float4>((size_t)n_cols);
  L->scale_inv = a.take<float>((size_t)n_cols);
  const int tm = (M + GE_BM - 1) / GE_BM, tn = (n_cols + GE_BN - 1) / GE_BN;
  L->tiles = a.take<int>((size_t)tm * tn);
  L->n_tiles = a.take<int>(1);
  L->total = a.off;
  return a.ok() ? MPN_OK : MPN_ERR_WORKSPACE;
}

int ge_col_mean_splits() { return GE_CM_SPLITS; }
bool gram_ef_shape_ok(int M, int N, int D) { return M >= 1 && N >= 2 && D >= GE_BK && (D % GE_BK) == 0 && N < 65536 * GE_BN && M < 65536 * GE_BM; }

// centred fp16 planes + records, tile list, persistent GEMM with the distance epilogue.  Every kernel returns at once when
// *not_one_gap != 0 (the graph is not dense cross-camera: the Gram + gather path runs instead).
static int g_profile_gram = 0;
static cudaEvent_t g_prof_ev[2] = {nullptr, nullptr};

int ge_col_mean(const void* x, int x_kind, int n, int D, double* part, unsigned int* ticket, float* mu, cudaStream_t st) {
  MPN_REQUIRE((D % 4) == 0 && x_vec4_aligned(x, x_kind), "column means: D must be a multiple of 4 and x aligned to four elements");
  const int splits = min(GE_CM_SPLITS, max(1, n / 8));
  return with_x_type(x_kind, [&](auto xt) {
    mpn::launch(ge_col_mean_kernel<x_elem_t<decltype(xt)>>, dim3(div_up(D, 128), splits), 256, 0, st, (decltype(xt))x, n, D, div_up(n, splits),
                part, ticket, mu);
    MPN_LAUNCH_OK();
    return MPN_OK;
  });
}

int gram_ef_run(const void* x, int x_kind, const float* mu, const mpn_graph* g, int D, int2* gap, int* not_one_gap, float2* edge_attr,
                int* refine_list, int* refine_count, double* partials, int* n_partial_rows, const GeWorkspace& L, cudaStream_t st,
                const GeShare* share) {
  const int N = g->n_cols, M = g->n_nodes;
  MPN_REQUIRE(gram_ef_shape_ok(M, N, D), "fused edge features: unsupported shape M=%d N=%d D=%d", M, N, D);
  const int cs_grid = min(kNumSMs * 16, div_up((long long)N, GE_CS_WARPS));
  MPN_TRY(with_x_type(x_kind, [&](auto xt) {
    using T = x_elem_t<decltype(xt)>;
    const size_t cs_smem = (size_t)GE_CS_WARPS * D * sizeof(T);
    if (cs_smem <= 48 * 1024) {                            // rows of up to 48 KB / GE_CS_WARPS are staged in shared memory
      mpn::launch(ge_center_split_kernel<true, T>, cs_grid, 32 * GE_CS_WARPS, cs_smem, st, (const T*)x, mu, N, D, (uint2*)L.hi, (uint2*)L.lo, L.rec,
                  L.scale_inv, *g, gap, not_one_gap);
    } else {
      mpn::launch(ge_center_split_kernel<false, T>, cs_grid, 32 * GE_CS_WARPS, 0, st, (const T*)x, mu, N, D, (uint2*)L.hi, (uint2*)L.lo, L.rec,
                  L.scale_inv, *g, gap, not_one_gap);
    }
    MPN_LAUNCH_OK();
    return MPN_OK;
  }));
  GeShare sh;
  memset(&sh, 0, sizeof(sh));
  if (share != nullptr) {
    sh = *share;
    MPN_REQUIRE(sh.world >= 2 && sh.world <= MPN_MAX_PEERS && sh.rank >= 0 && sh.rank < sh.world && sh.mode != nullptr, "shared Gram: bad rank/world");
    MPN_REQUIRE(sh.blk[sh.rank] == g->row_offset && sh.blk[sh.rank + 1] == g->row_offset + M && sh.blk[0] == 0 && sh.blk[sh.world] == N,
                "shared Gram: the row blocks do not match the graph (block [%d,%d), graph rows [%d,%d) of %d)", sh.blk[sh.rank],
                sh.blk[sh.rank + 1], g->row_offset, g->row_offset + M, N);
    MPN_REQUIRE((float2*)sh.ea[sh.rank] == edge_attr, "shared Gram: edge_attr must be this rank's peer-visible buffer");
    mpn::launch(ge_share_exchange_kernel, 1, 1024, 0, st, sh, g->rowptr, (const int2*)gap, M, (const int*)not_one_gap);
    MPN_LAUNCH_OK();
  }
  const int sym = (g->row_offset == 0 && M == N) ? 1 : 0;
  mpn::launch(ge_tile_list_kernel, 1, 1024, 0, st, gap, M, N, g->row_offset, sym, L.tiles, L.n_tiles, not_one_gap, sh);
  MPN_LAUNCH_OK();
  CUtensorMap ah, al, bh, bl;
  MPN_TRY(make_tma_map_2d(&ah, L.hi + (size_t)g->row_offset * D, M, D, GE_BM, true));
  MPN_TRY(make_tma_map_2d(&al, L.lo + (size_t)g->row_offset * D, M, D, GE_BM, true));
  MPN_TRY(make_tma_map_2d(&bh, L.hi, N, D, GE_BN, true));
  MPN_TRY(make_tma_map_2d(&bl, L.lo, N, D, GE_BN, true));
  static bool configured = false;
  if (!configured) {
    MPN_CUDA_OK(cudaFuncSetAttribute(gram_ef_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, GE_SMEM_BYTES));
    MPN_CUDA_OK(cudaFuncSetAttribute(gram_ef_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GE_SMEM_BYTES));
    configured = true;
  }
  GeArgs A;
  A.rec = L.rec; A.scale_inv = L.scale_inv; A.rowptr = g->rowptr; A.gap = gap; A.tiles = L.tiles; A.n_tiles = L.n_tiles;
  A.not_one_gap = not_one_gap; A.edge_attr = edge_attr; A.refine_list = refine_list; A.refine_count = refine_count;
  A.partials = partials; A.M = M; A.N = N; A.K = D; A.row_global0 = g->row_offset; A.sym = sym;
  A.d_eps2 = (float)((double)D * (double)PAIRWISE_EPS * (double)PAIRWISE_EPS);
  A.sh = sh;
  A.node_tab = share ? sh.tab[sh.rank] : nullptr;
  static int balance = -1;                               // MPN_GRAM_BALANCE=0: every block strides by the grid (diagnostics)
  if (balance < 0) { const char* e = getenv("MPN_GRAM_BALANCE"); balance = e ? atoi(e) : 1; }
  A.balance = balance;
  const int tm = (M + GE_BM - 1) / GE_BM, tn = (N + GE_BN - 1) / GE_BN;
  const int grid = (int)min((long long)kNumSMs, (long long)tm * tn);
  if (n_partial_rows) *n_partial_rows = grid;
  if (g_profile_gram) {                                  // bench.py: duration of the Gram launch(es) (events on the launching stream)
    if (!g_prof_ev[0]) { MPN_CUDA_OK(cudaEventCreate(&g_prof_ev[0])); MPN_CUDA_OK(cudaEventCreate(&g_prof_ev[1])); }
    MPN_CUDA_OK(cudaEventRecord(g_prof_ev[0], st));
  }
  mpn::launch(gram_ef_kernel<false>, grid, GE_THREADS, GE_SMEM_BYTES, st, ah, al, bh, bl, A);
  MPN_LAUNCH_OK();
  if (share != nullptr) {                                // exactly one of the two runs (GeShare::mode, decided on the device)
    mpn::launch(gram_ef_kernel<true>, grid, GE_THREADS, GE_SMEM_BYTES, st, ah, al, bh, bl, A);
    MPN_LAUNCH_OK();
  }
  if (g_profile_gram) MPN_CUDA_OK(cudaEventRecord(g_prof_ev[1], st));
  return MPN_OK;
}

}  // namespace mpn

// tests: the pair-ownership rule of the shared Gram as the kernels evaluate it (same functions, compiled for the host): the rows
// [out[0], out[1]) of rank `rank` compute their pair with column c; returns the owner of c, or -1 on bad arguments
extern "C" int mpn_shared_gram_row_range(int32_t rank, int32_t world, const int32_t* block_start, int32_t c, int32_t* out) {
  if (world < 1 || world > MPN_MAX_PEERS || rank < 0 || rank >= world || block_start == nullptr || out == nullptr) return -1;
  mpn::GeShare sh;
  memset(&sh, 0, sizeof(sh));
  sh.rank = rank; sh.world = world;
  for (int r = 0; r <= world; ++r) sh.blk[r] = block_start[r];
  if (c < sh.blk[0] || c >= sh.blk[world]) return -1;
  const int owner = mpn::ge_owner(sh, c);
  const int2 range = mpn::ge_row_range(sh, owner, c);
  out[0] = range.x; out[1] = range.y;
  return owner;
}

extern "C" int mpn_profile_gram(int enable) {
  mpn::g_profile_gram = enable != 0;
  return mpn::g_profile_gram;
}
extern "C" float mpn_profile_gram_ms(void) {
  float ms = -1.f;
  if (mpn::g_prof_ev[0] && cudaEventSynchronize(mpn::g_prof_ev[1]) == cudaSuccess) cudaEventElapsedTime(&ms, mpn::g_prof_ev[0], mpn::g_prof_ev[1]);
  return ms;
}
