// Shared helpers for the sm_100a kernels of the MPN path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/mpn_b200.h"

namespace mpn {

constexpr int kNumSMs = 148;          // B200: 2 dies x 74 SMs; grids are sized in multiples of this

void set_error(const char* fmt, ...);
extern unsigned long long g_kernel_launches;   // kernels launched by this library (bench.py's gpu_launches)

#define MPN_CUDA_OK(expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      mpn::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return MPN_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define MPN_LAUNCH_OK()                                                                        \
  do {                                                                                         \
    ++mpn::g_kernel_launches;                                                                  \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) {                                                                   \
      mpn::set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return MPN_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define MPN_REQUIRE(cond, ...)                                                                 \
  do {                                                                                         \
    if (!(cond)) {                                                                             \
      mpn::set_error(__VA_ARGS__);                                                             \
      return MPN_ERR_INVALID;                                                                  \
    }                                                                                          \
  } while (0)

#define MPN_TRY(expr)                                                                          \
  do {                                                                                         \
    int _rc = (expr);                                                                          \
    if (_rc != MPN_OK) return _rc;                                                             \
  } while (0)

// Bump allocator over a caller-provided device workspace (256-byte aligned slices).
struct Arena {
  char* base;
  size_t cap;
  size_t off;
  bool dry;                        // dry run: only measures
  Arena(void* p, size_t n) : base((char*)p), cap(n), off(0), dry(p == nullptr) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    char* p = dry ? nullptr : base + off;
    off += bytes;
    return (T*)p;
  }
  bool ok() const { return dry || off <= cap; }
};

static inline int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// Programmatic dependent launch (on by default; mpn_set_pdl(0) switches it off for A/B measurements).  A kernel launched
// through launch() carries the programmatic-stream-serialization attribute and may be scheduled while its predecessor in the
// stream drains; its first statement, pdl_wait() (griddepcontrol.wait), blocks every thread until the predecessor grid has
// completed and its writes are visible, so only the launch latency overlaps (measured on configs[1]: 0.838 -> 0.795 ms per
// step, profiles/r2_01_gap_experiments.md; triggering the dependent launch early inside the kernels gave nothing more).
// Rule: pdl_wait() is the FIRST statement of every kernel launched through launch(), before any early return (a grid whose
// blocks all skipped it would let its own successor overtake the predecessor).
extern int g_pdl_launch;             // run-time switch

#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... Params, typename... Args>
static inline void launch(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  if (g_pdl_launch) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<Args&&>(args)...);     // errors surface through MPN_LAUNCH_OK()
    return;
  }
  kernel<<<grid, block, smem, st>>>(static_cast<Args&&>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of K doubles per thread; result valid in thread 0..K-1 of warp 0 as out[k].
// Deterministic: fixed shuffle tree + fixed order over warps.
template <int K, int THREADS>
__device__ __forceinline__ void block_sum_doubles(double (&v)[K], double* smem /* [THREADS/32][K] */, double* out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double s = warp_sum(v[k]);
    if (lane == 0) smem[warp * K + k] = s;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    double s = 0.0;
    for (int w = 0; w < THREADS / 32; ++w) s += smem[w * K + threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// Block-wide sum of K columns held one per lane (lane k < K of every warp holds column k); result in out[0..K-1].
// Deterministic: fixed order over warps.
template <int K, int THREADS>
__device__ __forceinline__ void block_sum_lane_columns(double v, double* smem /* [THREADS/32][K] */, double* out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane < K) smem[warp * K + lane] = v;
  __syncthreads();
  if (threadIdx.x < K) {
    double s = 0.0;
    for (int w = 0; w < THREADS / 32; ++w) s += smem[w * K + threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// streaming (read-once) loads: bypass L1 allocation
__device__ __forceinline__ float4 ldg_stream4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float2 ldg_stream2(const float2* p) {
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ int ldg_stream_i32(const int* p) {
  int r;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
#endif

// ---- sequence flags in NVLink peer memory (sharded runs) ----
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// wait until *p >= seq; a protocol bug or a dead peer must surface as a trap, never as a hung GPU
__device__ __forceinline__ void wait_flag(const unsigned long long* p, unsigned long long seq) {
  if (ld_acquire_sys(p) >= seq) return;
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (ld_acquire_sys(p) < seq) {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 10000000000ull) __trap();
  }
}


}  // namespace mpn
