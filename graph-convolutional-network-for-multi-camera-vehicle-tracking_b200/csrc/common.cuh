// Shared helpers for the sm_100a kernels of the MPN path.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>

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

// node-feature element kinds (MPN_X_*): validity, element size, and the call of f with a typed null pointer of the element type
static inline bool x_kind_ok(int kind) { return kind == MPN_X_F32 || kind == MPN_X_F16 || kind == MPN_X_BF16; }
static inline size_t x_elem_bytes(int kind) { return kind == MPN_X_F32 ? sizeof(float) : 2; }
// the vector loads of x (ld4 / cvt4) read four elements at once: 16 bytes for fp32, 8 for 16-bit types
static inline bool x_vec4_aligned(const void* x, int kind) { return ((uintptr_t)x % (4 * x_elem_bytes(kind))) == 0; }
template <typename P>
using x_elem_t = std::remove_cv_t<std::remove_pointer_t<P>>;     // element type behind with_x_type's typed null pointer
template <typename F>
static inline int with_x_type(int kind, F&& f) {
  switch (kind) {
    case MPN_X_F32: return f((const float*)nullptr);
    case MPN_X_F16: return f((const __half*)nullptr);
    case MPN_X_BF16: return f((const __nv_bfloat16*)nullptr);
  }
  set_error("unknown node-feature element kind %d (MPN_X_F32, MPN_X_F16 or MPN_X_BF16)", kind);
  return MPN_ERR_INVALID;
}
#define MPN_X_KIND_OK(kind) MPN_REQUIRE(mpn::x_kind_ok(kind), "unknown node-feature element kind %d (MPN_X_F32, MPN_X_F16 or MPN_X_BF16)", (int)(kind))

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

// Node features x of element type T (float, __half, __nv_bfloat16: MPN_X_F32 / F16 / BF16), converted to fp32 on load.  Both
// 16-bit conversions are exact, so a kernel templated on T computes on the same fp32 values as on x.float().  ld4(p, i) reads
// the i-th group of four consecutive elements from p, which an fp32 kernel reads as one float4 (16 bytes for fp32, 8 for 16-bit
// types): every lane keeps its columns and every reduction its order and grouping, whatever the width of the element.
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
using vec4_t = std::conditional_t<sizeof(T) == 4, float4, uint2>;      // four elements of T as one load
template <typename T>
__device__ __forceinline__ float4 cvt4(const vec4_t<T>& v) {
  if constexpr (sizeof(T) == 4) {
    return v;
  } else {
    T e[4];
    memcpy(e, &v, sizeof(v));
    return make_float4(to_f32(e[0]), to_f32(e[1]), to_f32(e[2]), to_f32(e[3]));
  }
}
template <typename T, typename I>
__device__ __forceinline__ float4 ld4(const T* p, I i) {     // p: 16-byte aligned for fp32, 8-byte aligned for 16-bit types
  return cvt4<T>(reinterpret_cast<const vec4_t<T>*>(p)[i]);
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
