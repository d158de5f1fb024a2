// fp32 SIMT "NT" GEMM:  C[M,N] = f(A)[M,K] * B[N,K]^T + bias[N]
// f(A)[m,k] = A[m,k]                         (a_scale == nullptr)
//           = relu(A[m,k]*a_scale[k]+a_shift[k])   (fused BatchNorm+ReLU of the previous encoder layer, models/mlp.py:14-19)
// This is the exact-fp32 building block (and the checker for the tcgen05 3xTF32 kernel in gemm_tc.cu).
#include "common.cuh"
#include "kernels.h"

namespace mpn {

constexpr int BM = 64, BN = 64, BK = 16, GT = 256;

template <bool ALIGNED, typename T>
__device__ __forceinline__ float4 load4(const T* __restrict__ base, int r, int rows, int k, int K, long long ld) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r < rows) {
    const T* p = base + (long long)r * ld + k;
    if (ALIGNED && k + 3 < K) {
      v = ld4(p, 0);
    } else {
      if (k + 0 < K) v.x = to_f32(p[0]);
      if (k + 1 < K) v.y = to_f32(p[1]);
      if (k + 2 < K) v.z = to_f32(p[2]);
      if (k + 3 < K) v.w = to_f32(p[3]);
    }
  }
  return v;
}

template <bool ALIGNED, typename TA>
__global__ void __launch_bounds__(GT) gemm_nt_simt_kernel(const TA* __restrict__ A, const float* __restrict__ B,
                                                          const float* __restrict__ bias, const float* __restrict__ a_scale,
                                                          const float* __restrict__ a_shift, const int* __restrict__ row_gid,
                                                          float* __restrict__ C, int M, int N, int K) {
  pdl_wait();
  __shared__ float As[2][BK][BM + 4];
  __shared__ float Bs[2][BK][BN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int lr = tid >> 2, lk = (tid & 3) * 4;            // loader: row lr, k offset lk
  const int ty = tid >> 4, tx = tid & 15;                  // compute: 4x4 micro-tile
  float acc[4][4] = {};

  auto fetchA = [&](int k0) {
    float4 v = load4<ALIGNED>(A, m0 + lr, M, k0 + lk, K, K);
    if (a_scale != nullptr) {
      const int k = k0 + lk;
      const int m = min(m0 + lr, M - 1);
      const float* sc = a_scale + (row_gid ? (size_t)row_gid[m] * K : 0);     // per-graph BatchNorm (batched graphs)
      const float* sh = a_shift + (row_gid ? (size_t)row_gid[m] * K : 0);
      if (k + 0 < K) v.x = fmaxf(fmaf(v.x, sc[k + 0], sh[k + 0]), 0.f);
      if (k + 1 < K) v.y = fmaxf(fmaf(v.y, sc[k + 1], sh[k + 1]), 0.f);
      if (k + 2 < K) v.z = fmaxf(fmaf(v.z, sc[k + 2], sh[k + 2]), 0.f);
      if (k + 3 < K) v.w = fmaxf(fmaf(v.w, sc[k + 3], sh[k + 3]), 0.f);
      if (m0 + lr >= M) v = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    return v;
  };
  auto fetchB = [&](int k0) { return load4<ALIGNED>(B, n0 + lr, N, k0 + lk, K, K); };
  auto stash = [&](int buf, float4 a, float4 b) {
    As[buf][lk + 0][lr] = a.x; As[buf][lk + 1][lr] = a.y; As[buf][lk + 2][lr] = a.z; As[buf][lk + 3][lr] = a.w;
    Bs[buf][lk + 0][lr] = b.x; Bs[buf][lk + 1][lr] = b.y; Bs[buf][lk + 2][lr] = b.z; Bs[buf][lk + 3][lr] = b.w;
  };

  const int nk = (K + BK - 1) / BK;
  float4 ra = fetchA(0), rb = fetchB(0);
  stash(0, ra, rb);
  __syncthreads();
  for (int kb = 0; kb < nk; ++kb) {
    const int buf = kb & 1;
    if (kb + 1 < nk) { ra = fetchA((kb + 1) * BK); rb = fetchB((kb + 1) * BK); }
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (kb + 1 < nk) stash(buf ^ 1, ra, rb);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) C[(long long)m * N + n] = acc[i][j] + (bias ? bias[n] : 0.f);
    }
  }
}

int gemm_nt_simt(const void* A, const float* B, const float* bias, const float* a_scale, const float* a_shift, float* C,
                 int M, int N, int K, cudaStream_t st, const int* row_gid, int a_kind) {
  MPN_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: bad shape %d x %d x %d", M, N, K);
  dim3 grid(div_up(N, BN), div_up(M, BM));
  const bool aligned = (K % 4 == 0) && (((uintptr_t)A | (uintptr_t)B) % 16 == 0);
  return with_x_type(a_kind, [&](auto at) {
    using TA = x_elem_t<decltype(at)>;
    if (aligned)
      mpn::launch(gemm_nt_simt_kernel<true, TA>, grid, GT, 0, st, (const TA*)A, B, bias, a_scale, a_shift, row_gid, C, M, N, K);
    else
      mpn::launch(gemm_nt_simt_kernel<false, TA>, grid, GT, 0, st, (const TA*)A, B, bias, a_scale, a_shift, row_gid, C, M, N, K);
    MPN_LAUNCH_OK();
    return MPN_OK;
  });
}

}  // namespace mpn
