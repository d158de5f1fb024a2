// Rows (f2) and (f3) of SURVEY.md section 8: what the reference does with the decisions after the hot path.
//   edge confusion counts            compute_P_R_F                       inference.py:20-66
//   contingency table of two labelings (ARI / AMI / homogeneity / completeness / V-measure are functions of it;
//                                     the reference calls sklearn.metrics on ID_GT, ID_pred)     inference.py:507-519
//   expected mutual information      sklearn.metrics.cluster._expected_mutual_info_fast (scikit-learn 0.24.2, env_gnn.yml:107), host
//   tracking output                  relabel the detections by (id_cam, old id) -> ID_pred and write mtmc_*.txt
//                                                                        inference.py:540-551, main.py:114
// Integer work: every count is exact; floating-point metrics are derived from the counts on the host in fp64.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace mpn {

// ------------------------------------------------------------------------------------------------ confusion counts
// class of a value as the reference tests it: == 1 -> 1, == 0 -> 0, anything else -> 2 (ignored by every count)
template <typename T>
__device__ __forceinline__ int cls01(T v) { return v == (T)1 ? 1 : (v == (T)0 ? 0 : 2); }

template <typename PT, typename LT>
__global__ void __launch_bounds__(256) confusion_kernel(const PT* __restrict__ pred, const LT* __restrict__ labels, long long E,
                                                        unsigned long long* __restrict__ counts /*[3][3]: label x pred*/) {
  __shared__ unsigned int sh[9];
  if (threadIdx.x < 9) sh[threadIdx.x] = 0u;
  __syncthreads();
  unsigned int c[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    const int k = cls01(labels[e]) * 3 + cls01(pred[e]);
#pragma unroll
    for (int i = 0; i < 9; ++i) c[i] += (k == i) ? 1u : 0u;
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    unsigned int v = c[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sh[i], v);
  }
  __syncthreads();
  if (threadIdx.x < 9 && sh[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------ hash tables (open addressing)
constexpr unsigned long long EMPTY_KEY = ~0ull;
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {     // splitmix64 finaliser
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  x ^= x >> 31;
  return x;
}
// returns the slot of `key`, inserting it if absent (cap is a power of two, load factor <= 1/2)
__device__ __forceinline__ long long find_or_insert(unsigned long long* keys, long long cap, unsigned long long key) {
  long long s = (long long)(mix64(key) & (unsigned long long)(cap - 1));
  for (;;) {
    const unsigned long long cur = keys[s];
    if (cur == key) return s;
    if (cur == EMPTY_KEY) {
      const unsigned long long old = atomicCAS(&keys[s], EMPTY_KEY, key);
      if (old == EMPTY_KEY || old == key) return s;
    }
    s = (s + 1) & (cap - 1);
  }
}
__device__ __forceinline__ long long find_slot(const unsigned long long* keys, long long cap, unsigned long long key) {
  long long s = (long long)(mix64(key) & (unsigned long long)(cap - 1));
  for (;;) {
    const unsigned long long cur = keys[s];
    if (cur == key) return s;
    if (cur == EMPTY_KEY) return -1;
    s = (s + 1) & (cap - 1);
  }
}
__global__ void fill_u64_kernel(unsigned long long* p, long long n, unsigned long long v) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}

// ------------------------------------------------------------------------------------------------ contingency table
__global__ void contingency_insert_kernel(const long long* __restrict__ a, const long long* __restrict__ b, long long N, long long Ka,
                                          long long Kb, unsigned long long* keys, unsigned long long* cnt, long long cap,
                                          unsigned long long* row_sums, unsigned long long* col_sums, int* bad) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    const long long x = a[i], y = b[i];
    if (x < 0 || x >= Ka || y < 0 || y >= Kb) { *bad = 1; continue; }
    const long long s = find_or_insert(keys, cap, (unsigned long long)(x * Kb + y));
    atomicAdd(&cnt[s], 1ull);
    atomicAdd(&row_sums[x], 1ull);
    atomicAdd(&col_sums[y], 1ull);
  }
}
__global__ void contingency_compact_kernel(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ cnt,
                                           long long cap, long long Kb, long long* rows, long long* cols, long long* vals,
                                           unsigned long long* nnz) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += stride) {
    const unsigned long long k = keys[s];
    if (k == EMPTY_KEY) continue;
    const unsigned long long o = atomicAdd(nnz, 1ull);
    rows[o] = (long long)(k / (unsigned long long)Kb);
    cols[o] = (long long)(k % (unsigned long long)Kb);
    vals[o] = (long long)cnt[s];
  }
}

// ------------------------------------------------------------------------------------------------ tracking-output join
constexpr int CAM_BITS = 20, ID_BITS = 44;
__device__ __forceinline__ bool pack_key(long long cam, long long id, unsigned long long& key) {
  if (cam < 0 || cam >= (1ll << CAM_BITS) || id < 0 || id >= (1ll << ID_BITS)) return false;
  key = ((unsigned long long)cam << ID_BITS) | (unsigned long long)id;
  return true;
}
__global__ void relabel_build_kernel(const long long* __restrict__ node_cam, const long long* __restrict__ node_old, long long N,
                                     unsigned long long* keys, int* winner, long long cap, int* bad) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += stride) {
    unsigned long long key;
    if (!pack_key(node_cam[n], node_old[n], key)) { *bad = 1; continue; }
    const long long s = find_or_insert(keys, cap, key);
    atomicMax(&winner[s], (int)n);                      // the reference's loop runs n ascending: the last writer wins
  }
}
__global__ void relabel_apply_kernel(const long long* __restrict__ det_cam, const long long* __restrict__ det_id, long long M,
                                     const unsigned long long* __restrict__ keys, const int* __restrict__ winner, long long cap,
                                     const long long* __restrict__ node_new, long long* __restrict__ out_id) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += stride) {
    const long long old = det_id[r];
    unsigned long long key;
    long long s = -1;
    if (pack_key(det_cam[r], old, key)) s = find_slot(keys, cap, key);
    out_id[r] = (s >= 0) ? node_new[winner[s]] : old;   // detections of no tracklet keep their id
  }
}

static long long pow2_at_least(long long n) {
  long long c = 64;
  while (c < n) c <<= 1;
  return c;
}
static int grid_for(long long n) { return (int)std::min<long long>((long long)kNumSMs * 8, std::max<long long>(1, (n + 255) / 256)); }

}  // namespace mpn

using namespace mpn;

extern "C" {

int mpn_edge_confusion(const void* pred, int pred_kind, const void* labels, int label_kind, int64_t E, int64_t* counts_dev, void* stream) {
  MPN_REQUIRE(counts_dev && (E == 0 || (pred && labels)), "edge_confusion: NULL argument");
  MPN_REQUIRE(pred_kind >= 0 && pred_kind <= 2 && label_kind >= 0 && label_kind <= 2, "edge_confusion: kind must be 0 (uint8), 1 (int64) or 2 (float32)");
  cudaStream_t st = (cudaStream_t)stream;
  MPN_CUDA_OK(cudaMemsetAsync(counts_dev, 0, 9 * sizeof(int64_t), st));
  if (E == 0) return MPN_OK;
  unsigned long long* c = (unsigned long long*)counts_dev;
  const int grid = grid_for(E);
#define MPN_CONF(PT, LT) confusion_kernel<PT, LT><<<grid, 256, 0, st>>>((const PT*)pred, (const LT*)labels, E, c)
  switch (pred_kind * 3 + label_kind) {
    case 0: MPN_CONF(uint8_t, uint8_t); break;
    case 1: MPN_CONF(uint8_t, long long); break;
    case 2: MPN_CONF(uint8_t, float); break;
    case 3: MPN_CONF(long long, uint8_t); break;
    case 4: MPN_CONF(long long, long long); break;
    case 5: MPN_CONF(long long, float); break;
    case 6: MPN_CONF(float, uint8_t); break;
    case 7: MPN_CONF(float, long long); break;
    default: MPN_CONF(float, float); break;
  }
#undef MPN_CONF
  MPN_LAUNCH_OK();
  return MPN_OK;
}

size_t mpn_contingency_workspace_bytes(int64_t N) {
  const long long cap = pow2_at_least(2 * std::max<long long>(N, 1));
  return (size_t)cap * 16 + 1024;
}

// a, b: compact labels in [0,Ka) / [0,Kb).  Outputs: COO entries (unordered; sort on the host), nnz, marginals.  Synchronises.
int mpn_contingency(const int64_t* a_dev, const int64_t* b_dev, int64_t N, int64_t Ka, int64_t Kb, int64_t* rows_out_dev,
                    int64_t* cols_out_dev, int64_t* counts_out_dev, int64_t* nnz_host, int64_t* row_sums_dev, int64_t* col_sums_dev,
                    void* ws, size_t ws_bytes, void* stream) {
  MPN_REQUIRE(nnz_host && ws && row_sums_dev && col_sums_dev && Ka > 0 && Kb > 0 && N >= 0, "contingency: bad argument");
  MPN_REQUIRE(Ka < (1ll << 31) && Kb < (1ll << 31), "contingency: more than 2^31 classes");
  MPN_REQUIRE(ws_bytes >= mpn_contingency_workspace_bytes(N), "contingency workspace too small");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const long long cap = pow2_at_least(2 * std::max<long long>(N, 1));
  unsigned long long* keys = (unsigned long long*)ws;
  unsigned long long* cnt = keys + cap;
  unsigned long long* nnz_dev = cnt + cap;               // inside the +1024 tail
  int* bad = (int*)(nnz_dev + 1);
  fill_u64_kernel<<<grid_for(cap), 256, 0, st>>>(keys, cap, EMPTY_KEY);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaMemsetAsync(cnt, 0, (size_t)cap * 8 + 16, st));
  MPN_CUDA_OK(cudaMemsetAsync(row_sums_dev, 0, (size_t)Ka * 8, st));
  MPN_CUDA_OK(cudaMemsetAsync(col_sums_dev, 0, (size_t)Kb * 8, st));
  *nnz_host = 0;
  if (N == 0) return MPN_OK;
  MPN_REQUIRE(a_dev && b_dev && rows_out_dev && cols_out_dev && counts_out_dev, "contingency: NULL argument");
  contingency_insert_kernel<<<grid_for(N), 256, 0, st>>>((const long long*)a_dev, (const long long*)b_dev, N, Ka, Kb, keys, cnt, cap,
                                                         (unsigned long long*)row_sums_dev, (unsigned long long*)col_sums_dev, bad);
  MPN_LAUNCH_OK();
  contingency_compact_kernel<<<grid_for(cap), 256, 0, st>>>(keys, cnt, cap, Kb, (long long*)rows_out_dev, (long long*)cols_out_dev,
                                                            (long long*)counts_out_dev, nnz_dev);
  MPN_LAUNCH_OK();
  unsigned long long host[2] = {0, 0};
  MPN_CUDA_OK(cudaMemcpyAsync(host, nnz_dev, 16, cudaMemcpyDeviceToHost, st));
  MPN_CUDA_OK(cudaStreamSynchronize(st));
  MPN_REQUIRE(((const int*)&host[1])[0] == 0, "contingency: a label outside [0,Ka) x [0,Kb)");
  *nnz_host = (int64_t)host[0];
  return MPN_OK;
}

// sklearn.metrics.cluster._expected_mutual_info_fast.expected_mutual_information (0.24.2), restated; a/b = marginals.
double mpn_expected_mutual_information_host(const int64_t* a, int64_t R, const int64_t* b, int64_t C, int64_t n_samples) {
  if (!a || !b || R <= 0 || C <= 0 || n_samples <= 0) return 0.0;
  const double N = (double)n_samples;
  long long mx = 0;
  for (int64_t i = 0; i < R; ++i) mx = std::max<long long>(mx, a[i]);
  for (int64_t j = 0; j < C; ++j) mx = std::max<long long>(mx, b[j]);
  std::vector<double> term1(mx + 1), log_Nnij(mx + 1), gln_nij(mx + 1), log_a(R), log_b(C), gln_a(R), gln_b(C), gln_Na(R), gln_Nb(C);
  for (long long k = 0; k <= mx; ++k) {
    const double nij = (k == 0) ? 1.0 : (double)k;       // "stops divide by zero warnings": never used at nij = 0
    term1[k] = nij / N;
    log_Nnij[k] = log(N) + log(nij);
    gln_nij[k] = lgamma(nij + 1.0);
  }
  for (int64_t i = 0; i < R; ++i) { log_a[i] = log((double)a[i]); gln_a[i] = lgamma((double)a[i] + 1.0); gln_Na[i] = lgamma(N - (double)a[i] + 1.0); }
  for (int64_t j = 0; j < C; ++j) { log_b[j] = log((double)b[j]); gln_b[j] = lgamma((double)b[j] + 1.0); gln_Nb[j] = lgamma(N - (double)b[j] + 1.0); }
  const double gln_N = lgamma(N + 1.0);
  double emi = 0.0;
  for (int64_t i = 0; i < R; ++i) {
    for (int64_t j = 0; j < C; ++j) {
      const long long start = std::max<long long>(a[i] + b[j] - n_samples, 1), end = std::min<long long>(a[i], b[j]) + 1;
      for (long long nij = start; nij < end; ++nij) {
        const double term2 = log_Nnij[nij] - log_a[i] - log_b[j];
        const double gln = gln_a[i] + gln_b[j] + gln_Na[i] + gln_Nb[j] - gln_N - gln_nij[nij] - lgamma((double)(a[i] - nij) + 1.0) -
                           lgamma((double)(b[j] - nij) + 1.0) - lgamma((double)(n_samples - a[i] - b[j] + nij) + 1.0);
        emi += term1[nij] * term2 * exp(gln);
      }
    }
  }
  return emi;
}

size_t mpn_relabel_workspace_bytes(int64_t n_nodes) {
  const long long cap = pow2_at_least(2 * std::max<long long>(n_nodes, 1));
  return (size_t)cap * 12 + 1024;
}

// out_id[r] = node_new[n] for the LAST node n with (node_cam[n], node_old[n]) == (det_cam[r], det_id[r]); else det_id[r].
int mpn_relabel_detections(const int64_t* det_cam_dev, const int64_t* det_id_dev, int64_t M, const int64_t* node_cam_dev,
                           const int64_t* node_old_dev, const int64_t* node_new_dev, int64_t N, int64_t* out_id_dev, void* ws,
                           size_t ws_bytes, void* stream) {
  MPN_REQUIRE(ws && M >= 0 && N >= 0 && N < (1ll << 31), "relabel: bad argument");
  MPN_REQUIRE(ws_bytes >= mpn_relabel_workspace_bytes(N), "relabel workspace too small");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  if (M == 0) return MPN_OK;
  MPN_REQUIRE(det_cam_dev && det_id_dev && out_id_dev && (N == 0 || (node_cam_dev && node_old_dev && node_new_dev)), "relabel: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  const long long cap = pow2_at_least(2 * std::max<long long>(N, 1));
  unsigned long long* keys = (unsigned long long*)ws;
  int* winner = (int*)(keys + cap);
  int* bad = winner + cap;
  fill_u64_kernel<<<grid_for(cap), 256, 0, st>>>(keys, cap, EMPTY_KEY);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaMemsetAsync(winner, 0xff, (size_t)cap * 4, st));          // -1
  MPN_CUDA_OK(cudaMemsetAsync(bad, 0, 4, st));
  if (N > 0) {
    relabel_build_kernel<<<grid_for(N), 256, 0, st>>>((const long long*)node_cam_dev, (const long long*)node_old_dev, N, keys, winner, cap, bad);
    MPN_LAUNCH_OK();
  }
  relabel_apply_kernel<<<grid_for(M), 256, 0, st>>>((const long long*)det_cam_dev, (const long long*)det_id_dev, M, keys, winner, cap,
                                                    (const long long*)node_new_dev, (long long*)out_id_dev);
  MPN_LAUNCH_OK();
  int bad_host = 0;
  MPN_CUDA_OK(cudaMemcpyAsync(&bad_host, bad, 4, cudaMemcpyDeviceToHost, st));
  MPN_CUDA_OK(cudaStreamSynchronize(st));
  MPN_REQUIRE(bad_host == 0, "relabel: a tracklet has id_cam outside [0,2^%d) or id outside [0,2^%d)", CAM_BITS, ID_BITS);
  return MPN_OK;
}

// np.savetxt(path, table, fmt='%d') of main.py:114: one detection per line, columns separated by one space.  HOST pointers.
int mpn_write_mtmc_txt_host(const char* path, const int64_t* table_host, int64_t rows, int32_t cols) {
  MPN_REQUIRE(path && (rows == 0 || table_host) && cols > 0 && rows >= 0, "write_mtmc_txt: bad argument");
  FILE* f = fopen(path, "wb");
  MPN_REQUIRE(f != nullptr, "write_mtmc_txt: cannot open %s", path);
  std::vector<char> buf;
  buf.reserve(1 << 20);
  char tmp[32];
  for (int64_t r = 0; r < rows; ++r) {
    for (int32_t c = 0; c < cols; ++c) {
      long long v = table_host[r * cols + c];
      int n = 0;
      unsigned long long u = v < 0 ? (unsigned long long)(-(v + 1)) + 1ull : (unsigned long long)v;
      do { tmp[n++] = (char)('0' + u % 10); u /= 10; } while (u);
      if (v < 0) tmp[n++] = '-';
      while (n) buf.push_back(tmp[--n]);
      buf.push_back(c + 1 < cols ? ' ' : '\n');
    }
    if (buf.size() > (1 << 20) - 256) {
      if (fwrite(buf.data(), 1, buf.size(), f) != buf.size()) { fclose(f); set_error("write_mtmc_txt: short write to %s", path); return MPN_ERR_INVALID; }
      buf.clear();
    }
  }
  const bool ok = fwrite(buf.data(), 1, buf.size(), f) == buf.size();
  if (fclose(f) != 0 || !ok) { set_error("write_mtmc_txt: short write to %s", path); return MPN_ERR_INVALID; }
  return MPN_OK;
}

}  // extern "C"

// ================================================================================================
// Either side of the hot path (SURVEY.md section 8f rows 1 and 4): the graph-construction leftovers of inference.py:383-451.
//   mpn_edge_labels         edge_labels_g[e] = 1 if node_labels[row] == node_labels[col] else 0   (inference.py:446-450:
//                           an O(E*N) Python comprehension in the reference), float32, graph edge order
//   mpn_normalize_columns   F.normalize(node_embeds, p=2, dim=0) (inference.py:403-404): every FEATURE COLUMN is scaled to unit
//                           L2 norm over the nodes, eps 1e-12.  Sum of squares in fp64, then one scaling pass.
//   mpn_normalize_columns_batched   the same for every graph of a batch on its own (inference.py:403-404 per graph), one kernel.
// ================================================================================================
namespace mpn {

__global__ void __launch_bounds__(256) edge_labels_kernel(const mpn_graph g, const long long* __restrict__ node_labels,
                                                          float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n_tasks = *g.n_tasks;
  for (int t = gwarp; t < n_tasks; t += nwarps) {
    const int row = g.task_row[t];
    const int beg = g.rowptr[row] + (t - g.taskptr[row]) * g.chunk;
    const int end = min(beg + g.chunk, g.rowptr[row + 1]);
    const long long lr = node_labels[row + g.row_offset];
    for (int e = beg + lane; e < end; e += 32) out[e] = (node_labels[g.col[e]] == lr) ? 1.f : 0.f;
  }
}

constexpr int NC_SPLITS = 64;
template <typename T>
__global__ void __launch_bounds__(256) colsq_partial_kernel(const T* __restrict__ x, int n, int D, int rows_per_split,
                                                            double* __restrict__ part /*[NC_SPLITS][D]*/) {
  __shared__ double ssum[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  const int r0 = blockIdx.y * rows_per_split, r1 = min(r0 + rows_per_split, n);
  double s = 0.0;
  if (col < D)
    for (int r = r0 + ry; r < r1; r += 8) { const double v = to_f32(x[(size_t)r * D + col]); s += v * v; }
  ssum[ry][cx] = s;
  __syncthreads();
  if (ry == 0 && col < D) {
    for (int i = 1; i < 8; ++i) s += ssum[i][cx];
    part[(size_t)blockIdx.y * D + col] = s;
  }
}
__global__ void colnorm_finalize_kernel(const double* __restrict__ part, int D, float* __restrict__ norm_out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= D) return;
  double s = 0.0;
  for (int i = 0; i < NC_SPLITS; ++i) s += part[(size_t)i * D + col];
  const float nrm = fmaxf((float)sqrt(s), 1e-12f);                 // F.normalize: v / max(||v||_2, eps)
  norm_out[col] = nrm;
}
template <typename T>
__global__ void colnorm_apply_kernel(const T* __restrict__ x, long long total, int D, const float* __restrict__ norm,
                                     float* __restrict__ out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) out[i] = to_f32(x[i]) / norm[i % D];
}


// mpn_normalize_columns_batched: F.normalize(dim=0) of every graph of a batch alone.  One CTA per (graph, slab of sw columns);
// thread (ry, cx) sums the squares of column cx over the graph's rows ry, ry + 256/sw, ... in fp64, then the 256/sw partials are
// added in order (deterministic).  Pass 2 re-reads the slab, which is still in L2 (300 rows x 32 columns = 38 KB at S02 size), and
// writes it scaled.  A CTA writes only the slab it has finished summing, so out may alias x (no __restrict__).
template <typename T>
__global__ void __launch_bounds__(256) colnorm_graph_kernel(const T* x, int D, const int* __restrict__ graph_nptr, int sw,
                                                            float* out) {
  __shared__ double part[256];
  __shared__ float nrm[32];
  const int cx = threadIdx.x % sw, ry = threadIdx.x / sw, nry = 256 / sw;
  const int col = blockIdx.y * sw + cx;
  const int r0 = graph_nptr[blockIdx.x], r1 = graph_nptr[blockIdx.x + 1];
  double s = 0.0;
  if (col < D) {
#pragma unroll 4
    for (int r = r0 + ry; r < r1; r += nry) { const double v = to_f32(x[(size_t)r * D + col]); s += v * v; }
  }
  part[threadIdx.x] = s;
  __syncthreads();
  if (ry == 0) {
    for (int i = 1; i < nry; ++i) s += part[i * sw + cx];
    nrm[cx] = fmaxf((float)sqrt(s), 1e-12f);                       // F.normalize: v / max(||v||_2, eps)
  }
  __syncthreads();
  if (col < D) {
    const float q = nrm[cx];
#pragma unroll 4
    for (int r = r0 + ry; r < r1; r += nry) out[(size_t)r * D + col] = to_f32(x[(size_t)r * D + col]) / q;
  }
}

}  // namespace mpn

extern "C" {

int mpn_edge_labels(const mpn_graph* g, const int64_t* node_labels_dev, float* out_dev, void* stream) {
  MPN_REQUIRE(g && (g->n_edges == 0 || (node_labels_dev && out_dev)), "edge_labels: NULL argument");
  if (g->n_edges == 0) return MPN_OK;
  edge_labels_kernel<<<kNumSMs * 8, 256, 0, (cudaStream_t)stream>>>(*g, (const long long*)node_labels_dev, out_dev);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

size_t mpn_normalize_columns_workspace_bytes(int32_t D) { return (size_t)NC_SPLITS * D * sizeof(double) + (size_t)D * sizeof(float) + 512; }

int mpn_normalize_columns_x(const void* x_dev, int32_t x_kind, int32_t n, int32_t D, float* out_dev, void* ws, size_t ws_bytes,
                            void* stream) {
  MPN_X_KIND_OK(x_kind);
  MPN_REQUIRE(n >= 0 && D > 0 && ws, "normalize_columns: bad argument");
  MPN_REQUIRE(ws_bytes >= mpn_normalize_columns_workspace_bytes(D), "normalize_columns workspace too small");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  if (n == 0) return MPN_OK;
  MPN_REQUIRE(x_dev && out_dev, "normalize_columns: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  double* part = (double*)ws;
  float* norm = (float*)(part + (size_t)NC_SPLITS * D);
  const long long total = (long long)n * D;
  return with_x_type(x_kind, [&](auto xt) {
    colsq_partial_kernel<<<dim3(div_up(D, 32), NC_SPLITS), 256, 0, st>>>((decltype(xt))x_dev, n, D, div_up(n, NC_SPLITS), part);
    MPN_LAUNCH_OK();
    colnorm_finalize_kernel<<<div_up(D, 128), 128, 0, st>>>(part, D, norm);
    MPN_LAUNCH_OK();
    colnorm_apply_kernel<<<grid_for(total), 256, 0, st>>>((decltype(xt))x_dev, total, D, norm, out_dev);
    MPN_LAUNCH_OK();
    return MPN_OK;
  });
}

int mpn_normalize_columns(const float* x_dev, int32_t n, int32_t D, float* out_dev, void* ws, size_t ws_bytes, void* stream) {
  return mpn_normalize_columns_x(x_dev, MPN_X_F32, n, D, out_dev, ws, ws_bytes, stream);
}

int mpn_normalize_columns_batched_x(const void* x_dev, int32_t x_kind, int32_t n, int32_t D, const int32_t* graph_nptr_dev,
                                    int32_t n_graphs, float* out_dev, void* ws, size_t ws_bytes, void* stream) {
  if (n_graphs <= 1) return mpn_normalize_columns_x(x_dev, x_kind, n, D, out_dev, ws, ws_bytes, stream);
  MPN_X_KIND_OK(x_kind);
  MPN_REQUIRE(n > 0 && D > 0, "normalize_columns_batched: bad argument");
  MPN_REQUIRE(x_dev && out_dev && graph_nptr_dev, "normalize_columns_batched: NULL argument");
  MPN_REQUIRE(div_up(D, 8) <= 65535, "normalize_columns_batched: D must be <= 524280");
  // 32-column slabs (one 128-byte line per warp row); a batch of few graphs gets narrower slabs so that about one wave of
  // CTAs (8 per SM) is in flight
  int sw = 32;
  while (sw > 8 && (long long)n_graphs * div_up(D, sw) < kNumSMs * 8) sw >>= 1;
  return with_x_type(x_kind, [&](auto xt) {
    colnorm_graph_kernel<<<dim3(n_graphs, div_up(D, sw)), 256, 0, (cudaStream_t)stream>>>((decltype(xt))x_dev, D, graph_nptr_dev, sw, out_dev);
    MPN_LAUNCH_OK();
    return MPN_OK;
  });
}

int mpn_normalize_columns_batched(const float* x_dev, int32_t n, int32_t D, const int32_t* graph_nptr_dev, int32_t n_graphs,
                                  float* out_dev, void* ws, size_t ws_bytes, void* stream) {
  return mpn_normalize_columns_batched_x(x_dev, MPN_X_F32, n, D, graph_nptr_dev, n_graphs, out_dev, ws, ws_bytes, stream);
}

}  // extern "C"
