// Internal (non-ABI) declarations shared between the translation units of libmpn_b200.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace mpn {

// edge features (inference.py:453-456): eps of F.pairwise_distance / F.cosine_similarity, and the cancellation threshold below
// which a pair is recomputed directly from its two rows (edge_features.cu)
constexpr float PAIRWISE_EPS = 1e-6f;
constexpr float COSINE_EPS = 1e-8f;
constexpr float REFINE_FRACTION = 0.25f;

// gemm_tc.cu: 2-D tiled tensor map over a row-major [rows, K] plane (fp32: 32-element boxes, fp16: 64-element boxes = 128 bytes)
int make_tma_map_2d(CUtensorMap* map, const void* base, int rows, int K, int box_rows, bool f16);

// gram_ef.cu: edge features of a dense cross-camera graph in the epilogue of the Gram GEMM (every kernel is a no-op when
// *not_one_gap != 0).  partials: optional [n_partial_rows][MPN_SUMS_DOUBLES] block partial rows of the first encoder BatchNorm's
// moment sums (columns 0..4 = sum a, b, aa, ab, bb over the edges that were NOT sent to the refine list).
struct GeWorkspace {
  uint16_t *hi, *lo;          // [n_cols, D] fp16 planes of the centred, per-row scaled features
  float4* rec;                // [n_cols]
  float* scale_inv;           // [n_cols]
  int *tiles, *n_tiles;
  size_t total;
};
// Row-block shards that share ONE symmetric Gram (sharded forward, N > 1): every unordered pair of nodes is computed by exactly one
// rank, which stores the direct entry into its own edge_attr and the mirrored entry into the OWNER's edge_attr over NVLink.
// Pair (r in block R, c in block S) is computed by R iff  S == R: r < c;  else with d = (S - R) mod W:  2d < W: always,
// 2d > W: never, 2d == W (antipodal blocks): R < S ? c < mid(S) : r >= mid(R)   (mid = middle of the block: both ranks do half).
// Each rank first pushes (edge base, gap start, gap length, its not_one_gap flag) of its rows into every rank's node table; the
// shared mode is used only if every rank's rows are dense cross-camera rows, otherwise every rank falls back to its own rows.
struct GeShare {
  int rank, world;
  int blk[MPN_MAX_PEERS + 1];                 // row blocks: rank r owns nodes [blk[r], blk[r+1])
  float2* ea[MPN_MAX_PEERS];                  // peer-visible edge_attr of every rank ([E_r] float2)
  int4* tab[MPN_MAX_PEERS];                   // peer-visible node table [n_cols] of every rank (each rank holds a full copy)
  unsigned long long* flags[MPN_MAX_PEERS];   // flag block of every rank; word [3][src] = node-table sequence
  unsigned long long seq;                     // this call's sequence number
  int* mode;                                  // device word in the caller's workspace: 2 = shared, 0 = every rank its own rows
};
int ge_workspace_layout(int n_cols, int M, int D, GeWorkspace* L, void* ws, size_t ws_bytes);
bool gram_ef_shape_ok(int M, int N, int D);
// column means of x [n, D] (fp64 partial sums, fixed order): part [ge_col_mean_splits()][D] doubles, *ticket zeroed once
int ge_col_mean_splits();
// x: node features of element kind x_kind (MPN_X_*), read in place here and in gram_ef_run / edge_features_impl
int ge_col_mean(const void* x, int x_kind, int n, int D, double* part, unsigned int* ticket, float* mu, cudaStream_t st);
// fills gap / *not_one_gap (zeroed by the caller) for the rows of g, then runs the fused kernels
int gram_ef_run(const void* x, int x_kind, const float* mu, const mpn_graph* g, int D, int2* gap, int* not_one_gap, float2* edge_attr,
                int* refine_list, int* refine_count, double* partials, int* n_partial_rows, const GeWorkspace& L, cudaStream_t st,
                const GeShare* share = nullptr);

// edge_features.cu
struct EfMoments {                 // in: partials [>= kNumSMs][MPN_SUMS_DOUBLES] and fixed_sums [5], both zeroed by the caller
  double* partials;
  unsigned long long* fixed_sums;
  const int* handled_flag;         // out: device flag, 0 = features AND moments came from the fused kernel (nullptr: gather path)
  int known_fused;                 // out: 1 = the host already knows the fused kernel ran (the graph's layout hint)
};
int edge_features_impl(const mpn_graph* g, const void* x, int x_kind, int32_t D, float* edge_attr, int use_tc, void* ws, size_t ws_bytes,
                       cudaStream_t st, EfMoments* moments, const GeShare* share = nullptr);   // share->mode is set here

// gemm_simt.cu
// a_kind: element kind of A (MPN_X_*; layer 0 of the node encoder reads x in place)
int gemm_nt_simt(const void* A, const float* B, const float* bias, const float* a_scale, const float* a_shift,
                 float* C, int M, int N, int K, cudaStream_t st, const int* row_gid = nullptr, int a_kind = MPN_X_F32);

// gemm_tc.cu  (tcgen05 3xTF32; operands are pre-split hi/lo planes)
size_t gemm_tc_workspace_bytes(int M, int N, int K);
// a_scale/a_shift (optional, [K]): A is read as relu(A*scale + shift) while it is split (fused BatchNorm+ReLU)
int gemm_nt_tc(const void* A, const float* B, const float* bias, float* C, int M, int N, int K,
               void* workspace, size_t workspace_bytes, cudaStream_t st, const float* a_scale = nullptr,
               const float* a_shift = nullptr, const float* b_hi_cached = nullptr, const float* b_lo_cached = nullptr,
               const int* row_gid = nullptr,    // row_gid: a_scale/a_shift are [n_graphs][K] tables indexed by the row's graph
               int a_kind = MPN_X_F32);         // element kind of A (MPN_X_*)
int split_tf32(const float* x, long long n, float* hi, float* lo, cudaStream_t st);
// Gram block of the row block [a_row0, a_row0+M) of X [N,K] against all of X: 3xFP16 planes scaled by max|X| (amax_dev: float
// bits on the device) when K % 8 == 0, else / when amax_dev is NULL the TF32 path of gemm_nt_tc
// run_flag (optional, device): the launches return at once when *run_flag == 0
int gram_nt_tc(const float* X, int a_row0, float* C, int M, int N, int K, const float* amax_dev, void* workspace, size_t workspace_bytes,
               cudaStream_t st, const int* run_flag = nullptr);
bool gemm_tc_supported(int M, int N, int K);
// 3xFP16 variant for the node encoder: A is split here into fp16 planes (fused BatchNorm+ReLU; plane scale from a_amax_host, or
// measured on the device when a_amax_host <= 0), B planes (b_hi16/b_lo16, scaled by b_scale) are cached by the caller
int gemm_nt_tc_f16(const void* A, const float* bias, float* C, int M, int N, int K, void* workspace, size_t workspace_bytes,
                   cudaStream_t st, const float* a_scale, const float* a_shift, const int* row_gid, float a_amax_host,
                   const void* b_hi16, const void* b_lo16, float b_scale, int a_kind = MPN_X_F32);
int split_f16_host_scale(const float* x, long long n, float amax, void* hi, void* lo, float* scale_out, cudaStream_t st);
int gram_blockdiag_tc(const float* X, int N, int K, const int* graph_nptr, const long long* g_off, int n_graphs, int max_ng,
                      float* Gbuf, void* ws, size_t ws_bytes, cudaStream_t st, const float* amax_dev = nullptr);

}  // namespace mpn
