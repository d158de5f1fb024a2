// K1: initial edge features (inference.py:453-456)
//   edge_attr[e] = [ ||x_r - x_c + eps||_2 , 1 - cos(x_r, x_c) ],  eps = 1e-6 (F.pairwise_distance), cos eps = 1e-8
// via the Gram matrix of the CENTRED features x' = x - mean_row(x)  (distances are translation invariant, and ReID
// embeddings share a large common component that would otherwise dominate the cancellation):
//   ||a - b + eps||^2 = |a'|^2 + |b'|^2 - 2 a'.b' + 2 eps (sum a' - sum b') + D eps^2
//   a.b = a'.b' + mu.a' + mu.b' + |mu|^2 ,   cos = a.b / max(|a||b|, 1e-8)
// The reference gathers two [E,D] copies (8 KB per edge each); here the only per-edge traffic is one Gram read and
// one 8-byte write.  Pairs whose squared distance still cancels (d^2 < 25% of |a'|^2+|b'|^2: same-identity pairs)
// are recomputed directly from the rows, exactly as the reference sums them.
#include <string.h>

#include "common.cuh"
#include "kernels.h"

namespace mpn {

// column means of x [n, D] (fp64 accumulation): grid (32-column tiles, row splits) -> partials -> fixed-order finalize
constexpr int CM_SPLITS = 32;
template <typename T>
__global__ void __launch_bounds__(256) col_mean_partial_kernel(const T* __restrict__ x, int n, int D, int rows_per_split,
                                                               double* __restrict__ part /*[CM_SPLITS][D]*/) {
  pdl_wait();
  __shared__ double ssum[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  const int r0 = blockIdx.y * rows_per_split, r1 = min(r0 + rows_per_split, n);
  double s = 0.0;
  if (col < D)
    for (int r = r0 + ry; r < r1; r += 8) s += to_f32(x[(size_t)r * D + col]);
  ssum[ry][cx] = s;
  __syncthreads();
  if (ry == 0 && col < D) {
    for (int i = 1; i < 8; ++i) s += ssum[i][cx];
    part[(size_t)blockIdx.y * D + col] = s;
  }
}
__global__ void col_mean_finalize_kernel(const double* __restrict__ part, int n, int D, float* __restrict__ mu) {
  pdl_wait();
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= D) return;
  double s = 0.0;
  for (int i = 0; i < CM_SPLITS; ++i) s += part[(size_t)i * D + col];
  mu[col] = (float)(s / n);
}

// xc = x - mu; per-row statistics of the centred row (accumulated in fp64, stored as one float4 = one 16-byte gather
// per edge; the Gram entry they are combined with is itself only fp32-accurate): st[r] = {|a'|^2, sum a', mu.a' + |mu|^2/2, |a|}
template <typename T>
__global__ void __launch_bounds__(256) center_rows_kernel(const T* __restrict__ x, const float* __restrict__ mu, int n, int D,
                                                          float* __restrict__ xc, float4* __restrict__ st,
                                                          unsigned int* __restrict__ amax_bits, const int* __restrict__ run_flag) {
  pdl_wait();
  if (run_flag != nullptr && *run_flag == 0) return;
  const int lane = threadIdx.x & 31;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int r = gwarp; r < n; r += nwarps) {
    const T* p = x + (size_t)r * D;
    float* q = xc + (size_t)r * D;
    double sq = 0.0, sx = 0.0, md = 0.0, mm = 0.0;
    float amax = 0.f;
    for (int k = lane; k < D; k += 32) {
      const float m = mu[k];
      const float c = to_f32(p[k]) - m;
      q[k] = c;
      amax = fmaxf(amax, fabsf(c));
      sq += (double)c * c;
      sx += (double)c;
      md += (double)m * c;
      mm += (double)m * m;
    }
    sq = warp_sum(sq); sx = warp_sum(sx); md = warp_sum(md); mm = warp_sum(mm);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if (lane == 0 && amax_bits) atomicMax(amax_bits, __float_as_uint(amax));      // non-negative floats order like their bits
    if (lane == 0) {
      // a.b = g' + (mu.a' + |mu|^2/2) + (mu.b' + |mu|^2/2);  |a| = sqrt(|a'|^2 + 2 mu.a' + |mu|^2)
      st[r] = make_float4((float)sq, (float)sx, (float)(md + 0.5 * mm), (float)sqrt(fmax(sq + 2.0 * md + mm, 0.0)));
    }
  }
}

// batched graphs: offsets of the per-graph ng x ng Gram blocks (single thread; G <= 65535)
__global__ void gram_offsets_kernel(const int* __restrict__ graph_nptr, int n_graphs, long long* __restrict__ g_off) {
  pdl_wait();
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  long long run = 0;
  for (int i = 0; i < n_graphs; ++i) {
    g_off[i] = run;
    const long long ng = graph_nptr[i + 1] - graph_nptr[i];
    run += ng * ng;
  }
  g_off[n_graphs] = run;
}

// fp32 fallback for the block-diagonal Gram (tests / shapes the tensor-core kernel does not take): one warp per row
__global__ void __launch_bounds__(256) gram_blockdiag_simt_kernel(const float* __restrict__ X, int N, int K, const int* __restrict__ node_gid,
                                                                  const int* __restrict__ graph_nptr, const long long* __restrict__ g_off,
                                                                  float* __restrict__ Gbuf) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int r = gwarp; r < N; r += nwarps) {
    const int gi = node_gid[r];
    const int base = graph_nptr[gi], ng = graph_nptr[gi + 1] - base;
    float* out = Gbuf + g_off[gi] + (size_t)(r - base) * ng;
    const float* a = X + (size_t)r * K;
    for (int c = 0; c < ng; ++c) {
      const float* b = X + (size_t)(base + c) * K;
      float s = 0.f;
      for (int k = lane; k < K; k += 32) s = fmaf(a[k], b[k], s);
      s = warp_sum(s);
      if (lane == 0) out[c] = s;
    }
  }
}

// one warp per task (a run of edges of one row): coalesced Gram reads when the row's columns are consecutive.
// run_flag (optional): nothing to do when *run_flag == 0 (the fused kernel of gram_ef.cu wrote the features itself)
__global__ void __launch_bounds__(256) edge_feature_gather_kernel(const mpn_graph g, int r0, int r1, const float* __restrict__ G,
                                                                  const long long* __restrict__ g_off,
                                                                  const float4* __restrict__ st, int D,
                                                                  float2* __restrict__ edge_attr,
                                                                  int* __restrict__ refine_list, int* __restrict__ refine_count,
                                                                  const int* __restrict__ run_flag) {
  pdl_wait();
  if (run_flag != nullptr && *run_flag == 0) return;
#include "edge_feature_gather.inc"
}

// direct recomputation for the flagged pairs (one warp per pair), fp32 elementwise like ATen
// fixed_sums (optional, with the fused kernel only): the moment sums (a, b, aa, ab, bb) of the recomputed pairs are added as
// 2^40 fixed point integers, so the total does not depend on the order in which the list was filled
template <typename T>
__global__ void __launch_bounds__(256) edge_feature_refine_kernel(const mpn_graph g, const T* __restrict__ x, int D,
                                                                  const int* __restrict__ refine_list,
                                                                  const int* __restrict__ refine_count,
                                                                  float2* __restrict__ edge_attr,
                                                                  unsigned long long* __restrict__ fixed_sums,
                                                                  const int* __restrict__ not_one_gap, const GeShare sh) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int n = *refine_count;
  const bool with_sums = fixed_sums != nullptr && not_one_gap != nullptr && *not_one_gap == 0;
  // shared Gram (kernels.h): a listed pair is one this rank computed for both directions; the mirrored entry goes to the owner
  const bool shared = sh.mode != nullptr && *sh.mode == 2 && not_one_gap != nullptr && *not_one_gap == 0;
  for (int i = gwarp; i < n; i += nwarps) {
    const int e = refine_list[i];
    int lo = 0, hi = g.n_nodes;                       // row = last r with rowptr[r] <= e
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (g.rowptr[mid] <= e) lo = mid; else hi = mid;
    }
    const int cnode = g.col[e];
    const T* a = x + (size_t)(lo + g.row_offset) * D;
    const T* b = x + (size_t)cnode * D;
    double d2 = 0.0, d2m = 0.0, ab = 0.0, aa = 0.0, bb = 0.0;
    for (int k = lane; k < D; k += 32) {
      const float av = to_f32(a[k]), bv = to_f32(b[k]);
      const float df = av - bv + PAIRWISE_EPS;
      const float dfm = bv - av + PAIRWISE_EPS;
      d2 += (double)df * df;
      d2m += (double)dfm * dfm;
      ab += (double)av * bv;
      aa += (double)av * av;
      bb += (double)bv * bv;
    }
    d2 = warp_sum(d2); ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
    if (shared) d2m = warp_sum(d2m);
    if (lane == 0) {
      const double denom = fmax(sqrt(aa) * sqrt(bb), (double)COSINE_EPS);
      const float2 o = make_float2((float)sqrt(d2), (float)(1.0 - ab / denom));
      edge_attr[e] = o;
      const double sc = 1099511627776.0;                              // 2^40
      if (with_sums) {
        const double fa = o.x, fb = o.y;
        atomicAdd(fixed_sums + 0, (unsigned long long)__double2ll_rn(fa * sc));
        atomicAdd(fixed_sums + 1, (unsigned long long)__double2ll_rn(fb * sc));
        atomicAdd(fixed_sums + 2, (unsigned long long)__double2ll_rn(fa * fa * sc));
        atomicAdd(fixed_sums + 3, (unsigned long long)__double2ll_rn(fa * fb * sc));
        atomicAdd(fixed_sums + 4, (unsigned long long)__double2ll_rn(fb * fb * sc));
      }
      if (shared) {                                                   // (cnode -> row) in the shard of cnode's owner
        int owner = 0;
        while (owner + 1 < sh.world && cnode >= sh.blk[owner + 1]) ++owner;
        const int4 te = sh.tab[sh.rank][cnode];                       // (edge base, gap start, gap length) of row cnode
        const int rnode = lo + g.row_offset;
        const float2 om = make_float2((float)sqrt(d2m), o.y);
        sh.ea[owner][te.x + rnode - (rnode >= te.y + te.z ? te.z : 0)] = om;
        if (with_sums) {
          const double fa = om.x, fb = om.y;
          atomicAdd(fixed_sums + 0, (unsigned long long)__double2ll_rn(fa * sc));
          atomicAdd(fixed_sums + 1, (unsigned long long)__double2ll_rn(fb * sc));
          atomicAdd(fixed_sums + 2, (unsigned long long)__double2ll_rn(fa * fa * sc));
          atomicAdd(fixed_sums + 3, (unsigned long long)__double2ll_rn(fa * fb * sc));
          atomicAdd(fixed_sums + 4, (unsigned long long)__double2ll_rn(fb * fb * sc));
        }
      }
    }
  }
}

struct EfLayout {
  float4* st;
  float *mu, *xc;
  double* mu_part;
  float* G;
  int *refine_list, *refine_count;
  unsigned int* amax_bits;         // max |x'| over the centred features (float bits): scale of the fp16 operand planes
  unsigned int* mu_ticket;         // last-block ticket of the column-mean kernel
  long long* g_off;
  void* gemm_ws;
  size_t gemm_ws_bytes;
  int rows_per_block;
  int2* gap;                       // fused distance epilogue: one-gap table of the rows
  int* not_one_gap;
  int* share_mode;
  GeWorkspace ge;                  // planes / records / tile list of the fused kernel (gram_ef.cu)
  bool fused_possible;
  size_t total;
};

static EfLayout ef_layout(const mpn_graph* g, int D, void* ws, size_t ws_bytes) {
  EfLayout L;
  Arena a(ws, ws_bytes);
  L.st = a.take<float4>((size_t)g->n_cols);
  L.mu = a.take<float>(D);
  L.mu_part = a.take<double>((size_t)(ge_col_mean_splits() > CM_SPLITS ? ge_col_mean_splits() : CM_SPLITS) * D);
  L.xc = a.take<float>((size_t)g->n_cols * D);
  const bool batched = g->n_graphs > 1 && g->node_gid && g->graph_nptr;
  const size_t budget = (size_t)2 << 30;
  size_t rows = budget / ((size_t)g->n_cols * sizeof(float));
  if (rows < 128) rows = 128;
  if (rows > (size_t)g->n_nodes) rows = g->n_nodes;
  L.rows_per_block = (int)rows;
  // batched: block-diagonal Gram, sum of ng^2 <= max_graph_nodes * N entries
  L.G = a.take<float>(batched ? (size_t)g->max_graph_nodes * g->n_cols : rows * (size_t)g->n_cols);
  L.g_off = a.take<long long>((size_t)(batched ? g->n_graphs : 0) + 1);
  L.refine_list = a.take<int>((size_t)(g->n_edges > 0 ? g->n_edges : 1));
  L.refine_count = a.take<int>(1);
  L.amax_bits = a.take<unsigned int>(1);
  L.mu_ticket = a.take<unsigned int>(64);                    // one per 128-column tile (D <= 8192)
  L.not_one_gap = a.take<int>(1);
  L.share_mode = a.take<int>(1);                             // GeShare::mode (adjacent: cleared by the same memset)
  L.gemm_ws_bytes = batched ? gemm_tc_workspace_bytes(1, g->n_cols, D) : gemm_tc_workspace_bytes((int)rows, g->n_cols, D);
  L.gemm_ws = L.gemm_ws_bytes ? (void*)a.take<char>(L.gemm_ws_bytes) : nullptr;
  L.gap = a.take<int2>((size_t)(g->n_nodes > 0 ? g->n_nodes : 1));
  L.fused_possible = !batched && gram_ef_shape_ok(g->n_nodes, g->n_cols, D);
  memset(&L.ge, 0, sizeof(L.ge));
  if (L.fused_possible) {
    ge_workspace_layout(g->n_cols, g->n_nodes, D, &L.ge, ws ? (char*)ws + a.off : nullptr, ws ? (ws_bytes > a.off ? ws_bytes - a.off : 0) : 0);
    a.off += L.ge.total;
  }
  L.total = a.off;
  return L;
}

// the two launches of edge_features_impl that read x, instantiated for its element type
static int center_rows(const void* x, int x_kind, const EfLayout& L, int n, int D, const int* run_flag, cudaStream_t st) {
  return with_x_type(x_kind, [&](auto xt) {
    mpn::launch(center_rows_kernel<x_elem_t<decltype(xt)>>, min(kNumSMs * 8, div_up((long long)n * 32, 256)), 256, 0,
                st, (decltype(xt))x, L.mu, n, D, L.xc, L.st, L.amax_bits, run_flag);
    MPN_LAUNCH_OK();
    return MPN_OK;
  });
}
static int refine_pairs(const mpn_graph& g, const void* x, int x_kind, int D, const EfLayout& L, float2* edge_attr,
                        unsigned long long* fixed_sums, const int* not_one_gap, const GeShare& sh, cudaStream_t st) {
  return with_x_type(x_kind, [&](auto xt) {
    mpn::launch(edge_feature_refine_kernel<x_elem_t<decltype(xt)>>, kNumSMs * 4, 256, 0, st, g, (decltype(xt))x, D,
                L.refine_list, L.refine_count, edge_attr, fixed_sums, not_one_gap, sh);
    MPN_LAUNCH_OK();
    return MPN_OK;
  });
}

// moments (optional): the caller wants the first encoder BatchNorm's moment sums taken on the way (mpn_forward_with_edge_features).
//   partials   [>= 148][MPN_SUMS_DOUBLES] zeroed by the caller; the fused kernel writes one row per CTA
//   fixed_sums [5] zeroed by the caller; the refine pass adds the recomputed pairs' share as 2^40 fixed point
//   handled    out: device flag, 0 = the fused kernel produced features AND moments, != 0 = the caller must sweep edge_attr itself;
//              nullptr when that is already known on the host (known_fused tells which)
int edge_features_impl(const mpn_graph* g, const void* x, int x_kind, int32_t D, float* edge_attr, int use_tc, void* ws,
                       size_t ws_bytes, cudaStream_t st, EfMoments* moments, const GeShare* share) {
  MPN_REQUIRE(g && x && D > 0 && ws, "edge_features: NULL argument");
  MPN_X_KIND_OK(x_kind);
  MPN_REQUIRE(edge_attr || g->n_edges == 0, "edge_features: NULL output");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  EfLayout L = ef_layout(g, D, ws, ws_bytes);
  if (L.total > ws_bytes) {
    set_error("edge_features workspace too small: need %zu bytes, have %zu", L.total, ws_bytes);
    return MPN_ERR_WORKSPACE;
  }
  if (moments) { moments->handled_flag = nullptr; moments->known_fused = 0; }
  if (g->n_edges == 0) return MPN_OK;
  MPN_CUDA_OK(cudaMemsetAsync(L.refine_count, 0, 5 * 256, st));        // refine_count, amax_bits, mean ticket, not_one_gap, share mode (adjacent slices)
  if ((D % 4) == 0 && D <= 8192 && x_vec4_aligned(x, x_kind)) {          // (64 ticket slots: one per 128-column tile)
    MPN_TRY(ge_col_mean(x, x_kind, g->n_cols, D, L.mu_part, L.mu_ticket, L.mu, st));
  } else {
    MPN_TRY(with_x_type(x_kind, [&](auto xt) {
      mpn::launch(col_mean_partial_kernel<x_elem_t<decltype(xt)>>, dim3(div_up(D, 32), CM_SPLITS), 256, 0, st,
                  (decltype(xt))x, g->n_cols, D, div_up(g->n_cols, CM_SPLITS), L.mu_part);
      MPN_LAUNCH_OK();
      return MPN_OK;
    }));
    mpn::launch(col_mean_finalize_kernel, div_up(D, 128), 128, 0, st, L.mu_part, g->n_cols, D, L.mu);
    MPN_LAUNCH_OK();
  }
  if (g->n_graphs > 1 && g->node_gid && g->graph_nptr) {
    // batched small graphs: block-diagonal Gram (one ng x ng block per graph), gather epilogue
    MPN_TRY(center_rows(x, x_kind, L, g->n_cols, D, nullptr, st));
    MPN_REQUIRE(g->row_offset == 0 && g->n_cols == g->n_nodes && g->max_graph_nodes > 0, "batched edge features: bad graph");
    mpn::launch(gram_offsets_kernel, 1, 32, 0, st, g->graph_nptr, g->n_graphs, L.g_off);
    MPN_LAUNCH_OK();
    if (use_tc && gemm_tc_supported(g->n_cols, 64, D) && g->n_graphs <= 65535) {
      MPN_TRY(gram_blockdiag_tc(L.xc, g->n_cols, D, g->graph_nptr, L.g_off, g->n_graphs, g->max_graph_nodes, L.G, L.gemm_ws,
                                L.gemm_ws_bytes, st, (const float*)L.amax_bits));
    } else {
      mpn::launch(gram_blockdiag_simt_kernel, kNumSMs * 8, 256, 0, st, L.xc, g->n_cols, D, g->node_gid, g->graph_nptr, L.g_off, L.G);
      MPN_LAUNCH_OK();
    }
    mpn::launch(edge_feature_gather_kernel, kNumSMs * 8, 256, 0, st, *g, 0, g->n_nodes, L.G, L.g_off, L.st, D, (float2*)edge_attr, L.refine_list,
                                                           L.refine_count, (const int*)nullptr);
    MPN_LAUNCH_OK();
    return refine_pairs(*g, x, x_kind, D, L, (float2*)edge_attr, nullptr, nullptr, GeShare{}, st);
  }
  // Dense cross-camera graphs (every row = all columns but one gap; verified on the device unless the builder of the graph
  // vouches for it through g->layout_hint): the features are formed in the epilogue of the Gram GEMM (gram_ef.cu).  Any other
  // graph: Gram block in HBM + gather.  With an unknown layout both sets of launches are enqueued, each kernel tests the
  // device flag first and one set returns at once.
  const bool fused = use_tc && L.fused_possible && (((uintptr_t)x) & 15) == 0;     // (16-byte cp.async of the rows)
  const bool known_one_gap = fused && g->layout_hint == MPN_LAYOUT_ONE_GAP;
  GeShare sh;
  memset(&sh, 0, sizeof(sh));
  if (share != nullptr) {
    MPN_REQUIRE(fused, "shared Gram needs the fused edge-feature path (tensor cores, D a multiple of 64)");
    sh = *share;
    sh.mode = L.share_mode;
  }
  const int* run_gather = nullptr;                   // old path: unconditional
  if (fused) {
    int n_rows = 0;
    MPN_TRY(gram_ef_run(x, x_kind, L.mu, g, D, L.gap, L.not_one_gap, (float2*)edge_attr, L.refine_list, L.refine_count,
                        moments ? moments->partials : nullptr, &n_rows, L.ge, st, share ? &sh : nullptr));
    if (moments) { moments->handled_flag = L.not_one_gap; moments->known_fused = known_one_gap ? 1 : 0; }
    run_gather = L.not_one_gap;
  }
  if (!known_one_gap) {
    MPN_TRY(center_rows(x, x_kind, L, g->n_cols, D, run_gather, st));
    for (int r0 = 0; r0 < g->n_nodes; r0 += L.rows_per_block) {
      const int r1 = min(r0 + L.rows_per_block, g->n_nodes);
      const float* Ablk = L.xc + (size_t)(g->row_offset + r0) * D;
      if (use_tc && gemm_tc_supported(r1 - r0, g->n_cols, D))
        MPN_TRY(gram_nt_tc(L.xc, g->row_offset + r0, L.G, r1 - r0, g->n_cols, D, (const float*)L.amax_bits, L.gemm_ws, L.gemm_ws_bytes, st, run_gather));
      else
        MPN_TRY(gemm_nt_simt(Ablk, L.xc, nullptr, nullptr, nullptr, L.G, r1 - r0, g->n_cols, D, st));
      mpn::launch(edge_feature_gather_kernel, kNumSMs * 8, 256, 0, st, *g, r0, r1, L.G, (const long long*)nullptr, L.st, D, (float2*)edge_attr,
                                                             L.refine_list, L.refine_count, run_gather);
      MPN_LAUNCH_OK();
    }
  }
  return refine_pairs(*g, x, x_kind, D, L, (float2*)edge_attr, moments ? moments->fixed_sums : nullptr,
                      fused ? L.not_one_gap : nullptr, sh, st);
}

}  // namespace mpn

using namespace mpn;

extern "C" {

// tests / bench: which way the last mpn_forward_sharded_with_edge_features on this workspace went (synchronises the stream):
// 2 = shared symmetric Gram, 0 = every rank its own rows, -1 = error
int mpn_shared_gram_mode(const mpn_graph* g, int32_t D, const void* ws, size_t ws_bytes, void* stream) {
  if (g == nullptr || ws == nullptr) return -1;
  mpn::EfLayout L = mpn::ef_layout(g, D, const_cast<void*>(ws), ws_bytes);
  if (L.total > ws_bytes) return -1;
  int mode = -1;
  if (cudaMemcpyAsync(&mode, L.share_mode, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess) return -1;
  if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) return -1;
  return mode;
}

size_t mpn_edge_features_workspace_bytes(const mpn_graph* g, int32_t D) {
  if (!g || D <= 0) return 0;
  return ef_layout(g, D, nullptr, 0).total + 256;
}

int mpn_edge_features_x(const mpn_graph* g, const void* x, int32_t x_kind, int32_t D, float* edge_attr, int use_tc, void* ws,
                        size_t ws_bytes, void* stream) {
  return mpn::edge_features_impl(g, x, x_kind, D, edge_attr, use_tc, ws, ws_bytes, (cudaStream_t)stream, nullptr);
}

int mpn_edge_features(const mpn_graph* g, const float* x, int32_t D, float* edge_attr, int use_tc, void* ws, size_t ws_bytes,
                      void* stream) {
  return mpn_edge_features_x(g, x, MPN_X_F32, D, edge_attr, use_tc, ws, ws_bytes, stream);
}

}  // extern "C"
