// K5: CUTTING / PRUNING / SPLITTING and strongly-connected-component labelling on the GPU.
// Reference: inference.post_processing (inference.py:70-169) and utils.py:30-52, 54-123, 125-142, 144-339.
//
// All stages work on an order-preserving compaction of the active edges (A << E): one pass over the
// 1-byte activity flags, then every fixed-point round touches only A entries plus O(N) node arrays.
// Integer / index results are bit-exact by construction: counts use integer atomics, arg-min uses a
// packed (prob bits, edge id) 64-bit atomicMin (ties -> lowest edge id, as torch.argmin over ascending
// candidates, utils.py:288-289), components use min-id union-find.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "common.cuh"

namespace mpn {

constexpr int EPB = 4096;            // edges per compaction block (256 threads x 16 flags)
constexpr unsigned int HASH_EMPTY = 0xFFFFFFFFu;

// Which graph a node belongs to and that graph's camera count (PRUNE bounds degrees by it minus one, SPLIT cluster sizes by it).
// A batch reads node_gid and the per-graph counts on the device; gid == nullptr is one graph, graph 0 with ncam1 cameras, with no
// load.  The single-graph entry points pass that view for any table, so a batch given to them is one disjoint-union graph.
struct Graphs {
  const int* gid;
  const int* ncam;
  int ncam1;
  __device__ __forceinline__ int graph_of(int n) const { return gid ? gid[n] : 0; }
  __device__ __forceinline__ int limit_of(int n) const { return gid ? ncam[gid[n]] : ncam1; }
};
static Graphs one_graph(int num_cameras) { return Graphs{nullptr, nullptr, num_cameras}; }

struct PostCtx {
  mpn_graph g;
  cudaStream_t st;
  int n_blocks;
  // device
  int *blockoff, *a_eid, *a_src, *a_dst, *a_rev;
  int *fo, *fi, *label, *size, *od_src, *od_dst, *counters;      // counters[8]
  int *dirty_nodes, *dirty_edges;                                // SPLIT: nodes of oversized clusters, active-list entries touching them
  unsigned long long *mo, *mi;
  unsigned int* mbits;
  unsigned long long* hash;                                      // SPLIT: the dropped minima, keyed by (graph id, probability bits)
  int hash_cap;
  int *wcc, *wccflag;                                            // SPLIT: weakly connected components and the flagged ones
  unsigned long long* tie_keys;                                  // SPLIT: (graph id, probability) of the dirty edges ...
  int* tie_counts;                                               // ... and how many active edges of that graph carry each
  int tie_cap;
  float* a_prob;                                                 // SPLIT: probabilities in active-list order
  uint8_t *sel, *tiedb;                                          // SPLIT: entry selected for the host; value carried by >= 2 active edges
  int *a_gptr, *gflag, *groots;      // first active-list entry per graph [G+1]; SPLIT host-order flag per graph [G] + tied-edge count
                                     // (one copy to the host); SCC count per graph [G]
  size_t total;
  // host
  int n_active;
};

static void post_layout(PostCtx& c, void* ws, size_t ws_bytes) {
  Arena a(ws, ws_bytes);
  const size_t E = (size_t)(c.g.n_edges > 0 ? c.g.n_edges : 1), N = (size_t)c.g.n_nodes;
  c.n_blocks = div_up((long long)E, EPB);
  c.blockoff = a.take<int>(c.n_blocks + 1);
  c.a_eid = a.take<int>(E);
  c.a_src = a.take<int>(E);
  c.a_dst = a.take<int>(E);
  c.a_rev = a.take<int>(E);
  c.od_src = a.take<int>(E);
  c.od_dst = a.take<int>(E);
  c.dirty_nodes = a.take<int>(N);
  c.dirty_edges = a.take<int>(E);
  c.fo = a.take<int>(N);
  c.fi = a.take<int>(N);
  c.label = a.take<int>(N);
  c.size = a.take<int>(N);
  c.mo = a.take<unsigned long long>(N);
  c.mi = a.take<unsigned long long>(N);
  c.mbits = a.take<unsigned int>(N);
  int cap = 1024;
  while ((size_t)cap < N) cap <<= 1;
  c.hash_cap = cap;
  // the SPLIT sets key (graph id, probability bits) for one graph too: 8 B a slot where a value-only set would take 4, which at
  // configs[3] (1 M nodes, ~92 M edges) is ~138 MB more, and one set of kernels serves one graph and a batch
  c.hash = a.take<unsigned long long>(cap);
  c.wcc = a.take<int>(N);
  c.wccflag = a.take<int>(N);
  int tcap = 1024;
  while ((size_t)tcap < E / 4) tcap <<= 1;
  c.tie_cap = tcap;
  c.tie_keys = a.take<unsigned long long>(tcap);
  c.tie_counts = a.take<int>(tcap);
  c.a_prob = a.take<float>(E);
  c.sel = a.take<uint8_t>(E);
  c.tiedb = a.take<uint8_t>(E);
  c.counters = a.take<int>(16);
  const size_t G = (size_t)std::max(1, c.g.n_graphs);
  c.a_gptr = a.take<int>(G + 1);
  c.gflag = a.take<int>(G + 1);
  c.groots = a.take<int>(G);
  c.total = a.off;
}

// ------------------------------------------------------------------------------------------------
// order-preserving compaction of active edges
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) count_active_kernel(const uint8_t* __restrict__ act, long long E, int* __restrict__ blockcnt) {
  __shared__ int wsum[8];
  const long long base = (long long)blockIdx.x * EPB + (long long)threadIdx.x * 16;
  int cnt = 0;
  if (base + 16 <= E && (((uintptr_t)act) & 15) == 0) {
    const uint4 v = *reinterpret_cast<const uint4*>(act + base);
    const unsigned int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int b = 0; b < 4; ++b) cnt += ((w[i] >> (8 * b)) & 0xFFu) != 0;
  } else {
    for (int i = 0; i < 16; ++i)
      if (base + i < E) cnt += act[base + i] != 0;
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int i = 0; i < 8; ++i) s += wsum[i];
    blockcnt[blockIdx.x] = s;
  }
}

// single-block exclusive scan (in place) + total
__global__ void __launch_bounds__(1024) scan_blocks_kernel(int* __restrict__ v, int n, int* __restrict__ total) {
  __shared__ int strip[1024];
  const int t = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int lo = min(t * per, n), hi = min(lo + per, n);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += v[i];
  strip[t] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    int x = (t >= off) ? strip[t - off] : 0;
    __syncthreads();
    strip[t] += x;
    __syncthreads();
  }
  int run = (t == 0) ? 0 : strip[t - 1];
  for (int i = lo; i < hi; ++i) { const int x = v[i]; v[i] = run; run += x; }
  if (t == 1023) { v[n] = strip[1023]; *total = strip[1023]; }
}

__device__ __forceinline__ int find_row(const int* __restrict__ rowptr, int n_rows, int e) {
  int lo = 0, hi = n_rows;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (rowptr[mid] <= e) lo = mid; else hi = mid;
  }
  return lo;
}
// index of edge (u -> v) or -1; columns are sorted within a row
__device__ __forceinline__ int find_edge(const mpn_graph& g, int u, int v) {
  int lo = g.rowptr[u], hi = g.rowptr[u + 1];
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int c = g.col[mid];
    if (c == v) return mid;
    if (c < v) lo = mid + 1; else hi = mid;
  }
  return -1;
}

// SHARD: row-block graph (global src = row_offset + local row), no reverse-edge lookup (the reverse edge lives on another rank),
// the edge's probability is compacted along
template <bool SHARD>
__global__ void __launch_bounds__(256) write_active_kernel(const mpn_graph g, const uint8_t* __restrict__ act,
                                                           const int* __restrict__ blockoff, int* __restrict__ a_eid,
                                                           int* __restrict__ a_src, int* __restrict__ a_dst, int* __restrict__ a_rev,
                                                           const float* __restrict__ prob, int pstride, float* __restrict__ a_prob) {
  __shared__ int tsum[256];
  const long long E = g.n_edges;
  const long long base = (long long)blockIdx.x * EPB + (long long)threadIdx.x * 16;
  unsigned int mask = 0;
  for (int i = 0; i < 16; ++i)
    if (base + i < E && act[base + i] != 0) mask |= 1u << i;
  const int cnt = __popc(mask);
  tsum[threadIdx.x] = cnt;
  __syncthreads();
  for (int off = 1; off < 256; off <<= 1) {
    int x = (threadIdx.x >= off) ? tsum[threadIdx.x - off] : 0;
    __syncthreads();
    tsum[threadIdx.x] += x;
    __syncthreads();
  }
  int pos = blockoff[blockIdx.x] + tsum[threadIdx.x] - cnt;
  while (mask) {
    const int i = __ffs(mask) - 1;
    mask &= mask - 1;
    const int e = (int)(base + i);
    const int u = find_row(g.rowptr, g.n_nodes, e);
    const int v = g.col[e];
    a_eid[pos] = e;
    a_dst[pos] = v;
    if (SHARD) {
      a_src[pos] = g.row_offset + u;
      a_prob[pos] = prob[(size_t)e * pstride];
    } else {
      a_src[pos] = u;
      a_rev[pos] = find_edge(g, v, u);
    }
    ++pos;
  }
}

static int build_active_list(PostCtx& c, const uint8_t* act) {
  if (c.g.n_edges == 0) { c.n_active = 0; return MPN_OK; }
  count_active_kernel<<<c.n_blocks, 256, 0, c.st>>>(act, c.g.n_edges, c.blockoff);
  MPN_LAUNCH_OK();
  scan_blocks_kernel<<<1, 1024, 0, c.st>>>(c.blockoff, c.n_blocks, c.counters);
  MPN_LAUNCH_OK();
  write_active_kernel<false><<<c.n_blocks, 256, 0, c.st>>>(c.g, act, c.blockoff, c.a_eid, c.a_src, c.a_dst, c.a_rev, nullptr, 0, nullptr);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaMemcpyAsync(&c.n_active, c.counters, sizeof(int), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  return MPN_OK;
}

static inline int list_grid(int n) { return std::max(1, std::min(kNumSMs * 8, div_up(n, 256))); }

// ------------------------------------------------------------------------------------------------
// CUT (utils.py:125-142): an active edge survives only if its reverse is active
// ------------------------------------------------------------------------------------------------
__global__ void cut_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_rev, uint8_t* __restrict__ act) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    const int e = a_eid[i];
    if (!act[e]) continue;
    const int r = a_rev[i];
    // race-free in place: act[e] is only read by the thread owning rev(e), which exists only while act[rev(e)] == 1,
    // and in that case act[e] is not cleared here
    if (r < 0 || !act[r]) act[e] = 0;
  }
}

// ------------------------------------------------------------------------------------------------
// PRUNE (utils.py:161-188, 277-317)
// ------------------------------------------------------------------------------------------------
__global__ void flow_count_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                  const uint8_t* __restrict__ act, int* __restrict__ fo, int* __restrict__ fi) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    if (!act[a_eid[i]]) continue;
    atomicAdd(&fo[a_src[i]], 1);
    atomicAdd(&fi[a_dst[i]], 1);
  }
}
// the bound of a node is the camera count of its graph minus one (an edge's endpoints lie in one graph)
__global__ void prune_pick_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                  const uint8_t* __restrict__ act, const float* __restrict__ prob, int pstride, const Graphs graphs,
                                  const int* __restrict__ fo, const int* __restrict__ fi, unsigned long long* __restrict__ mo,
                                  unsigned long long* __restrict__ mi, int* __restrict__ any_violation) {
  bool viol = false;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    const int e = a_eid[i];
    if (!act[e]) continue;
    const int u = a_src[i], v = a_dst[i];
    const int limit = graphs.limit_of(u) - 1;
    const bool bo = fo[u] > limit, bi = fi[v] > limit;
    if (!(bo || bi)) continue;
    viol = true;
    const unsigned long long key = ((unsigned long long)__float_as_uint(prob[(size_t)e * pstride]) << 32) | (unsigned int)e;
    if (bo) atomicMin(&mo[u], key);
    if (bi) atomicMin(&mi[v], key);
  }
  if (viol) *any_violation = 1;
}
__global__ void prune_remove_kernel(int N, const unsigned long long* __restrict__ mo, const unsigned long long* __restrict__ mi,
                                    uint8_t* __restrict__ act) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
    const unsigned long long a = mo[n], b = mi[n];
    if (a != ~0ull) act[(unsigned int)(a & 0xFFFFFFFFull)] = 0;
    if (b != ~0ull) act[(unsigned int)(b & 0xFFFFFFFFull)] = 0;
  }
}

__global__ void prune_reset_kernel(int N, int* __restrict__ fo, int* __restrict__ fi, unsigned long long* __restrict__ mo,
                                   unsigned long long* __restrict__ mi) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
    fo[n] = 0; fi[n] = 0; mo[n] = ~0ull; mi[n] = ~0ull;
  }
}

// Rounds are enqueued PRUNE_BATCH at a time with one flag word each and the host reads the flags once per batch: a round without
// a violating node removes nothing, so the rounds enqueued past the fixed point are no-ops (the violation flags of a batch are a
// prefix of ones).  One host round trip per 8 rounds instead of one per round (the smoke graph needs 87 rounds).
// In a batch a graph that has converged sees no-op rounds while the others go on.
constexpr int PRUNE_BATCH = 8;
static int prune_stage(PostCtx& c, uint8_t* act, const float* prob, int pstride, const Graphs& graphs, int* changed, int* rounds) {
  const int A = c.n_active, N = c.g.n_nodes;
  *changed = 0;
  *rounds = 0;
  if (A == 0) return MPN_OK;
  int* flags = c.counters + 8;                          // PRUNE_BATCH flag words
  for (;;) {
    MPN_CUDA_OK(cudaMemsetAsync(flags, 0, sizeof(int) * PRUNE_BATCH, c.st));
    for (int r = 0; r < PRUNE_BATCH; ++r) {
      prune_reset_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.fo, c.fi, c.mo, c.mi);
      MPN_LAUNCH_OK();
      flow_count_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.fo, c.fi);
      MPN_LAUNCH_OK();
      prune_pick_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, prob, pstride, graphs, c.fo, c.fi, c.mo,
                                                        c.mi, flags + r);
      MPN_LAUNCH_OK();
      prune_remove_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.mo, c.mi, act);
      MPN_LAUNCH_OK();
    }
    int viol[PRUNE_BATCH];
    MPN_CUDA_OK(cudaMemcpyAsync(viol, flags, sizeof(int) * PRUNE_BATCH, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaStreamSynchronize(c.st));
    int n_viol = 0;
    while (n_viol < PRUNE_BATCH && viol[n_viol]) ++n_viol;
    *rounds += n_viol;
    if (n_viol > 0) *changed = 1;
    if (n_viol < PRUNE_BATCH) break;
  }
  return MPN_OK;
}

// ------------------------------------------------------------------------------------------------
// SCC: min-id union-find over mutual edges, then (rarely) a host Tarjan on the condensed digraph of the
// remaining one-directional edges.  Every mutual-edge component lies inside one SCC, so the condensation
// is exact.  label[n] = smallest node id of n's SCC.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int uf_find(int* __restrict__ parent, int x) {
  int p = parent[x];
  while (p != x) {
    const int gp = parent[p];
    if (gp != p) parent[x] = gp;          // path halving (benign race: only ever points closer to the root)
    x = p;
    p = gp;
  }
  return x;
}
__device__ __forceinline__ void uf_union(int* __restrict__ parent, int a, int b) {
  for (;;) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }      // hook the larger root under the smaller one
    if (atomicCAS(&parent[a], a, b) == a) return;
  }
}
__global__ void iota_kernel(int N, int* __restrict__ v) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) v[n] = n;
}
__global__ void union_mutual_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                    const int* __restrict__ a_rev, const uint8_t* __restrict__ act, int* __restrict__ parent) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    if (!act[a_eid[i]]) continue;
    const int u = a_src[i], v = a_dst[i];
    if (u >= v) continue;                               // the (v,u) twin handles u > v
    const int r = a_rev[i];
    if (r >= 0 && act[r]) uf_union(parent, u, v);
  }
}
__global__ void flatten_kernel(int N, int* __restrict__ parent, int* __restrict__ n_roots) {
  int roots = 0;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
    int x = n;
    while (parent[x] != x) x = parent[x];
    roots += (x == n);
    // safe without a second buffer: roots never change in this kernel and only non-root entries are rewritten to roots
    if (x != n) parent[n] = x;
  }
  if (n_roots) {
    roots = __reduce_add_sync(0xffffffffu, roots);
    if ((threadIdx.x & 31) == 0 && roots) atomicAdd(n_roots, roots);
  }
}
__global__ void one_dir_edges_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                     const int* __restrict__ a_rev, const uint8_t* __restrict__ act, const int* __restrict__ label,
                                     int* __restrict__ od_src, int* __restrict__ od_dst, int* __restrict__ od_count) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    if (!act[a_eid[i]]) continue;
    const int r = a_rev[i];
    if (r >= 0 && act[r]) continue;
    const int lu = label[a_src[i]], lv = label[a_dst[i]];
    if (lu == lv) continue;
    const int slot = atomicAdd(od_count, 1);
    od_src[slot] = lu;
    od_dst[slot] = lv;
  }
}
__global__ void hook_pairs_kernel(int n, const int* __restrict__ from, const int* __restrict__ to, int* __restrict__ parent) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) parent[from[i]] = to[i];
}

// iterative Tarjan on a small digraph given as edge arrays over arbitrary ids; returns (id -> min id of its SCC) for
// every id that belongs to an SCC with more than one member
static void host_condensed_scc(const std::vector<int>& s, const std::vector<int>& d, std::vector<int>& from, std::vector<int>& to) {
  std::unordered_map<int, int> idx;
  std::vector<int> ids;
  auto get = [&](int v) {
    auto it = idx.find(v);
    if (it != idx.end()) return it->second;
    const int k = (int)ids.size();
    idx.emplace(v, k);
    ids.push_back(v);
    return k;
  };
  const size_t m = s.size();
  std::vector<int> us(m), vs(m);
  for (size_t i = 0; i < m; ++i) { us[i] = get(s[i]); vs[i] = get(d[i]); }
  const int n = (int)ids.size();
  std::vector<int> ptr(n + 1, 0), adj(m);
  for (size_t i = 0; i < m; ++i) ptr[us[i] + 1]++;
  for (int i = 0; i < n; ++i) ptr[i + 1] += ptr[i];
  {
    std::vector<int> cur(ptr.begin(), ptr.end() - 1);
    for (size_t i = 0; i < m; ++i) adj[cur[us[i]]++] = vs[i];
  }
  std::vector<int> index(n, -1), low(n, 0), cursor(n, 0), stack, call;
  std::vector<char> on(n, 0);
  int counter = 0;
  for (int root = 0; root < n; ++root) {
    if (index[root] >= 0) continue;
    call.push_back(root);
    while (!call.empty()) {
      const int v = call.back();
      if (index[v] < 0) { index[v] = low[v] = counter++; stack.push_back(v); on[v] = 1; cursor[v] = ptr[v]; }
      bool descended = false;
      while (cursor[v] < ptr[v + 1]) {
        const int w = adj[cursor[v]++];
        if (index[w] < 0) { call.push_back(w); descended = true; break; }
        if (on[w]) low[v] = std::min(low[v], index[w]);
      }
      if (descended) continue;
      call.pop_back();
      if (!call.empty()) low[call.back()] = std::min(low[call.back()], low[v]);
      if (low[v] == index[v]) {
        std::vector<int> comp;
        for (;;) {
          const int w = stack.back();
          stack.pop_back();
          on[w] = 0;
          comp.push_back(w);
          if (w == v) break;
        }
        if (comp.size() > 1) {
          int mn = ids[comp[0]];
          for (int w : comp) mn = std::min(mn, ids[w]);
          for (int w : comp)
            if (ids[w] != mn) { from.push_back(ids[w]); to.push_back(mn); }
        }
      }
    }
  }
}

// labels into c.label; n_components optional
static int scc_stage(PostCtx& c, const uint8_t* act, int* n_components) {
  const int A = c.n_active, N = c.g.n_nodes;
  iota_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.label);
  MPN_LAUNCH_OK();
  if (A > 0) {
    union_mutual_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, c.a_rev, act, c.label);
    MPN_LAUNCH_OK();
  }
  MPN_CUDA_OK(cudaMemsetAsync(c.counters + 2, 0, 2 * sizeof(int), c.st));
  flatten_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.label, c.counters + 2);
  MPN_LAUNCH_OK();
  if (A > 0) {
    one_dir_edges_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, c.a_rev, act, c.label, c.od_src, c.od_dst,
                                                         c.counters + 3);
    MPN_LAUNCH_OK();
  }
  int h[2] = {0, 0};
  MPN_CUDA_OK(cudaMemcpyAsync(h, c.counters + 2, 2 * sizeof(int), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  int n_comp = h[0];
  const int n_od = h[1];
  if (n_od > 0) {
    std::vector<int> s(n_od), d(n_od), from, to;
    MPN_CUDA_OK(cudaMemcpyAsync(s.data(), c.od_src, sizeof(int) * n_od, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(d.data(), c.od_dst, sizeof(int) * n_od, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaStreamSynchronize(c.st));
    host_condensed_scc(s, d, from, to);
    if (!from.empty()) {
      const int k = (int)from.size();
      // reuse od buffers for the (root -> new root) pairs
      MPN_CUDA_OK(cudaMemcpyAsync(c.od_src, from.data(), sizeof(int) * k, cudaMemcpyHostToDevice, c.st));
      MPN_CUDA_OK(cudaMemcpyAsync(c.od_dst, to.data(), sizeof(int) * k, cudaMemcpyHostToDevice, c.st));
      hook_pairs_kernel<<<list_grid(k), 256, 0, c.st>>>(k, c.od_src, c.od_dst, c.label);
      MPN_LAUNCH_OK();
      flatten_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.label, nullptr);
      MPN_LAUNCH_OK();
      MPN_CUDA_OK(cudaStreamSynchronize(c.st));      // host vectors must outlive the copies
      n_comp -= k;
    }
  }
  if (n_components) *n_components = n_comp;
  return MPN_OK;
}

// ------------------------------------------------------------------------------------------------
// SPLIT (utils.py:54-123) as parallel rounds: every oversized SCC contributes the minimum probability among the
// active edges touching it (either endpoint, utils.py:71); every edge of its graph whose probability equals one of those
// values is deactivated (float equality, utils.py:96-98); repeat until no SCC has more than C nodes.
// The reference removes the edges of ITS graph only, so in a batch a value shared by two different graphs must neither couple
// them nor count as a tie: the sets below are keyed by (graph id, probability bits).
// ------------------------------------------------------------------------------------------------
__global__ void comp_size_kernel(int N, const int* __restrict__ label, int* __restrict__ size) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) atomicAdd(&size[label[n]], 1);
}
__device__ __forceinline__ unsigned int hash_u32(unsigned int x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
constexpr unsigned long long HASH64_EMPTY = ~0ull;         // never a key: graph ids are < 2^31
__device__ __forceinline__ unsigned long long graph_value_key(int g, unsigned int bits) {
  return ((unsigned long long)(unsigned int)g << 32) | bits;
}
__device__ __forceinline__ unsigned int hash_u64(unsigned long long k) {
  return hash_u32((unsigned int)k ^ hash_u32((unsigned int)(k >> 32) + 0x9e3779b9u));
}
__device__ __forceinline__ void set64_insert(unsigned long long* __restrict__ t, int cap, unsigned long long key) {
  unsigned int slot = hash_u64(key) & (cap - 1);
  for (;;) {
    const unsigned long long old = atomicCAS(&t[slot], HASH64_EMPTY, key);
    if (old == HASH64_EMPTY || old == key) return;
    slot = (slot + 1) & (cap - 1);
  }
}
__device__ __forceinline__ int set64_find(const unsigned long long* __restrict__ t, int cap, unsigned long long key) {
  unsigned int slot = hash_u64(key) & (cap - 1);
  for (;;) {
    const unsigned long long v = t[slot];
    if (v == key) return (int)slot;
    if (v == HASH64_EMPTY) return -1;
    slot = (slot + 1) & (cap - 1);
  }
}

// ---- list-restricted rounds: after the first round only the nodes of oversized clusters ("dirty") and the active
// edges touching them can change the outcome, so every later round works on those two lists only.
// skip (optional): graphs whose clusters are left out (they went through the reference order on the host)
__global__ void mark_dirty_nodes_kernel(int N, const int* __restrict__ label, const int* __restrict__ size, const Graphs graphs,
                                        const int* __restrict__ skip, int* __restrict__ list, int* __restrict__ count) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x)
    if ((skip == nullptr || !skip[graphs.graph_of(n)]) && size[label[n]] > graphs.limit_of(n)) list[atomicAdd(count, 1)] = n;
}
__global__ void mark_dirty_edges_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                        const uint8_t* __restrict__ act, const int* __restrict__ label, const int* __restrict__ size,
                                        const Graphs graphs, const int* __restrict__ skip, int* __restrict__ list, int* __restrict__ count) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    if (!act[a_eid[i]]) continue;
    const int u = a_src[i];
    if (skip != nullptr && skip[graphs.graph_of(u)]) continue;
    const int limit = graphs.limit_of(u);
    if (size[label[u]] > limit || size[label[a_dst[i]]] > limit) list[atomicAdd(count, 1)] = i;
  }
}
__global__ void reset_nodes_kernel(int n_list, const int* __restrict__ list, int* __restrict__ label, int* __restrict__ size,
                                   unsigned int* __restrict__ mbits, int what) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int n = list[k];
    if (what & 1) label[n] = n;
    if (what & 2) size[n] = 0;
    if (what & 4) mbits[n] = HASH_EMPTY;
  }
}
__global__ void union_mutual_list_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ a_eid,
                                         const int* __restrict__ a_src, const int* __restrict__ a_dst, const int* __restrict__ a_rev,
                                         const uint8_t* __restrict__ act, int* __restrict__ parent) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int i = list[k];
    if (!act[a_eid[i]]) continue;
    const int u = a_src[i], v = a_dst[i];
    if (u >= v) continue;
    const int r = a_rev[i];
    if (r >= 0 && act[r]) uf_union(parent, u, v);
  }
}
__global__ void flatten_list_kernel(int n_list, const int* __restrict__ list, int* __restrict__ parent) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int n = list[k];
    int x = n;
    while (parent[x] != x) x = parent[x];
    if (x != n) parent[n] = x;
  }
}
__global__ void one_dir_edges_list_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ a_eid,
                                          const int* __restrict__ a_src, const int* __restrict__ a_dst, const int* __restrict__ a_rev,
                                          const uint8_t* __restrict__ act, const int* __restrict__ label, int* __restrict__ od_src,
                                          int* __restrict__ od_dst, int* __restrict__ od_count) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int i = list[k];
    if (!act[a_eid[i]]) continue;
    const int r = a_rev[i];
    if (r >= 0 && act[r]) continue;
    const int lu = label[a_src[i]], lv = label[a_dst[i]];
    if (lu == lv) continue;
    const int slot = atomicAdd(od_count, 1);
    od_src[slot] = lu;
    od_dst[slot] = lv;
  }
}
__global__ void comp_size_list_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ label, int* __restrict__ size) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) atomicAdd(&size[label[list[k]]], 1);
}
__global__ void split_min_list_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ a_eid, const int* __restrict__ a_src,
                                      const int* __restrict__ a_dst, const uint8_t* __restrict__ act, const float* __restrict__ prob,
                                      int pstride, const int* __restrict__ label, const int* __restrict__ size, const Graphs graphs,
                                      unsigned int* __restrict__ mbits) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int i = list[k];
    const int e = a_eid[i];
    if (!act[e]) continue;
    const int u = a_src[i];
    const int lu = label[u], lv = label[a_dst[i]];
    const int limit = graphs.limit_of(u);
    const unsigned int pb = __float_as_uint(prob[(size_t)e * pstride]);
    if (size[lu] > limit) atomicMin(&mbits[lu], pb);
    if (lv != lu && size[lv] > limit) atomicMin(&mbits[lv], pb);
  }
}
__global__ void split_collect_list_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ label,
                                          const int* __restrict__ size, const Graphs graphs, const unsigned int* __restrict__ mbits,
                                          unsigned long long* __restrict__ hash, int cap, int* __restrict__ n_big) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int n = list[k];
    if (label[n] != n || size[n] <= graphs.limit_of(n)) continue;
    atomicAdd(n_big, 1);
    const unsigned int bits = mbits[n];
    if (bits == HASH_EMPTY) continue;
    set64_insert(hash, cap, graph_value_key(graphs.graph_of(n), bits));
  }
}
// every active edge of a graph whose probability equals one of that graph's dropped minima (utils.py:96-98)
__global__ void split_remove_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const Graphs graphs,
                                    uint8_t* __restrict__ act, const float* __restrict__ prob, int pstride,
                                    const unsigned long long* __restrict__ hash, int cap) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    const int e = a_eid[i];
    if (!act[e]) continue;
    if (set64_find(hash, cap, graph_value_key(graphs.graph_of(a_src[i]), __float_as_uint(prob[(size_t)e * pstride]))) >= 0) act[e] = 0;
  }
}

// SCC restricted to the dirty lists (labels of clean nodes are left alone; they cannot become oversized)
static int scc_dirty(PostCtx& c, const uint8_t* act, int Dn, int De) {
  reset_nodes_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label, c.size, c.mbits, 1);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaMemsetAsync(c.counters + 3, 0, sizeof(int), c.st));
  if (De > 0) {
    union_mutual_list_kernel<<<list_grid(De), 256, 0, c.st>>>(De, c.dirty_edges, c.a_eid, c.a_src, c.a_dst, c.a_rev, act, c.label);
    MPN_LAUNCH_OK();
  }
  flatten_list_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label);
  MPN_LAUNCH_OK();
  if (De > 0) {
    one_dir_edges_list_kernel<<<list_grid(De), 256, 0, c.st>>>(De, c.dirty_edges, c.a_eid, c.a_src, c.a_dst, c.a_rev, act, c.label,
                                                             c.od_src, c.od_dst, c.counters + 3);
    MPN_LAUNCH_OK();
  }
  int n_od = 0;
  MPN_CUDA_OK(cudaMemcpyAsync(&n_od, c.counters + 3, sizeof(int), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  static const bool dbg = getenv("MPN_POST_DEBUG") != nullptr;
  if (dbg) fprintf(stderr, "[scc_dirty] one-directional inter-component edges: %d\n", n_od);
  if (n_od > 0) {
    std::vector<int> s(n_od), d(n_od), from, to;
    MPN_CUDA_OK(cudaMemcpyAsync(s.data(), c.od_src, sizeof(int) * n_od, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(d.data(), c.od_dst, sizeof(int) * n_od, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaStreamSynchronize(c.st));
    host_condensed_scc(s, d, from, to);
    if (!from.empty()) {
      const int k = (int)from.size();
      MPN_CUDA_OK(cudaMemcpyAsync(c.od_src, from.data(), sizeof(int) * k, cudaMemcpyHostToDevice, c.st));
      MPN_CUDA_OK(cudaMemcpyAsync(c.od_dst, to.data(), sizeof(int) * k, cudaMemcpyHostToDevice, c.st));
      hook_pairs_kernel<<<list_grid(k), 256, 0, c.st>>>(k, c.od_src, c.od_dst, c.label);
      MPN_LAUNCH_OK();
      flatten_list_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label);
      MPN_LAUNCH_OK();
      MPN_CUDA_OK(cudaStreamSynchronize(c.st));
    }
  }
  return MPN_OK;
}

// ---- probability ties -------------------------------------------------------------------------------------------------
// The rounds above equal the reference's one-cluster-at-a-time loop exactly when no probability value that an oversized
// cluster can drop is carried by a second active edge of its graph: the reference removes EVERY edge with that value
// (utils.py:96-98), so a shared value couples two clusters and the order in which the reference visits them (utils.py:60-64,112)
// decides the outcome.  Ties are detected on the device; a graph that has one goes through the exact order on the host
// (split_exact.cu), restricted to the weakly connected components that SPLITTING can touch.
//   table: open addressing over (graph, probability bits) of the active edges touching oversized clusters ("dirty" edges);
//   count: how many active edges of the same graph carry each of those values.
__global__ void tie_insert_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ a_eid, const int* __restrict__ a_src,
                                  const Graphs graphs, const uint8_t* __restrict__ act, const float* __restrict__ prob, int pstride,
                                  unsigned long long* __restrict__ keys, int cap) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) {
    const int i = list[k];
    const int e = a_eid[i];
    if (!act[e]) continue;
    set64_insert(keys, cap, graph_value_key(graphs.graph_of(a_src[i]), __float_as_uint(prob[(size_t)e * pstride])));
  }
}
__global__ void tie_count_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const Graphs graphs,
                                 const uint8_t* __restrict__ act, const float* __restrict__ prob, int pstride,
                                 const unsigned long long* __restrict__ keys, int* __restrict__ counts, int cap) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    const int e = a_eid[i];
    if (!act[e]) continue;
    const int slot = set64_find(keys, cap, graph_value_key(graphs.graph_of(a_src[i]), __float_as_uint(prob[(size_t)e * pstride])));
    if (slot >= 0) atomicAdd(&counts[slot], 1);
  }
}
// weakly connected components: union-find over every active edge
__global__ void union_all_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                 const uint8_t* __restrict__ act, int* __restrict__ parent) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x)
    if (act[a_eid[i]]) uf_union(parent, a_src[i], a_dst[i]);
}
// flag the components SPLITTING can touch: those holding an oversized cluster, those holding an edge with a tied value; and the
// graphs that have a tie (gtied)
__global__ void flag_wcc_nodes_kernel(int n_list, const int* __restrict__ list, const int* __restrict__ wcc, int* __restrict__ flag) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) flag[wcc[list[k]]] = 1;
}
__global__ void flag_wcc_ties_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const Graphs graphs,
                                     const uint8_t* __restrict__ act, const float* __restrict__ prob, int pstride,
                                     const unsigned long long* __restrict__ keys, const int* __restrict__ counts, int cap,
                                     const int* __restrict__ wcc, int* __restrict__ flag, uint8_t* __restrict__ tiedb,
                                     int* __restrict__ gtied, int* __restrict__ n_tied_edges) {
  int tied = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    const int e = a_eid[i];
    uint8_t t = 0;
    if (act[e]) {
      const int g = graphs.graph_of(a_src[i]);
      const int slot = set64_find(keys, cap, graph_value_key(g, __float_as_uint(prob[(size_t)e * pstride])));
      if (slot >= 0 && counts[slot] >= 2) { flag[wcc[a_src[i]]] = 1; gtied[g] = 1; ++tied; t = 1; }
    }
    tiedb[i] = t;
  }
  tied = __reduce_add_sync(0xffffffffu, tied);
  if ((threadIdx.x & 31) == 0 && tied) atomicAdd(n_tied_edges, tied);
}
__global__ void flag_graphs_of_nodes_kernel(int n_list, const int* __restrict__ list, const Graphs graphs, int* __restrict__ gflag) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_list; k += gridDim.x * blockDim.x) gflag[graphs.graph_of(list[k])] = 1;
}
// per active-list entry: probability (compacted) and whether its component is flagged (activity included)
__global__ void gather_select_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const uint8_t* __restrict__ act,
                                     const float* __restrict__ prob, int pstride, const int* __restrict__ wcc, const int* __restrict__ flag,
                                     float* __restrict__ a_prob, uint8_t* __restrict__ sel) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    const int e = a_eid[i];
    a_prob[i] = prob[(size_t)e * pstride];
    sel[i] = (act[e] && flag[wcc[a_src[i]]]) ? 1 : 0;
  }
}
// a_gptr[g] = first active-list entry at or after the first edge of graph g (a_eid ascends); a_gptr[G] = A
__global__ void active_graph_ptr_kernel(int G, const int* __restrict__ rowptr, const int* __restrict__ nptr, const int* __restrict__ a_eid,
                                        int A, int* __restrict__ a_gptr) {
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g <= G; g += gridDim.x * blockDim.x) {
    const int e0 = rowptr[nptr[g]];
    int lo = 0, hi = A;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (a_eid[mid] < e0) lo = mid + 1; else hi = mid;
    }
    a_gptr[g] = lo;
  }
}

// grow-only pinned host buffer of the calling thread (never freed: no CUDA calls from static destructors)
struct PinnedScratch {
  void* p = nullptr;
  size_t cap = 0;
  void* get(size_t n) {
    if (n > cap) {
      if (p) cudaFreeHost(p);
      p = nullptr; cap = 0;
      const size_t want = n + n / 4 + 4096;
      if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { p = nullptr; cudaGetLastError(); return nullptr; }
      cap = want;
    }
    return p;
  }
};
static thread_local PinnedScratch g_split_pin;

static thread_local long long g_split_stats[4] = {0, 0, 0, 0};     // tie values' edges, steps / rounds, off-lowest steps, mode

__global__ void apply_keep_kernel(int A, const int* __restrict__ a_eid, const uint8_t* __restrict__ keep, uint8_t* __restrict__ act) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x)
    if (!keep[i]) act[a_eid[i]] = 0;
}

int split_exact_host_impl(const int* src, const int* dst, const float* prob, long long m, int n_nodes, int C, uint8_t* keep,
                          int64_t* stats_out, const uint8_t* tied, const int* seeds, long long n_seeds, const uint8_t* sel);      // split_exact.cu

// The reference order on the host for the graphs flagged in host_graph: one split_exact_host_impl call per graph on its own slice of
// the active list, with graph-local node ids, its own node count and camera bound — exactly the call a single-graph
// post-processing of that graph makes, so the engine's numbering and its re-read of the integer label (utils.py:112) are the
// graph's own.  Graphs are independent: they run on a few host threads, each writing its own slice, and the result depends
// neither on the thread count nor on the order of the seeds.
static int split_host_graphs(PostCtx& c, uint8_t* act, const float* prob, int pstride, const std::vector<int>& ncam,
                             const std::vector<int>& nptr, const std::vector<int>& host_graph, int Dn, bool have_ties,
                             long long* steps, long long* off_lowest) {
  const int A = c.n_active, G = (int)ncam.size();
  gather_select_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, act, prob, pstride, c.wcc, c.wccflag, c.a_prob, c.sel);
  MPN_LAUNCH_OK();
  std::vector<int> agp{0, A}, seeds(Dn);                // one graph: its slice is the whole active list
  if (G > 1) {
    agp.resize((size_t)G + 1);
    active_graph_ptr_kernel<<<list_grid(G + 1), 256, 0, c.st>>>(G, c.g.rowptr, c.g.graph_nptr, c.a_eid, A, c.a_gptr);
    MPN_LAUNCH_OK();
    MPN_CUDA_OK(cudaMemcpyAsync(agp.data(), c.a_gptr, sizeof(int) * (G + 1), cudaMemcpyDeviceToHost, c.st));
  }
  MPN_CUDA_OK(cudaMemcpyAsync(seeds.data(), c.dirty_nodes, sizeof(int) * Dn, cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  // runs of consecutive host-order graphs = contiguous ranges of the active list, packed back to back in pinned staging (pageable
  // destinations would be staged by the driver at a few GB/s)
  struct Run { int g0, g1; long long a0, a1, h0; };
  std::vector<Run> runs;
  long long staged = 0;
  for (int g = 0; g < G; ++g) {
    if (!host_graph[g]) continue;
    if (!runs.empty() && runs.back().g1 == g) { runs.back().g1 = g + 1; runs.back().a1 = agp[g + 1]; continue; }
    runs.push_back(Run{g, g + 1, agp[g], agp[g + 1], 0});
  }
  for (Run& r : runs) { r.h0 = staged; staged += r.a1 - r.a0; }
  const size_t S16 = ((size_t)staged + 15) & ~(size_t)15;
  char* pin = (char*)g_split_pin.get(15 * S16 + 64);
  MPN_REQUIRE(pin != nullptr, "split: out of pinned host memory (%zu bytes)", 15 * S16 + 64);
  int* hs = (int*)pin;
  int* hd = (int*)(pin + 4 * S16);
  float* hp = (float*)(pin + 8 * S16);
  uint8_t* hsel = (uint8_t*)(pin + 12 * S16);
  uint8_t* htied = hsel + S16;
  uint8_t* keep = htied + S16;
  for (const Run& r : runs) {
    const size_t n = (size_t)(r.a1 - r.a0);
    if (n == 0) continue;
    MPN_CUDA_OK(cudaMemcpyAsync(hs + r.h0, c.a_src + r.a0, sizeof(int) * n, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(hd + r.h0, c.a_dst + r.a0, sizeof(int) * n, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(hp + r.h0, c.a_prob + r.a0, sizeof(float) * n, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(hsel + r.h0, c.sel + r.a0, n, cudaMemcpyDeviceToHost, c.st));
    if (have_ties) MPN_CUDA_OK(cudaMemcpyAsync(htied + r.h0, c.tiedb + r.a0, n, cudaMemcpyDeviceToHost, c.st));
  }
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  // per host-order graph: where its slice sits in the staging, its seeds in graph-local ids
  std::vector<int> graphs;
  std::vector<long long> h_of((size_t)G, -1);
  for (const Run& r : runs)
    for (int g = r.g0; g < r.g1; ++g) { graphs.push_back(g); h_of[g] = r.h0 + (agp[g] - r.a0); }
  std::vector<std::vector<int>> gseeds((size_t)G);
  if (G == 1) {
    gseeds[0] = std::move(seeds);                  // one graph: every seed is its own, in its own ids
  } else {
    for (int v : seeds) {
      const int g = (int)(std::upper_bound(nptr.begin(), nptr.end(), v) - nptr.begin()) - 1;
      if (host_graph[g]) gseeds[g].push_back(v - nptr[g]);
    }
  }
  std::vector<int64_t> gst(4 * (size_t)G, 0);
  std::vector<int> rc((size_t)G, MPN_OK);
  std::vector<std::string> err((size_t)G);
  std::atomic<size_t> next{0};
  auto worker = [&] {
    std::vector<int> ls, ld;
    for (size_t k = next++; k < graphs.size(); k = next++) {
      const int g = graphs[k];
      const long long h = h_of[g], m = agp[g + 1] - agp[g];
      const int n0 = nptr[g];
      long long n_sel = 0;
      for (long long i = 0; i < m; ++i) n_sel += hsel[h + i];
      if (n_sel == 0) { memset(keep + h, 1, (size_t)m); continue; }
      const int *s = hs + h, *d = hd + h;             // node ids are graph-local already when the graph starts at node 0
      if (n0 != 0) {
        ls.resize(m); ld.resize(m);
        for (long long i = 0; i < m; ++i) { ls[i] = s[i] - n0; ld[i] = d[i] - n0; }
        s = ls.data(); d = ld.data();
      }
      rc[g] = split_exact_host_impl(s, d, hp + h, m, nptr[g + 1] - n0, ncam[g], keep + h, &gst[4 * (size_t)g],
                                    have_ties ? htied + h : nullptr, gseeds[g].data(), (long long)gseeds[g].size(), hsel + h);
      if (rc[g] != MPN_OK) err[g] = mpn_last_error();
    }
  };
  const int n_threads = (int)std::min<size_t>(graphs.size(), std::max(1u, std::min(8u, std::thread::hardware_concurrency())));
  if (n_threads <= 1) {
    worker();
  } else {
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; ++t) pool.emplace_back(worker);
    for (std::thread& t : pool) t.join();
  }
  for (int g : graphs)
    if (rc[g] != MPN_OK) { set_error("split (graph %d of the batch): %s", g, err[g].c_str()); return rc[g]; }
  *steps = *off_lowest = 0;
  for (int g : graphs) { *steps += gst[4 * (size_t)g]; *off_lowest += gst[4 * (size_t)g + 1]; }
  // write back: keep = 1 everywhere but in the slices the engine decided
  if (staged < A) MPN_CUDA_OK(cudaMemsetAsync(c.sel, 1, (size_t)A, c.st));
  for (const Run& r : runs)
    if (r.a1 > r.a0) MPN_CUDA_OK(cudaMemcpyAsync(c.sel + r.a0, keep + r.h0, (size_t)(r.a1 - r.a0), cudaMemcpyHostToDevice, c.st));
  apply_keep_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.sel, act);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));        // the staging buffer is reused by the next call
  return MPN_OK;
}

// SPLITTING of every graph; ncam / nptr: camera count and first node of each graph ({C} and {0, N} for one graph).  The mode is
// chosen per graph: a graph with a tie among the values its oversized clusters can drop (or every graph with an oversized
// cluster, when the tie table does not fit) goes through the reference order on the host; the others drop their minima in
// parallel rounds on the device, restricted to their own dirty lists.  Graphs are independent, so both modes run on one batch and
// the result is exact.
static int split_stage(PostCtx& c, uint8_t* act, const float* prob, int pstride, const Graphs& graphs, const std::vector<int>& ncam,
                       const std::vector<int>& nptr) {
  const int A = c.n_active, N = c.g.n_nodes, G = (int)ncam.size();
  g_split_stats[0] = g_split_stats[1] = g_split_stats[2] = g_split_stats[3] = 0;
  if (A == 0) return MPN_OK;
  // round 0 on the whole graph: components, sizes, dirty lists
  MPN_TRY(scc_stage(c, act, nullptr));
  MPN_CUDA_OK(cudaMemsetAsync(c.size, 0, sizeof(int) * N, c.st));
  MPN_CUDA_OK(cudaMemsetAsync(c.counters + 5, 0, 2 * sizeof(int), c.st));
  comp_size_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.label, c.size);
  MPN_LAUNCH_OK();
  mark_dirty_nodes_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.label, c.size, graphs, nullptr, c.dirty_nodes, c.counters + 5);
  MPN_LAUNCH_OK();
  mark_dirty_edges_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.label, c.size, graphs, nullptr,
                                                         c.dirty_edges, c.counters + 6);
  MPN_LAUNCH_OK();
  int h[2] = {0, 0};
  MPN_CUDA_OK(cudaMemcpyAsync(h, c.counters + 5, 2 * sizeof(int), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  int Dn = h[0], De = h[1];
  static const bool dbg = getenv("MPN_POST_DEBUG") != nullptr;
  if (dbg) fprintf(stderr, "[split] A=%d N=%d dirty nodes=%d dirty edges=%d\n", A, N, Dn, De);
  if (Dn == 0) return MPN_OK;
  // ---- which graphs have a tie among the values their oversized clusters can drop?
  iota_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.wcc);
  MPN_LAUNCH_OK();
  union_all_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.wcc);
  MPN_LAUNCH_OK();
  flatten_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.wcc, nullptr);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaMemsetAsync(c.wccflag, 0, sizeof(int) * N, c.st));
  MPN_CUDA_OK(cudaMemsetAsync(c.gflag, 0, sizeof(int) * (G + 1), c.st));
  const bool table_fits = (long long)De * 5 <= (long long)c.tie_cap * 3;       // load factor <= 0.6
  if (table_fits) {
    MPN_CUDA_OK(cudaMemsetAsync(c.tie_keys, 0xFF, sizeof(unsigned long long) * c.tie_cap, c.st));
    MPN_CUDA_OK(cudaMemsetAsync(c.tie_counts, 0, sizeof(int) * c.tie_cap, c.st));
    if (De > 0) {
      tie_insert_kernel<<<list_grid(De), 256, 0, c.st>>>(De, c.dirty_edges, c.a_eid, c.a_src, graphs, act, prob, pstride, c.tie_keys,
                                                         c.tie_cap);
      MPN_LAUNCH_OK();
    }
    tie_count_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, graphs, act, prob, pstride, c.tie_keys, c.tie_counts, c.tie_cap);
    MPN_LAUNCH_OK();
    flag_wcc_ties_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, graphs, act, prob, pstride, c.tie_keys, c.tie_counts,
                                                         c.tie_cap, c.wcc, c.wccflag, c.tiedb, c.gflag, c.gflag + G);
    MPN_LAUNCH_OK();
  } else {
    MPN_CUDA_OK(cudaMemsetAsync(c.wccflag, 0x01, sizeof(int) * N, c.st));   // every component of the host-order graphs
    flag_graphs_of_nodes_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, graphs, c.gflag);
    MPN_LAUNCH_OK();
  }
  std::vector<int> host_graph((size_t)G + 1);
  MPN_CUDA_OK(cudaMemcpyAsync(host_graph.data(), c.gflag, sizeof(int) * (G + 1), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  const int n_tied = host_graph[G];
  long long n_host = 0, host_steps = 0, host_off_lowest = 0;
  for (int g = 0; g < G; ++g) n_host += host_graph[g] != 0;
  g_split_stats[0] = table_fits ? n_tied : -1;
  if (dbg) fprintf(stderr, "[split] active edges carrying a tied value: %d%s; graphs in the reference order: %lld of %d\n", n_tied,
                   table_fits ? "" : " (table too small: every graph with an oversized cluster goes to the host)", n_host, G);
  if (n_host > 0) {
    if (table_fits) {                               // the components of the oversized clusters go to the host with their graph
      flag_wcc_nodes_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.wcc, c.wccflag);
      MPN_LAUNCH_OK();
    }
    MPN_TRY(split_host_graphs(c, act, prob, pstride, ncam, nptr, host_graph, Dn, table_fits, &host_steps, &host_off_lowest));
    if (n_host == G) {
      Dn = 0;                                       // no graph is left for the device rounds
    } else {                                        // the device rounds below only see the other graphs
      MPN_CUDA_OK(cudaMemsetAsync(c.counters + 5, 0, 2 * sizeof(int), c.st));
      mark_dirty_nodes_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.label, c.size, graphs, c.gflag, c.dirty_nodes, c.counters + 5);
      MPN_LAUNCH_OK();
      mark_dirty_edges_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.label, c.size, graphs, c.gflag,
                                                             c.dirty_edges, c.counters + 6);
      MPN_LAUNCH_OK();
      MPN_CUDA_OK(cudaMemcpyAsync(h, c.counters + 5, 2 * sizeof(int), cudaMemcpyDeviceToHost, c.st));
      MPN_CUDA_OK(cudaStreamSynchronize(c.st));
      Dn = h[0];
      De = h[1];
    }
  }
  // ---- no tie inside any of the remaining graphs: every oversized cluster drops its minimum in the same round
  int rounds = 0;
  while (Dn > 0) {
    // per-cluster minimum probability over the active edges touching each oversized cluster
    reset_nodes_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label, c.size, c.mbits, 4);
    MPN_LAUNCH_OK();
    MPN_CUDA_OK(cudaMemsetAsync(c.hash, 0xFF, sizeof(unsigned long long) * c.hash_cap, c.st));
    MPN_CUDA_OK(cudaMemsetAsync(c.counters + 4, 0, sizeof(int), c.st));
    if (De > 0) {
      split_min_list_kernel<<<list_grid(De), 256, 0, c.st>>>(De, c.dirty_edges, c.a_eid, c.a_src, c.a_dst, act, prob, pstride, c.label,
                                                           c.size, graphs, c.mbits);
      MPN_LAUNCH_OK();
    }
    split_collect_list_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label, c.size, graphs, c.mbits, c.hash, c.hash_cap,
                                                              c.counters + 4);
    MPN_LAUNCH_OK();
    int n_big = 0;
    MPN_CUDA_OK(cudaMemcpyAsync(&n_big, c.counters + 4, sizeof(int), cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaStreamSynchronize(c.st));
    if (n_big == 0) break;
    ++rounds;
    if (rounds > A + 1) { set_error("split did not converge"); return MPN_ERR_INVALID; }
    split_remove_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, graphs, act, prob, pstride, c.hash, c.hash_cap);
    MPN_LAUNCH_OK();
    // recompute components and sizes of the dirty part only
    MPN_TRY(scc_dirty(c, act, Dn, De));
    reset_nodes_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label, c.size, c.mbits, 2);
    MPN_LAUNCH_OK();
    comp_size_list_kernel<<<list_grid(Dn), 256, 0, c.st>>>(Dn, c.dirty_nodes, c.label, c.size);
    MPN_LAUNCH_OK();
  }
  g_split_stats[1] = rounds + host_steps;
  g_split_stats[2] = host_off_lowest;
  g_split_stats[3] = n_host;
  return MPN_OK;
}

static int post_begin(PostCtx& c, const mpn_graph* g, const uint8_t* act, void* ws, size_t ws_bytes, void* stream) {
  MPN_REQUIRE(g && ws, "post: NULL argument");
  MPN_REQUIRE(act || g->n_edges == 0, "post: NULL activity flags");
  MPN_REQUIRE(g->row_offset == 0 && g->n_cols == g->n_nodes, "post-processing runs on an unsharded graph (replicas only)");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  c.g = *g;
  c.st = (cudaStream_t)stream;
  post_layout(c, ws, ws_bytes);
  if (c.total > ws_bytes) {
    set_error("post workspace too small: need %zu bytes, have %zu", c.total, ws_bytes);
    return MPN_ERR_WORKSPACE;
  }
  return build_active_list(c, act);
}

static int copy_graph_ptr(const PostCtx& c, std::vector<int>& nptr) {
  nptr.resize((size_t)c.g.n_graphs + 1);
  MPN_CUDA_OK(cudaMemcpyAsync(nptr.data(), c.g.graph_nptr, sizeof(int) * nptr.size(), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  return MPN_OK;
}

// ------------------------------------------------------------------------------------------------
// reference label numbering on the host (utils.py:30-52 + networkx SCC emission order)
// ------------------------------------------------------------------------------------------------
struct TarjanNode {                       // everything the traversal touches about one node, in one cache line
  int beg, end, cur;                      // successor list [beg, end) in adj, resumable iterator
  int pre, low, comp;                     // preorder number (0 = unvisited), lowlink, emission index of its component (-1 = open)
};
static void labels_reference(const int* src, const int* dst, long long m, int n_nodes, long long* labels, int* n_comp) {
  // flat arrays throughout (one allocation each, no per-component vectors): this runs once per post_processing call on up to
  // millions of active edges (m < 2^31: edge ids are int32 everywhere), and once per dropped value in split_reference
  std::vector<int> order;                 // nodes in first-appearance order (u then v per edge): DiGraph insertion order
  order.reserve((size_t)std::min<long long>(2 * m, n_nodes));
  std::vector<TarjanNode> node((size_t)n_nodes + 1, TarjanNode{0, 0, 0, 0, 0, -2});     // comp -2: not in the digraph yet
  for (long long i = 0; i < m; ++i) {
    const int u = src[i], v = dst[i];
    if (node[u].comp == -2) { node[u].comp = -1; order.push_back(u); }
    if (node[v].comp == -2) { node[v].comp = -1; order.push_back(v); }
    node[u].end++;                        // out-degree for now
  }
  int run = 0;
  for (int i = 0; i < n_nodes; ++i) { const int deg = node[i].end; node[i].beg = node[i].cur = run; run += deg; node[i].end = run; }
  std::vector<int> adj((size_t)m);
  for (long long i = 0; i < m; ++i) adj[node[src[i]].cur++] = dst[i];     // successor order = edge insertion order
  for (int i = 0; i < n_nodes; ++i) node[i].cur = node[i].beg;
  std::vector<int> queue, scc_queue, comp_size;
  int counter = 0;
  for (int source : order) {
    if (node[source].comp >= 0) continue;
    queue.assign(1, source);
    while (!queue.empty()) {
      const int v = queue.back();
      TarjanNode& nv = node[v];
      if (nv.pre == 0) nv.pre = ++counter;
      bool done = true;
      while (nv.cur < nv.end) {
        const int w = adj[nv.cur++];
        if (node[w].pre == 0) { queue.push_back(w); done = false; break; }
      }
      if (!done) continue;
      int low = nv.pre;
      for (int k = nv.beg; k < nv.end; ++k) {
        const TarjanNode& nw = node[adj[k]];
        if (nw.comp < 0) low = std::min(low, nw.pre > nv.pre ? nw.low : nw.pre);
      }
      nv.low = low;
      queue.pop_back();
      if (low == nv.pre) {
        const int c = (int)comp_size.size();                              // emission index of this component
        int size = 1;
        nv.comp = c;
        while (!scc_queue.empty() && node[scc_queue.back()].pre > nv.pre) { node[scc_queue.back()].comp = c; scc_queue.pop_back(); ++size; }
        comp_size.push_back(size);
      } else {
        scc_queue.push_back(v);
      }
    }
  }
  // sorted(key=len), stable: counting sort of the emission indices by component size (utils.py:31)
  const int nc = (int)comp_size.size();
  std::vector<int> start((size_t)n_nodes + 2, 0), rank(nc);
  for (int c = 0; c < nc; ++c) start[comp_size[c] + 1]++;
  for (int sz = 0; sz <= n_nodes; ++sz) start[sz + 1] += start[sz];
  for (int c = 0; c < nc; ++c) rank[c] = start[comp_size[c]]++;
  long long k = nc;
  for (int i = 0; i < n_nodes; ++i) labels[i] = node[i].comp >= 0 ? rank[node[i].comp] : k++;   // no active edge: last, index order
  *n_comp = (int)k;
}

// ------------------------------------------------------------------------------------------------
// Reference label numbering (utils.py:30-52) without a sequential pass over the active edges.
// networkx emits the SCCs source by source (sources in first-appearance order of the nodes in the active edge list, u before v),
// each source's DFS in post-order, and a DFS never leaves its weakly connected component.  So
//   label = rank of (size, first-appearance key of the emitting source, index within that DFS)   among the SCCs with an edge,
// then the nodes without an active edge in index order.  For an SCC that is alone in its weakly connected component (no
// one-directional edge to another SCC — every component after CUTTING, almost every component otherwise) the emitting source is
// its own earliest node: key = min over its nodes of the first-appearance key, index 0 — an atomicMin per active edge on the
// device.  Only the components that one-directional edges tie together go through the sequential generator (split_exact.cu),
// restricted to those components.
// ------------------------------------------------------------------------------------------------
__global__ void first_appearance_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                        const uint8_t* __restrict__ act, unsigned int* __restrict__ fa) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    if (!act[a_eid[i]]) continue;
    atomicMin(&fa[a_src[i]], 2u * (unsigned int)i);
    atomicMin(&fa[a_dst[i]], 2u * (unsigned int)i + 1u);
  }
}
__global__ void inter_scc_flag_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const int* __restrict__ a_dst,
                                      const uint8_t* __restrict__ act, const int* __restrict__ label, const int* __restrict__ wcc,
                                      int* __restrict__ wccflag, int* __restrict__ count) {
  int c = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x) {
    if (!act[a_eid[i]]) continue;
    if (label[a_src[i]] != label[a_dst[i]]) {
      ++c;
      if (wcc != nullptr) wccflag[wcc[a_src[i]]] = 1;
    }
  }
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, c);
}
__global__ void select_flagged_kernel(int A, const int* __restrict__ a_eid, const int* __restrict__ a_src, const uint8_t* __restrict__ act,
                                      const int* __restrict__ wcc, const int* __restrict__ wccflag, uint8_t* __restrict__ sel) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < A; i += gridDim.x * blockDim.x)
    sel[i] = (act[a_eid[i]] && wccflag[wcc[a_src[i]]]) ? 1 : 0;
}

void scc_emission_keys_host(const int* src, const int* dst, long long m, int n_nodes, std::vector<int>& node_out,
                            std::vector<long long>& key_out, std::vector<int>& idx_out, std::vector<int>& size_out);   // split_exact.cu

// per SCC (root = smallest node id) of the active digraph: size, first-appearance key and index within the emitting DFS;
// label[n] = root of n, fa[n] = first-appearance key of n (0xFFFFFFFF: no active edge)
struct RefKeys {
  std::vector<int> label;
  std::vector<unsigned int> fa, size, idx;
  std::vector<unsigned long long> key;
};
static int reference_keys(PostCtx& c, const uint8_t* act, RefKeys& k) {
  const int A = c.n_active, N = c.g.n_nodes;
  MPN_TRY(scc_stage(c, act, nullptr));
  unsigned int* fa = reinterpret_cast<unsigned int*>(c.fo);
  MPN_CUDA_OK(cudaMemsetAsync(fa, 0xFF, sizeof(unsigned int) * N, c.st));
  MPN_CUDA_OK(cudaMemsetAsync(c.counters + 7, 0, sizeof(int), c.st));
  int n_inter = 0;
  if (A > 0) {
    first_appearance_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, fa);
    MPN_LAUNCH_OK();
    inter_scc_flag_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.label, nullptr, nullptr, c.counters + 7);
    MPN_LAUNCH_OK();
  }
  std::vector<int>& h_label = k.label;
  std::vector<unsigned int>& h_fa = k.fa;
  h_label.resize(N);
  h_fa.resize(N);
  MPN_CUDA_OK(cudaMemcpyAsync(h_label.data(), c.label, sizeof(int) * N, cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaMemcpyAsync(h_fa.data(), fa, sizeof(unsigned int) * N, cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaMemcpyAsync(&n_inter, c.counters + 7, sizeof(int), cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  // components that one-directional edges tie together: their emission order comes from the sequential generator
  std::vector<int> cx_node, cx_idx, cx_size;
  std::vector<long long> cx_key;
  std::vector<int> pos;
  if (n_inter > 0) {
    iota_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.wcc);
    MPN_LAUNCH_OK();
    union_all_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.wcc);
    MPN_LAUNCH_OK();
    flatten_kernel<<<list_grid(N), 256, 0, c.st>>>(N, c.wcc, nullptr);
    MPN_LAUNCH_OK();
    MPN_CUDA_OK(cudaMemsetAsync(c.wccflag, 0, sizeof(int) * N, c.st));
    MPN_CUDA_OK(cudaMemsetAsync(c.counters + 7, 0, sizeof(int), c.st));
    inter_scc_flag_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, c.a_dst, act, c.label, c.wcc, c.wccflag, c.counters + 7);
    MPN_LAUNCH_OK();
    select_flagged_kernel<<<list_grid(A), 256, 0, c.st>>>(A, c.a_eid, c.a_src, act, c.wcc, c.wccflag, c.sel);
    MPN_LAUNCH_OK();
    const size_t A16 = ((size_t)A + 15) & ~(size_t)15;
    char* pin = (char*)g_split_pin.get(9 * A16 + 64);          // pinned staging (see split_host_graphs)
    MPN_REQUIRE(pin != nullptr, "reference numbering: out of pinned host memory");
    int *hs = (int*)pin, *hd = (int*)(pin + 4 * A16);
    uint8_t* hsel = (uint8_t*)(pin + 8 * A16);
    MPN_CUDA_OK(cudaMemcpyAsync(hs, c.a_src, sizeof(int) * A, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(hd, c.a_dst, sizeof(int) * A, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(hsel, c.sel, A, cudaMemcpyDeviceToHost, c.st));
    MPN_CUDA_OK(cudaStreamSynchronize(c.st));
    std::vector<int> ss, dd;
    for (int i = 0; i < A; ++i)
      if (hsel[i]) { pos.push_back(i); ss.push_back(hs[i]); dd.push_back(hd[i]); }
    scc_emission_keys_host(ss.data(), dd.data(), (long long)ss.size(), N, cx_node, cx_key, cx_idx, cx_size);
  }
  std::vector<unsigned int>&size = k.size, &idx = k.idx;
  std::vector<unsigned long long>& key = k.key;
  size.assign(N, 0u);
  idx.assign(N, 0u);
  key.assign(N, ~0ull);
  for (int n = 0; n < N; ++n) {
    if (h_fa[n] == 0xFFFFFFFFu) continue;
    const int r = h_label[n];
    ++size[r];
    if ((unsigned long long)h_fa[n] < key[r]) key[r] = h_fa[n];
  }
  for (size_t v = 0; v < cx_node.size(); ++v) {
    const int r = h_label[cx_node[v]];
    // local key = 2 * (index in the gathered list) + side  ->  2 * (position in the active list) + side
    key[r] = 2ull * (unsigned long long)pos[(size_t)(cx_key[v] >> 1)] + (unsigned long long)(cx_key[v] & 1);
    idx[r] = (unsigned int)cx_idx[v];
    if ((unsigned int)cx_size[v] != size[r]) { set_error("reference numbering: component sizes disagree (device %u, host %d)", size[r], cx_size[v]); return MPN_ERR_INVALID; }
  }
  return MPN_OK;
}

// The roots of the SCCs with an active edge in (key, idx) order, then stably by size.  Keys are positions in the active list
// (< 2A + 2): one bucket pass puts the components in (key, idx) order — several components share a key only when one DFS source
// of the sequential generator emitted them, those few are sorted by idx — and a stable counting sort by size finishes the order.
static int roots_in_reference_order(const RefKeys& k, int A, std::vector<int>& order) {
  const int N = (int)k.label.size();
  const size_t n_keys = 2 * (size_t)A + 2;
  std::vector<int> head(n_keys, -1), nxt((size_t)N, -1);
  unsigned int max_size = 0;
  size_t n_reps = 0;
  for (int r = N - 1; r >= 0; --r) {
    if (k.size[r] == 0) continue;
    if (k.key[r] >= n_keys) { set_error("reference numbering: first-appearance key out of range"); return MPN_ERR_INVALID; }
    nxt[r] = head[k.key[r]];
    head[k.key[r]] = r;
    max_size = std::max(max_size, k.size[r]);
    ++n_reps;
  }
  std::vector<int> by_key;
  by_key.reserve(n_reps);
  std::vector<int> same;
  for (size_t q = 0; q < n_keys; ++q) {
    int r = head[q];
    if (r < 0) continue;
    if (nxt[r] < 0) { by_key.push_back(r); continue; }
    same.clear();
    for (; r >= 0; r = nxt[r]) same.push_back(r);
    std::sort(same.begin(), same.end(), [&](int a, int b) { return k.idx[a] < k.idx[b]; });
    by_key.insert(by_key.end(), same.begin(), same.end());
  }
  std::vector<size_t> first((size_t)max_size + 2, 0);
  for (int r : by_key) ++first[k.size[r] + 1];
  for (size_t z = 1; z < first.size(); ++z) first[z] += first[z - 1];
  order.resize(n_reps);
  for (int r : by_key) order[first[k.size[r]]++] = r;
  return MPN_OK;
}

// Reference numbering of each graph from 0 on its own; nptr = first node of each graph ({0, N} for one graph).  A DFS never leaves
// its graph and the active list holds the graphs one after the other, so a component's (key, idx) orders it within its graph
// exactly as numbering that graph alone does (keys shifted by the graph's first active entry); the order (size, key, idx) then
// becomes (graph, size, key, idx) — a stable pass by graph over the whole order — and the nodes without an active edge follow
// their own graph's components, in node order.
static int labels_reference_per_graph(PostCtx& c, const uint8_t* act, const std::vector<int>& nptr, long long* labels_out,
                                      int* n_comp_out) {
  const int N = c.g.n_nodes, G = (int)nptr.size() - 1;
  RefKeys k;
  MPN_TRY(reference_keys(c, act, k));
  std::vector<int> order;
  MPN_TRY(roots_in_reference_order(k, c.n_active, order));
  std::vector<int> rank((size_t)N, -1), count((size_t)G, 0);      // rank[r]: the place of root r among its graph's SCCs
  if (G == 1) {                                                    // one graph: its place in the order, no per-node graph ids
    for (size_t i = 0; i < order.size(); ++i) rank[order[i]] = (int)i;
    count[0] = (int)order.size();
  } else {
    // graph ids in an array of their own: reading them back from rank would chain each root on the previous root's store
    std::vector<int> gid((size_t)N);
    for (int g = 0; g < G; ++g) std::fill(gid.begin() + nptr[g], gid.begin() + nptr[g + 1], g);
    for (int r : order) rank[r] = count[gid[r]]++;
  }
  for (int g = 0; g < G; ++g) {
    long long next = count[g];
    for (int n = nptr[g]; n < nptr[g + 1]; ++n) labels_out[n] = (k.fa[n] != 0xFFFFFFFFu) ? rank[k.label[n]] : next++;
    n_comp_out[g] = (int)next;
  }
  return MPN_OK;
}

// canonical graph-local labels (smallest node id of the SCC minus the graph's first node) and the number of SCCs per graph
__global__ void graph_labels_kernel(int N, const int* __restrict__ label, const Graphs graphs, const int* __restrict__ nptr,
                                    int* __restrict__ local, int* __restrict__ roots) {
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
    const int g = graphs.graph_of(n), l = label[n];
    if (local) local[n] = l - nptr[g];
    if (l == n) atomicAdd(&roots[g], 1);
  }
}

// inference.post_processing (inference.py:70-169) on every graph: CUT, PRUNE, CUT, SPLIT, then the SCC labels.  labels (optional,
// device): canonical labels, graph-local in a batch; n_components (host): one count per graph; prune_changed (optional): whether
// PRUNE removed an edge.
static int post_pipeline(PostCtx& c, uint8_t* act, const float* prob1, int pstride, const Graphs& graphs, const std::vector<int>& ncam,
                         const std::vector<int>& nptr, int flags, int32_t* labels, int32_t* n_components, int32_t* prune_changed) {
  int ch = 0, r = 0;
  if ((flags & MPN_POST_CUT) && c.n_active) {
    cut_kernel<<<list_grid(c.n_active), 256, 0, c.st>>>(c.n_active, c.a_eid, c.a_rev, act);
    MPN_LAUNCH_OK();
  }
  if (flags & MPN_POST_PRUNE) MPN_TRY(prune_stage(c, act, prob1, pstride, graphs, &ch, &r));
  if ((flags & MPN_POST_CUT) && c.n_active) {
    cut_kernel<<<list_grid(c.n_active), 256, 0, c.st>>>(c.n_active, c.a_eid, c.a_rev, act);
    MPN_LAUNCH_OK();
  }
  if (flags & MPN_POST_SPLIT) MPN_TRY(split_stage(c, act, prob1, pstride, graphs, ncam, nptr));
  int nc = 0;
  MPN_TRY(scc_stage(c, act, &nc));
  if (graphs.gid) {
    const int G = (int)ncam.size();
    MPN_CUDA_OK(cudaMemsetAsync(c.groots, 0, sizeof(int) * G, c.st));
    graph_labels_kernel<<<list_grid(c.g.n_nodes), 256, 0, c.st>>>(c.g.n_nodes, c.label, graphs, c.g.graph_nptr, labels, c.groots);
    MPN_LAUNCH_OK();
    MPN_CUDA_OK(cudaMemcpyAsync(n_components, c.groots, sizeof(int) * G, cudaMemcpyDeviceToHost, c.st));
  } else {
    if (labels) MPN_CUDA_OK(cudaMemcpyAsync(labels, c.label, sizeof(int) * c.g.n_nodes, cudaMemcpyDeviceToDevice, c.st));
    if (n_components) *n_components = nc;
  }
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  if (prune_changed) *prune_changed = ch;
  return MPN_OK;
}

__global__ void clear_inactive_kernel(long long n, const int* __restrict__ eid, const uint8_t* __restrict__ keep,
                                      uint8_t* __restrict__ act) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    if (!keep[i]) act[eid[i]] = 0;
}

// workspace of the shard compaction: block offsets + one counter
struct CompactCtx {
  int n_blocks;
  int *blockoff, *counter;
  size_t total;
};
static void compact_layout(CompactCtx& c, const mpn_graph& g, void* ws, size_t ws_bytes) {
  Arena a(ws, ws_bytes);
  c.n_blocks = div_up((long long)(g.n_edges > 0 ? g.n_edges : 1), EPB);
  c.blockoff = a.take<int>(c.n_blocks + 1);
  c.counter = a.take<int>(8);
  c.total = a.off;
}

}  // namespace mpn

using namespace mpn;

extern "C" {

size_t mpn_post_workspace_bytes(const mpn_graph* g) {
  if (!g) return 0;
  PostCtx c;
  c.g = *g;
  post_layout(c, nullptr, 0);
  return c.total + 256;
}

int mpn_cut(const mpn_graph* g, uint8_t* act, void* ws, size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  if (c.n_active == 0) return MPN_OK;
  cut_kernel<<<list_grid(c.n_active), 256, 0, c.st>>>(c.n_active, c.a_eid, c.a_rev, act);
  MPN_LAUNCH_OK();
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  return MPN_OK;
}

int mpn_prune(const mpn_graph* g, uint8_t* act, const float* prob1, int32_t pstride, int32_t num_cameras, int32_t* changed,
              int32_t* rounds, void* ws, size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_REQUIRE(prob1 && pstride >= 1 && num_cameras >= 1, "prune: bad arguments");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  int ch = 0, r = 0;
  MPN_TRY(prune_stage(c, act, prob1, pstride, one_graph(num_cameras), &ch, &r));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  if (changed) *changed = ch;
  if (rounds) *rounds = r;
  return MPN_OK;
}

int mpn_split(const mpn_graph* g, uint8_t* act, const float* prob1, int32_t pstride, int32_t num_cameras, int32_t* rounds,
              void* ws, size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_REQUIRE(prob1 && pstride >= 1 && num_cameras >= 1, "split: bad arguments");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  MPN_TRY(split_stage(c, act, prob1, pstride, one_graph(num_cameras), {num_cameras}, {0, g->n_nodes}));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  if (rounds) *rounds = (int)g_split_stats[1];                 // device rounds, or the values the host order dropped
  return MPN_OK;
}

void mpn_split_last_stats(int64_t out[4]) {
  if (out) for (int i = 0; i < 4; ++i) out[i] = g_split_stats[i];
}

int mpn_scc_labels(const mpn_graph* g, const uint8_t* act, int32_t* labels, int32_t* n_components, void* ws, size_t ws_bytes,
                   void* stream) {
  PostCtx c;
  MPN_REQUIRE(labels, "scc_labels: NULL output");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  int nc = 0;
  MPN_TRY(scc_stage(c, act, &nc));
  MPN_CUDA_OK(cudaMemcpyAsync(labels, c.label, sizeof(int) * g->n_nodes, cudaMemcpyDeviceToDevice, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  if (n_components) *n_components = nc;
  return MPN_OK;
}

int mpn_post_processing(const mpn_graph* g, uint8_t* act, const float* prob1, int32_t pstride, int32_t num_cameras, int32_t flags,
                        int32_t* labels, int32_t* n_components, int32_t* prune_changed, void* ws, size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_REQUIRE(prob1 && pstride >= 1 && num_cameras >= 1, "post_processing: bad arguments");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  return post_pipeline(c, act, prob1, pstride, one_graph(num_cameras), {num_cameras}, {0, g->n_nodes}, flags, labels, n_components,
                       prune_changed);
}

int mpn_post_processing_batched(const mpn_graph* g, uint8_t* act, const float* prob1, int32_t pstride, const int32_t* num_cameras_dev,
                                int32_t flags, int32_t* labels, int32_t* n_components, void* ws, size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_REQUIRE(prob1 && pstride >= 1 && num_cameras_dev && n_components, "post_processing_batched: bad arguments");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  const int G = std::max(1, g->n_graphs);
  std::vector<int> ncam((size_t)G);
  MPN_CUDA_OK(cudaMemcpyAsync(ncam.data(), num_cameras_dev, sizeof(int) * G, cudaMemcpyDeviceToHost, c.st));
  MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  for (int k = 0; k < G; ++k) MPN_REQUIRE(ncam[k] >= 1, "post_processing_batched: num_cameras[%d] = %d < 1", k, ncam[k]);
  Graphs graphs = one_graph(ncam[0]);
  std::vector<int> nptr{0, g->n_nodes};
  if (g->n_graphs > 1) {
    MPN_REQUIRE(g->node_gid && g->graph_nptr, "post_processing_batched: batched graph without node_gid / graph_nptr");
    MPN_TRY(copy_graph_ptr(c, nptr));
    graphs = Graphs{g->node_gid, num_cameras_dev, 0};
  }
  return post_pipeline(c, act, prob1, pstride, graphs, ncam, nptr, flags, labels, n_components, nullptr);
}

int mpn_active_edges(const mpn_graph* g, const uint8_t* act, int32_t* src_out, int32_t* dst_out, int64_t capacity,
                     int64_t* n_active, void* ws, size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  if (n_active) *n_active = c.n_active;
  MPN_REQUIRE(c.n_active <= capacity, "active_edges: capacity %lld < %d active edges", (long long)capacity, c.n_active);
  if (c.n_active) {
    MPN_REQUIRE(src_out && dst_out, "active_edges: NULL output");
    MPN_CUDA_OK(cudaMemcpyAsync(src_out, c.a_src, sizeof(int) * c.n_active, cudaMemcpyDeviceToDevice, c.st));
    MPN_CUDA_OK(cudaMemcpyAsync(dst_out, c.a_dst, sizeof(int) * c.n_active, cudaMemcpyDeviceToDevice, c.st));
    MPN_CUDA_OK(cudaStreamSynchronize(c.st));
  }
  return MPN_OK;
}

size_t mpn_compact_workspace_bytes(const mpn_graph* g) {
  if (!g) return 0;
  CompactCtx c;
  compact_layout(c, *g, nullptr, 0);
  return c.total + 256;
}

static int compact_begin(CompactCtx& c, const mpn_graph* g, const uint8_t* act, void* ws, size_t ws_bytes) {
  MPN_REQUIRE(g && ws, "compact: NULL argument");
  MPN_REQUIRE(act || g->n_edges == 0, "compact: NULL activity flags");
  MPN_REQUIRE(g->n_graphs <= 1, "compact: batched graphs are not row-sharded");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  compact_layout(c, *g, ws, ws_bytes);
  if (c.total > ws_bytes) {
    set_error("compact workspace too small: need %zu bytes, have %zu", c.total, ws_bytes);
    return MPN_ERR_WORKSPACE;
  }
  return MPN_OK;
}

int mpn_count_active(const mpn_graph* g, const uint8_t* act, int64_t* n_active, void* ws, size_t ws_bytes, void* stream) {
  CompactCtx c;
  MPN_REQUIRE(n_active, "count_active: NULL output");
  MPN_TRY(compact_begin(c, g, act, ws, ws_bytes));
  *n_active = 0;
  if (g->n_edges == 0) return MPN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  count_active_kernel<<<c.n_blocks, 256, 0, st>>>(act, g->n_edges, c.blockoff);
  MPN_LAUNCH_OK();
  scan_blocks_kernel<<<1, 1024, 0, st>>>(c.blockoff, c.n_blocks, c.counter);
  MPN_LAUNCH_OK();
  int n = 0;
  MPN_CUDA_OK(cudaMemcpyAsync(&n, c.counter, sizeof(int), cudaMemcpyDeviceToHost, st));
  MPN_CUDA_OK(cudaStreamSynchronize(st));
  *n_active = n;
  return MPN_OK;
}

int mpn_compact_active(const mpn_graph* g, const uint8_t* act, const float* prob1, int32_t pstride, int32_t* src_out,
                       int32_t* dst_out, int32_t* eid_out, float* prob_out, void* ws, size_t ws_bytes, void* stream) {
  CompactCtx c;
  MPN_TRY(compact_begin(c, g, act, ws, ws_bytes));
  if (g->n_edges == 0) return MPN_OK;
  MPN_REQUIRE(prob1 && pstride >= 1 && src_out && dst_out && eid_out && prob_out, "compact_active: bad arguments");
  write_active_kernel<true><<<c.n_blocks, 256, 0, (cudaStream_t)stream>>>(*g, act, c.blockoff, eid_out, src_out, dst_out, nullptr,
                                                                          prob1, pstride, prob_out);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_clear_inactive(uint8_t* act, const int32_t* eid, const uint8_t* keep, int64_t n, void* stream) {
  if (n <= 0) return MPN_OK;
  MPN_REQUIRE(act && eid && keep, "clear_inactive: NULL argument");
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(kNumSMs * 8, (n + 255) / 256));
  clear_inactive_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(n, eid, keep, act);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_labels_reference(const mpn_graph* g, const uint8_t* act, int64_t* labels_out_host, int32_t* n_components, void* ws,
                         size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_REQUIRE(labels_out_host, "labels_reference: NULL output");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  MPN_REQUIRE((long long)c.n_active < (1ll << 30), "labels_reference: more than 2^30 active edges");
  int nc = 0;
  MPN_TRY(labels_reference_per_graph(c, act, {0, g->n_nodes}, (long long*)labels_out_host, &nc));
  if (n_components) *n_components = nc;
  return MPN_OK;
}

int mpn_labels_reference_batched(const mpn_graph* g, const uint8_t* act, int64_t* labels_out_host, int32_t* n_components_host, void* ws,
                                 size_t ws_bytes, void* stream) {
  PostCtx c;
  MPN_REQUIRE(labels_out_host && n_components_host, "labels_reference_batched: NULL output");
  MPN_TRY(post_begin(c, g, act, ws, ws_bytes, stream));
  MPN_REQUIRE((long long)c.n_active < (1ll << 30), "labels_reference_batched: more than 2^30 active edges");
  std::vector<int> nptr{0, g->n_nodes};
  if (g->n_graphs > 1) {
    MPN_REQUIRE(g->graph_nptr, "labels_reference_batched: batched graph without graph_nptr");
    MPN_TRY(copy_graph_ptr(c, nptr));
  }
  return labels_reference_per_graph(c, act, nptr, (long long*)labels_out_host, n_components_host);
}

int mpn_labels_reference_host(const int32_t* src, const int32_t* dst, int64_t n_active, int32_t n_nodes, int64_t* labels_out,
                              int32_t* n_components) {
  MPN_REQUIRE(labels_out && n_nodes > 0 && n_active >= 0 && n_active < (1ll << 31) && (n_active == 0 || (src && dst)),
              "labels_reference_host: bad arguments");
  for (int64_t i = 0; i < n_active; ++i)
    MPN_REQUIRE(src[i] >= 0 && src[i] < n_nodes && dst[i] >= 0 && dst[i] < n_nodes, "labels_reference_host: node id out of range");
  int nc = 0;
  labels_reference(src, dst, n_active, n_nodes, (long long*)labels_out, &nc);
  if (n_components) *n_components = nc;
  return MPN_OK;
}

}  // extern "C"
