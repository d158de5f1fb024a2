// K0: int32 CSR + task tables from the reference's edge_index (models/mpn.py:44 `row, col = edge_index`), or built on the device
// from the camera layout of one graph or of a batch (inference.py:407-414).
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"

namespace mpn {

static thread_local char g_err[512] = "";
unsigned long long g_kernel_launches = 0;
int g_pdl_launch = 1;
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// One pass over the edges: narrow to int32, validate ordering / ranges, emit row boundaries.
template <typename IdxT>
__global__ void __launch_bounds__(256) csr_scan_edges(const IdxT* __restrict__ row, const IdxT* __restrict__ col,
                                                      long long E, int n_rows, int n_cols, int row_offset,
                                                      int* __restrict__ rowptr, int* __restrict__ col32,
                                                      int* __restrict__ flags) {
  pdl_wait();
  long long stride = (long long)gridDim.x * blockDim.x;
  int bad = 0;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    long long r = (long long)row[e] - row_offset, c = (long long)col[e];
    if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) { bad |= 2; continue; }
    col32[e] = (int)c;
    long long pr = -1, pc = -1;
    if (e > 0) {
      pr = (long long)row[e - 1] - row_offset;
      pc = (long long)col[e - 1];
      if (pr > r || (pr == r && pc >= c)) bad |= 1;
      if (pr < 0 || pr >= n_rows) pr = r;          // reported via the other thread's range check
    }
    for (long long q = pr + 1; q <= r; ++q) rowptr[q] = (int)e;      // rows (pr, r] start at e
    if (e == E - 1)
      for (long long q = r + 1; q <= n_rows; ++q) rowptr[q] = (int)E;
  }
  if (bad) atomicOr(flags, bad);
}

// int64 fast path: two consecutive edges per thread with 16-byte loads (E even, both rows of edge_index 16-byte aligned)
__global__ void __launch_bounds__(256) csr_scan_edges_x2(const long long* __restrict__ row, const long long* __restrict__ col,
                                                         long long E, int n_rows, int n_cols, int row_offset,
                                                         int* __restrict__ rowptr, int* __restrict__ col32, int* __restrict__ flags) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long pairs = E >> 1;
  int bad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += stride) {
    const longlong2 r2 = *reinterpret_cast<const longlong2*>(row + 2 * i);
    const longlong2 c2 = *reinterpret_cast<const longlong2*>(col + 2 * i);
    long long pr = -1, pc = -1;
    if (i > 0) { pr = row[2 * i - 1] - row_offset; pc = col[2 * i - 1]; }
    const long long rr[2] = {r2.x - row_offset, r2.y - row_offset}, cc[2] = {c2.x, c2.y};
    int out[2] = {0, 0};
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const long long e = 2 * i + j, r = rr[j], c = cc[j];
      if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) { bad |= 2; pr = r; pc = c; continue; }
      out[j] = (int)c;
      if (e > 0) {
        if (pr > r || (pr == r && pc >= c)) bad |= 1;
        if (pr < 0 || pr >= n_rows) pr = r;
      }
      for (long long q = pr + 1; q <= r; ++q) rowptr[q] = (int)e;
      if (e == E - 1)
        for (long long q = r + 1; q <= n_rows; ++q) rowptr[q] = (int)E;
      pr = r;
      pc = c;
    }
    *reinterpret_cast<int2*>(col32 + 2 * i) = make_int2(out[0], out[1]);
  }
  if (bad) atomicOr(flags, bad);
}

__global__ void csr_empty(int n_rows, int* rowptr) {
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= n_rows; i += gridDim.x * blockDim.x) rowptr[i] = 0;
}

// Single-block exclusive scan of ceil(deg/chunk) -> taskptr, n_tasks.  n_rows <= a few million.
__global__ void __launch_bounds__(1024) task_scan(const int* __restrict__ rowptr, int n_rows, int chunk,
                                                  int* __restrict__ taskptr, int* __restrict__ n_tasks) {
  pdl_wait();
  __shared__ int strip_sum[1024];
  const int t = threadIdx.x;
  const int per = (n_rows + 1023) / 1024;
  const int lo = min(t * per, n_rows), hi = min(lo + per, n_rows);
  int s = 0;
  for (int r = lo; r < hi; ++r) s += (rowptr[r + 1] - rowptr[r] + chunk - 1) / chunk;
  strip_sum[t] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {          // Hillis-Steele inclusive scan
    int v = (t >= off) ? strip_sum[t - off] : 0;
    __syncthreads();
    strip_sum[t] += v;
    __syncthreads();
  }
  int run = (t == 0) ? 0 : strip_sum[t - 1];
  for (int r = lo; r < hi; ++r) {
    taskptr[r] = run;
    run += (rowptr[r + 1] - rowptr[r] + chunk - 1) / chunk;
  }
  if (t == 1023) {
    taskptr[n_rows] = strip_sum[1023];
    *n_tasks = strip_sum[1023];
  }
}

__global__ void task_fill(const int* __restrict__ taskptr, int n_rows, int max_tasks, int* __restrict__ task_row) {
  pdl_wait();
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += gridDim.x * blockDim.x)
    for (int t = taskptr[r]; t < taskptr[r + 1] && t < max_tasks; ++t) task_row[t] = r;
}

// deferred validation: an invalid edge list must not reach the sweeps as inconsistent tables -> turn it into an empty graph
// (rowptr = 0 everywhere, hence no tasks); the host raises when it reads the flag word later
__global__ void csr_guard(const int* __restrict__ flags, int n_rows, int* __restrict__ rowptr) {
  pdl_wait();
  if (*flags == 0) return;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r <= n_rows; r += gridDim.x * blockDim.x) rowptr[r] = 0;
}

template <typename IdxT>
static int graph_build_impl(mpn_graph* g, const IdxT* row, const IdxT* col, cudaStream_t st, int* flags_dev = nullptr,
                            int* flags_host_pinned = nullptr) {
  MPN_REQUIRE(g != nullptr, "graph is NULL");
  MPN_REQUIRE(g->n_nodes > 0 && g->n_cols > 0 && g->n_edges >= 0, "bad graph sizes");
  MPN_REQUIRE(g->n_edges < (1ll << 31), "n_edges must be < 2^31 per shard");
  MPN_REQUIRE(g->chunk >= 32 && g->chunk <= 4096 && (g->chunk & (g->chunk - 1)) == 0, "chunk must be a power of two in [32,4096]");
  MPN_REQUIRE(g->max_tasks >= g->n_edges / g->chunk + g->n_nodes, "max_tasks too small (need E/chunk + N)");
  MPN_REQUIRE(g->rowptr && g->taskptr && g->task_row && g->n_tasks && (g->col || g->n_edges == 0), "graph table pointer is NULL");
  const bool deferred = flags_dev != nullptr && flags_host_pinned != nullptr;
  int* flags = deferred ? flags_dev : g->n_tasks;  // (sync mode: n_tasks doubles as the flag word until task_scan overwrites it)
  MPN_CUDA_OK(cudaMemsetAsync(flags, 0, sizeof(int), st));
  if (g->n_edges == 0) {
    mpn::launch(csr_empty, div_up(g->n_nodes + 1, 256), 256, 0, st, g->n_nodes, g->rowptr);
  } else {
    int grid = (int)min((long long)kNumSMs * 16, (long long)div_up(g->n_edges, 256));
    const bool x2 = sizeof(IdxT) == 8 && (g->n_edges & 1) == 0 && ((((uintptr_t)row) | ((uintptr_t)col)) & 15) == 0 &&
                    (((uintptr_t)g->col) & 7) == 0;
    if (x2)
      mpn::launch(csr_scan_edges_x2, grid, 256, 0, st, (const long long*)row, (const long long*)col, g->n_edges, g->n_nodes, g->n_cols,
                                              g->row_offset, g->rowptr, g->col, flags);
    else
      mpn::launch(csr_scan_edges<IdxT>, grid, 256, 0, st, row, col, g->n_edges, g->n_nodes, g->n_cols, g->row_offset,
                                                 g->rowptr, g->col, flags);
  }
  MPN_LAUNCH_OK();
  if (deferred) {
    // no host round trip on the critical path: the flag word travels to pinned host memory behind the scan, the tables of an
    // invalid edge list are emptied on the device, and the caller checks *flags_host_pinned at its next synchronisation point
    MPN_CUDA_OK(cudaMemcpyAsync(flags_host_pinned, flags, sizeof(int), cudaMemcpyDeviceToHost, st));
    mpn::launch(csr_guard, min(kNumSMs, div_up(g->n_nodes + 1, 256)), 256, 0, st, flags, g->n_nodes, g->rowptr);
    MPN_LAUNCH_OK();
  } else {
    int h_flags = 0;
    MPN_CUDA_OK(cudaMemcpyAsync(&h_flags, flags, sizeof(int), cudaMemcpyDeviceToHost, st));
    MPN_CUDA_OK(cudaStreamSynchronize(st));
    if (h_flags & 2) {
      set_error("edge_index has node ids outside [row_offset, row_offset+n_nodes) x [0, n_cols)");
      return MPN_ERR_INVALID;
    }
    if (h_flags & 1) {
      set_error("edge_index is not strictly (row, col)-sorted (unsorted or duplicate edges)");
      return MPN_ERR_UNSORTED;
    }
  }
  mpn::launch(task_scan, 1, 1024, 0, st, g->rowptr, g->n_nodes, g->chunk, g->taskptr, g->n_tasks);
  MPN_LAUNCH_OK();
  mpn::launch(task_fill, min(kNumSMs * 8, div_up(g->n_nodes, 256)), 256, 0, st, g->taskptr, g->n_nodes, g->max_tasks, g->task_row);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

struct CamLayout {
  int n_cams;
  int ptr[MPN_MAX_CAMERAS + 1];            // first node of each camera
  long long ebase[MPN_MAX_CAMERAS + 1];    // first edge of each camera's row block
};

// One warp writes the columns of global row r: [c0, c0 + deg + nk) without the row's own camera segment [lo, lo + nk), in
// ascending order from local edge le0 on (coalesced, no per-edge division).  The reference's int64 pair goes to edge_index_out
// ([2,E]) when that is not NULL.
__device__ __forceinline__ void cross_camera_row_cols(int lane, long long r, int c0, int deg, int lo, int nk, long long le0,
                                                      long long E, int* __restrict__ col32, long long* __restrict__ edge_index_out) {
  for (int idx = lane; idx < deg; idx += 32) {
    int c = c0 + idx;
    if (c >= lo) c += nk;
    col32[le0 + idx] = c;
    if (edge_index_out) { edge_index_out[le0 + idx] = r; edge_index_out[E + le0 + idx] = c; }
  }
}

// dense cross-camera graph straight from the camera layout: row r (camera k) lists every node outside [ptr[k], ptr[k+1]).
// Works on a row block [row0, row0 + n_rows): local edge e corresponds to global edge e + gbase.
__global__ void __launch_bounds__(256) cross_camera_kernel(const CamLayout L, int n_total, int row0, int n_rows, long long gbase,
                                                           long long E, int* __restrict__ rowptr, int* __restrict__ col32,
                                                           long long* __restrict__ edge_index_out) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long long lr = tid; lr <= n_rows; lr += stride) {            // rowptr of the local rows
    const long long r = row0 + lr;
    if (lr == n_rows) { rowptr[lr] = (int)E; continue; }
    int k = 0;
    while (k + 1 < L.n_cams && r >= L.ptr[k + 1]) ++k;
    const long long deg = n_total - (L.ptr[k + 1] - L.ptr[k]);
    rowptr[lr] = (int)(L.ebase[k] + (r - L.ptr[k]) * deg - gbase);
  }
  // one warp per local row: its columns are 0..n_total-1 without the row's own camera block
  const int lane = threadIdx.x & 31;
  const long long warp0 = tid >> 5, nwarps = stride >> 5;
  for (long long lr = warp0; lr < n_rows; lr += nwarps) {
    const long long r = row0 + lr;
    int k = 0;
    while (k + 1 < L.n_cams && r >= L.ptr[k + 1]) ++k;
    const int lo = L.ptr[k], nk = L.ptr[k + 1] - lo;
    const int deg = n_total - nk;
    cross_camera_row_cols(lane, r, 0, deg, lo, nk, L.ebase[k] + (r - lo) * (long long)deg - gbase, E, col32, edge_index_out);
  }
}

// last i in [0, n) with a[i] <= v (a ascending, a[0] <= v)
__device__ __forceinline__ int last_le(const int* __restrict__ a, int n, long long v) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (a[mid] <= v) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Block-diagonal cross-camera tables of a batch: row r of graph g = [gs, ge) in camera segment [ss, se) lists [gs, ss) and
// [se, ge).  Segment s = (graph, camera) starts at node seg_ptr[s] and its row block at edge seg_ebase[s]; graph g owns
// segments [graph_seg[g], graph_seg[g+1]).  One warp per row finds its segment and graph (binary searches that every lane makes
// on the same words), writes rowptr / node_gid (and graph_nptr on a graph's first row), then the row's columns.
__global__ void __launch_bounds__(256) cross_camera_batched_kernel(const int* __restrict__ seg_ptr, int n_segs,
                                                                   const int* __restrict__ graph_seg, int n_graphs,
                                                                   const long long* __restrict__ seg_ebase, int n, long long E,
                                                                   int* __restrict__ rowptr, int* __restrict__ col32,
                                                                   int* __restrict__ node_gid, int* __restrict__ graph_nptr,
                                                                   long long* __restrict__ edge_index_out) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += nwarps) {
    const int s = last_le(seg_ptr, n_segs, r);
    const int g = last_le(graph_seg, n_graphs, s);
    const int gs = seg_ptr[graph_seg[g]], ge = seg_ptr[graph_seg[g + 1]];
    const int ss = seg_ptr[s], nk = seg_ptr[s + 1] - ss;
    const int deg = ge - gs - nk;
    const long long le0 = seg_ebase[s] + (r - ss) * (long long)deg;
    if (lane == 0) {
      rowptr[r] = (int)le0;
      node_gid[r] = g;
      if (r == gs) graph_nptr[g] = gs;
      if (r == n - 1) { rowptr[n] = (int)E; graph_nptr[n_graphs] = n; }
    }
    cross_camera_row_cols(lane, r, gs, deg, ss, nk, le0, E, col32, edge_index_out);
  }
}

}  // namespace mpn

extern "C" {

int64_t mpn_cross_camera_edges(const int32_t* cam_ptr, int32_t n_cams) {
  if (!cam_ptr || n_cams < 1) return -1;
  const long long n = cam_ptr[n_cams];
  long long e = 0;
  for (int k = 0; k < n_cams; ++k) {
    const long long nk = cam_ptr[k + 1] - cam_ptr[k];
    if (nk < 0) return -1;
    e += nk * (n - nk);
  }
  return e;
}

// global edge id of the first edge of row r
static long long cross_camera_row_start(const int32_t* cam_ptr, int n_cams, int n_total, long long r) {
  long long run = 0;
  for (int k = 0; k < n_cams; ++k) {
    const long long nk = cam_ptr[k + 1] - cam_ptr[k], deg = n_total - nk;
    if (r < cam_ptr[k + 1]) return run + (r - cam_ptr[k]) * deg;
    run += nk * deg;
  }
  return run;
}

int64_t mpn_cross_camera_block_edges(const int32_t* cam_ptr, int32_t n_cams, int32_t row0, int32_t n_rows) {
  if (!cam_ptr || n_cams < 1 || row0 < 0 || n_rows < 0 || row0 + n_rows > cam_ptr[n_cams]) return -1;
  const int n_total = cam_ptr[n_cams];
  return cross_camera_row_start(cam_ptr, n_cams, n_total, (long long)row0 + n_rows) - cross_camera_row_start(cam_ptr, n_cams, n_total, row0);
}

int mpn_graph_build_cross_camera(mpn_graph* g, const int32_t* cam_ptr, int32_t n_cams, int64_t* edge_index_out, void* stream) {
  using namespace mpn;
  MPN_REQUIRE(g && cam_ptr, "cross_camera: NULL argument");
  MPN_REQUIRE(n_cams >= 1 && n_cams <= MPN_MAX_CAMERAS, "cross_camera: n_cams must be in [1,%d]", MPN_MAX_CAMERAS);
  MPN_REQUIRE(cam_ptr[0] == 0 && cam_ptr[n_cams] == g->n_cols && g->row_offset >= 0 && g->row_offset + g->n_nodes <= g->n_cols,
              "cross_camera: cam_ptr must run from 0 to n_cols and the row block must lie inside it");
  const int n_total = g->n_cols;
  const long long gbase = cross_camera_row_start(cam_ptr, n_cams, n_total, g->row_offset);
  const long long E = cross_camera_row_start(cam_ptr, n_cams, n_total, (long long)g->row_offset + g->n_nodes) - gbase;
  MPN_REQUIRE(E >= 0 && E == g->n_edges, "cross_camera: g->n_edges (%lld) must be %lld", (long long)g->n_edges, E);
  MPN_REQUIRE(E < (1ll << 31), "n_edges must be < 2^31");
  MPN_REQUIRE(g->chunk >= 32 && g->chunk <= 4096 && (g->chunk & (g->chunk - 1)) == 0, "chunk must be a power of two in [32,4096]");
  MPN_REQUIRE(g->max_tasks >= g->n_edges / g->chunk + g->n_nodes, "max_tasks too small (need E/chunk + N)");
  MPN_REQUIRE(g->rowptr && g->taskptr && g->task_row && g->n_tasks && (g->col || E == 0), "graph table pointer is NULL");
  CamLayout L;
  L.n_cams = n_cams;
  long long run = 0;
  for (int k = 0; k <= n_cams; ++k) {
    L.ptr[k] = cam_ptr[k];
    L.ebase[k] = run;
    if (k < n_cams) run += (long long)(cam_ptr[k + 1] - cam_ptr[k]) * (n_total - (cam_ptr[k + 1] - cam_ptr[k]));
  }
  cudaStream_t st = (cudaStream_t)stream;
  const long long work = E > g->n_nodes ? E : g->n_nodes + 1;
  mpn::launch(cross_camera_kernel, (int)min((long long)kNumSMs * 16, (work + 255) / 256), 256, 0, st, L, n_total, g->row_offset, g->n_nodes, gbase, E,
                                                                                          g->rowptr, g->col, (long long*)edge_index_out);
  MPN_LAUNCH_OK();
  mpn::launch(task_scan, 1, 1024, 0, st, g->rowptr, g->n_nodes, g->chunk, g->taskptr, g->n_tasks);
  MPN_LAUNCH_OK();
  mpn::launch(task_fill, min(kNumSMs * 8, div_up(g->n_nodes, 256)), 256, 0, st, g->taskptr, g->n_nodes, g->max_tasks, g->task_row);
  MPN_LAUNCH_OK();
  g->layout_hint = MPN_LAYOUT_ONE_GAP;         // every row: all nodes but its own camera's range
  return MPN_OK;
}

int64_t mpn_cross_camera_batched_layout(const int32_t* seg_ptr, int32_t n_segs, const int32_t* graph_seg, int32_t n_graphs,
                                        int64_t* seg_ebase) {
  if (!seg_ptr || !graph_seg || n_segs < 1 || n_graphs < 1) return -1;
  if (seg_ptr[0] != 0 || graph_seg[0] != 0 || graph_seg[n_graphs] != n_segs) return -1;
  for (int s = 0; s < n_segs; ++s)
    if (seg_ptr[s + 1] <= seg_ptr[s]) return -1;
  long long e = 0;
  for (int g = 0; g < n_graphs; ++g) {
    const int s0 = graph_seg[g], s1 = graph_seg[g + 1];
    if (s1 <= s0) return -1;
    const long long ng = (long long)seg_ptr[s1] - seg_ptr[s0];
    for (int s = s0; s < s1; ++s) {
      const long long nk = (long long)seg_ptr[s + 1] - seg_ptr[s];
      if (seg_ebase) seg_ebase[s] = e;
      e += nk * (ng - nk);
    }
  }
  if (seg_ebase) seg_ebase[n_segs] = e;
  return e;
}

int mpn_graph_build_cross_camera_batched(mpn_graph* g, const int32_t* seg_ptr, int32_t n_segs, const int32_t* graph_seg,
                                         const int64_t* seg_ebase, int64_t* edge_index_out, void* stream) {
  using namespace mpn;
  MPN_REQUIRE(g && seg_ptr && graph_seg && seg_ebase, "cross_camera_batched: NULL argument");
  MPN_REQUIRE(n_segs >= 1 && g->n_graphs >= 1 && n_segs >= g->n_graphs, "cross_camera_batched: need n_segs >= n_graphs >= 1");
  MPN_REQUIRE(g->n_nodes > 0 && g->n_cols == g->n_nodes && g->row_offset == 0, "cross_camera_batched: batched graphs cannot be row-sharded");
  MPN_REQUIRE(g->n_edges >= 0 && g->n_edges < (1ll << 31), "n_edges must be < 2^31");
  MPN_REQUIRE(g->chunk >= 32 && g->chunk <= 4096 && (g->chunk & (g->chunk - 1)) == 0, "chunk must be a power of two in [32,4096]");
  MPN_REQUIRE(g->max_tasks >= g->n_edges / g->chunk + g->n_nodes, "max_tasks too small (need E/chunk + N)");
  MPN_REQUIRE(g->rowptr && g->taskptr && g->task_row && g->n_tasks && (g->col || g->n_edges == 0) && g->node_gid && g->graph_nptr,
              "graph table pointer is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  mpn::launch(cross_camera_batched_kernel, min(kNumSMs * 16, div_up((long long)g->n_nodes * 32, 256)), 256, 0, st,
              seg_ptr, n_segs, graph_seg, g->n_graphs, (const long long*)seg_ebase, g->n_nodes, (long long)g->n_edges, g->rowptr,
              g->col, g->node_gid, g->graph_nptr, (long long*)edge_index_out);
  MPN_LAUNCH_OK();
  mpn::launch(task_scan, 1, 1024, 0, st, g->rowptr, g->n_nodes, g->chunk, g->taskptr, g->n_tasks);
  MPN_LAUNCH_OK();
  mpn::launch(task_fill, min(kNumSMs * 8, div_up(g->n_nodes, 256)), 256, 0, st, g->taskptr, g->n_nodes, g->max_tasks, g->task_row);
  MPN_LAUNCH_OK();
  g->layout_hint = MPN_LAYOUT_UNKNOWN;         // a row lists its own graph's columns only, not all columns but one gap
  return MPN_OK;
}

int mpn_abi_version(void) { return MPN_B200_ABI_VERSION; }
const char* mpn_last_error(void) { return mpn::g_err; }
uint64_t mpn_kernel_launches(void) { return mpn::g_kernel_launches; }

int mpn_set_pdl(int enable) {
  if (enable >= 0) mpn::g_pdl_launch = enable != 0;
  return mpn::g_pdl_launch ? 2 : 1;
}

int mpn_check_device(int dev) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || dev < 0 || dev >= n) {
    mpn::set_error("no CUDA device %d (device count %d): the MPN path has no CPU fallback", dev, n);
    cudaGetLastError();
    return MPN_ERR_NO_DEVICE;
  }
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess || p.major != 10) {
    mpn::set_error("device %d is sm_%d%d; this library is built for sm_100a only", dev, p.major, p.minor);
    return MPN_ERR_NO_DEVICE;
  }
  return MPN_OK;
}

int mpn_graph_build(mpn_graph* g, const int64_t* edge_index_dev, void* stream) {
  if (!g) { mpn::set_error("graph is NULL"); return MPN_ERR_INVALID; }
  return mpn::graph_build_impl<long long>(g, (const long long*)edge_index_dev,
                                          (const long long*)edge_index_dev + g->n_edges, (cudaStream_t)stream);
}

int mpn_graph_build_deferred(mpn_graph* g, const int64_t* edge_index_dev, int32_t* flags_dev, int32_t* flags_host_pinned, void* stream) {
  if (!g || !flags_dev || !flags_host_pinned) { mpn::set_error("graph_build_deferred: NULL argument"); return MPN_ERR_INVALID; }
  return mpn::graph_build_impl<long long>(g, (const long long*)edge_index_dev, (const long long*)edge_index_dev + g->n_edges,
                                          (cudaStream_t)stream, flags_dev, flags_host_pinned);
}

int mpn_graph_build_i32(mpn_graph* g, const int32_t* row_dev, const int32_t* col_dev, void* stream) {
  return mpn::graph_build_impl<int>(g, row_dev, col_dev, (cudaStream_t)stream);
}

}  // extern "C"
