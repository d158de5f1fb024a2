// MOTMPNet.forward (models/mpn.py:250-299) as HBM-bound edge sweeps + small node kernels.
//
// Algebra (exact up to fp32 re-association, see DESIGN.md):
//   edge update  y  = W_e[68->4]·[h_r;h_c;e] + b = Ps[row] + Pd[col] + We·e      (models/mpn.py:48,68-69)
//                e' = relu(BN(y))                       BN over all E edges        (models/mlp.py:16)
//   node update  z  = W_n[36->32]·[h_r;e'] + b = A[row] + Wn·e'                    (models/mpn.py:97-98)
//                h' = segment_sum_row(relu(BN(z)))      BN over all E edges        (models/mpn.py:99,202)
// BatchNorm uses batch statistics, so every BN is a global reduction followed by a second sweep.
// Moments are accumulated in fp64, block partials are reduced in a fixed order (deterministic).
#include <mutex>
#include <new>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.h"
#include "tcgen05.cuh"

namespace mpn {

// ------------------------------------------------------------------------------------------------
// folded constants living in device memory (floats)
// ------------------------------------------------------------------------------------------------
enum {
  FC_ENC1_W = 0,     // [4][2]  s1 * W1
  FC_ENC1_C = 8,     // [4]     s1 * b1 + t1
  FC_ENC2_W = 12,    // [4][4]  s2 * W2
  FC_ENC2_C = 28,    // [4]
  FC_EDGE_WE = 32,   // [4][4]  W_edge[:, 64:68]
  FC_BN3_S = 48,     // [4]     edge-model BN scale of the most recent finalised step
  FC_BN3_T = 52,     // [4]
  FC_NODE_WE = 64,   // [32][4] s4 * W_node[:, 32:36]
  FC_BN4_S = 192,    // [32]
  FC_BN4_T = 224,    // [32]
  FC_CLS_W = 256,    // [2][4]
  FC_CLS_B = 264,    // [2]
  FC_EDGE_WE0 = 272, // [4][4]  reattach_initial_edges: W_edge columns of the initial edge encoding e0 (steps >= 2)
  FC_TOTAL = 288
};

constexpr int SUMS = MPN_SUMS_DOUBLES;     // 96 doubles per partial row
constexpr int SWEEP_THREADS = 256;
constexpr int SWEEP_BLOCKS_PER_SM = 4;
constexpr int SWEEP_GRID = kNumSMs * SWEEP_BLOCKS_PER_SM;
// The node-moment sweep over stored y (SB) is capped at 80 registers (__launch_bounds__ minimum of 3 blocks; no spills), so 3
// blocks = 24 warps fit on an SM and its grid is exactly one resident wave: a second, partial wave would start late and finish
// late.  The sweep is bound by the bytes each SM has in flight; 24 warps instead of 16 at the same loads per lane is the gain.
// (The variant that recomputes y spills at 80 registers and keeps 2 blocks per SM and SWEEP_GRID.)
constexpr int SWEEP_RESIDENT_BLOCKS = 3;
constexpr int SWEEP_RESIDENT_GRID = kNumSMs * SWEEP_RESIDENT_BLOCKS;
constexpr float BN_EPS = 1e-5f;

struct EdgeConsts {           // staged in shared memory by every sweep
  float v[FC_TOTAL];
};

__device__ __forceinline__ void load_consts(EdgeConsts& sc, const float* __restrict__ consts) {
  for (int i = threadIdx.x; i < FC_TOTAL; i += blockDim.x) sc.v[i] = consts[i];
  __syncthreads();
}

// batched graphs: every graph has its own folded constants; a warp re-stages them when its task moves to another graph
constexpr int TASK_PART = 16;                  // doubles per task in the per-task moment partials (batched mode)
__device__ __forceinline__ void warp_load_consts(EdgeConsts& sc, const float* __restrict__ consts_g, int lane) {
  __syncwarp();
  for (int i = lane; i < FC_TOTAL; i += 32) sc.v[i] = consts_g[i];
  __syncwarp();
}

// encoder edge MLP with folded BatchNorm: 2 -> 4 -> 4, ReLU after each (models/mpn.py:128-142)
__device__ __forceinline__ void enc_layer1(const EdgeConsts& sc, float2 ea, float (&a1)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    a1[j] = fmaxf(fmaf(sc.v[FC_ENC1_W + 2 * j], ea.x, fmaf(sc.v[FC_ENC1_W + 2 * j + 1], ea.y, sc.v[FC_ENC1_C + j])), 0.f);
}
__device__ __forceinline__ void enc_layer2_pre(const float* __restrict__ w2 /*[4][4]*/, const float* __restrict__ c2,
                                               const float (&a1)[4], float (&u)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float s = c2[j];
#pragma unroll
    for (int k = 0; k < 4; ++k) s = fmaf(w2[4 * j + k], a1[k], s);
    u[j] = s;
  }
}
__device__ __forceinline__ void enc_full(const EdgeConsts& sc, float2 ea, float (&e0)[4]) {
  float a1[4];
  enc_layer1(sc, ea, a1);
  enc_layer2_pre(&sc.v[FC_ENC2_W], &sc.v[FC_ENC2_C], a1, e0);
#pragma unroll
  for (int j = 0; j < 4; ++j) e0[j] = fmaxf(e0[j], 0.f);
}
// y = Ps[row] + Pd[col] + We·e_in
__device__ __forceinline__ void edge_pre(const EdgeConsts& sc, const float4 ps, const float4 pd, const float (&ein)[4], float (&y)[4]) {
  const float p[4] = {ps.x + pd.x, ps.y + pd.y, ps.z + pd.z, ps.w + pd.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float s = p[j];
#pragma unroll
    for (int k = 0; k < 4; ++k) s = fmaf(sc.v[FC_EDGE_WE + 4 * j + k], ein[k], s);
    y[j] = s;
  }
}
__device__ __forceinline__ void bn3_relu(const EdgeConsts& sc, const float (&y)[4], float (&e)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) e[j] = fmaxf(fmaf(sc.v[FC_BN3_S + j], y[j], sc.v[FC_BN3_T + j]), 0.f);
}

struct TaskRange {
  int row, beg, end;
};
__device__ __forceinline__ TaskRange task_range(const mpn_graph& g, int t) {
  TaskRange r;
  r.row = g.task_row[t];
  const int rb = g.rowptr[r.row];
  r.beg = rb + (t - g.taskptr[r.row]) * g.chunk;
  r.end = min(r.beg + g.chunk, g.rowptr[r.row + 1]);
  return r;
}

// Task ranges two strides ahead: task_range() is a chain of dependent loads (task_row -> rowptr/taskptr), ~2 L2 round trips that
// a warp would otherwise pay at the start of every task.  Stage A fetches the row of task t + 2*stride, stage B the range of task
// t + stride from the row fetched one iteration earlier; the current task never waits.  stride < 0 walks the tasks backwards.
__device__ __forceinline__ bool task_in(int t, int n_tasks) { return (unsigned)t < (unsigned)n_tasks; }
struct TaskPrefetch {
  TaskRange cur, nxt;
  int row_n;                                         // row of task t + stride (stage A result of the previous iteration)
  __device__ __forceinline__ void start(const mpn_graph& g, int t, int stride, int n_tasks) {
    if (task_in(t, n_tasks)) cur = task_range(g, t);
    row_n = task_in(t + stride, n_tasks) ? g.task_row[t + stride] : 0;
  }
  // call at the top of the iteration for task t; afterwards `cur` is valid; call rotate() at the bottom
  __device__ __forceinline__ int issue(const mpn_graph& g, int t, int stride, int n_tasks) {
    if (task_in(t + stride, n_tasks)) {
      const int tn = t + stride;
      nxt.row = row_n;
      const int rb = g.rowptr[row_n];
      nxt.beg = rb + (tn - g.taskptr[row_n]) * g.chunk;
      nxt.end = min(nxt.beg + g.chunk, g.rowptr[row_n + 1]);
    }
    return task_in(t + 2 * stride, n_tasks) ? g.task_row[t + 2 * stride] : 0;
  }
  __device__ __forceinline__ void rotate(int row_nn) { cur = nxt; row_n = row_nn; }
};

// ------------------------------------------------------------------------------------------------
// finalize: fixed-order reduction of block partials -> sums; sums -> folded constants.  Runs either as its own
// one-block kernel (sharded runs: the host all-reduces the sums in between) or inside the LAST block of the sweep that
// produced the partials (single-GPU: saves a launch per BatchNorm).  Partials written by other blocks of the same kernel
// are read with ld.global.cg (L2), never through the non-coherent path.
// ------------------------------------------------------------------------------------------------
struct PeerArgs;
struct FinArgs {
  int stage;
  const double* partials;
  int n_partials;
  int row_stride;             // rows from one partial row read by the fold to the next (1; FOLD_GROUP for the group rows)
  const double* partials2;
  int n_partials2;
  double* sums;
  float* consts;
  const float* small;
  double n_total;
  unsigned int* counter;      // != nullptr: fuse into the producing kernel's last block
  double* n_total_dev;        // != nullptr: total edge count lives on the device (exchanged with the first all-reduce)
  double local_edges;         // this rank's edge count (sharded runs)
  const unsigned long long* fixed;   // ENC0, optional: 2^40 fixed-point sums of the edges the fused edge-feature kernel left to the
                              // refine pass (gram_ef.cu / edge_features.cu), added to columns 0..4
  const struct PeerArgs* peers;      // sharded runs with the finalize fused into the sweep's last block: device copy of the peer
  unsigned long long seq;            // table and this exchange's sequence number (peers == nullptr: single GPU)
  int re_e;                   // reattach_initial_edges: 0 off, 1 on (y of the current step is recomputed later: keep the folded
                              // step-1 weights), 2 on and y stored (switch to the split weights after the first edge update)
};

__device__ __forceinline__ int fin_ncols(int stage) { return (stage == MPN_STAGE_NODE) ? 74 : 8; }   // live partial columns

// Fixed-order fold of n_rows partial rows (row r at rows + r * row_stride * SUMS); thread k < ncols returns column k's total, the
// others 0.  Every thread of the block calls it.  It runs in the serial tail of a sweep: a thread owns a PAIR of adjacent live
// columns (one 16-byte L2 load per partial row) and every `groups`-th row, four loads in flight; the row groups are then added
// through shared memory in group order.  Fixed pattern => bit-reproducible.
__device__ __forceinline__ double fold_rows(const double* rows, int n_rows, int row_stride, int ncols) {
  __shared__ double red[2048];
  const int k = threadIdx.x;
  const size_t rs = (size_t)row_stride * SUMS;
  const int pairs = ncols >> 1;
  int groups = (int)blockDim.x / pairs;
  if (groups * ncols > 2048) groups = 2048 / ncols;
  if (k < groups * pairs) {
    const int cp = k % pairs, gi = k / pairs;
    const double* base = rows + 2 * cp;
    double2 a0 = make_double2(0.0, 0.0), a1 = a0, a2 = a0, a3 = a0;
    int p = gi;
    for (; p + 3 * groups < n_rows; p += 4 * groups) {
      const double2 v0 = __ldcg(reinterpret_cast<const double2*>(base + (size_t)p * rs));
      const double2 v1 = __ldcg(reinterpret_cast<const double2*>(base + (size_t)(p + groups) * rs));
      const double2 v2 = __ldcg(reinterpret_cast<const double2*>(base + (size_t)(p + 2 * groups) * rs));
      const double2 v3 = __ldcg(reinterpret_cast<const double2*>(base + (size_t)(p + 3 * groups) * rs));
      a0.x += v0.x; a0.y += v0.y; a1.x += v1.x; a1.y += v1.y; a2.x += v2.x; a2.y += v2.y; a3.x += v3.x; a3.y += v3.y;
    }
    for (; p < n_rows; p += groups) {
      const double2 v = __ldcg(reinterpret_cast<const double2*>(base + (size_t)p * rs));
      a0.x += v.x; a0.y += v.y;
    }
    red[gi * ncols + 2 * cp] = (a0.x + a1.x) + (a2.x + a3.x);
    red[gi * ncols + 2 * cp + 1] = (a0.y + a1.y) + (a2.y + a3.y);
  }
  __syncthreads();
  double t = 0.0;
  if (k < ncols)
    for (int gi = 0; gi < groups; ++gi) t += red[gi * ncols + k];
  __syncthreads();                                   // red is free again
  return t;
}

__device__ __forceinline__ void finalize_body(const FinArgs& f, int do_reduce, int do_consts) {
  const int stage = f.stage;
  double* sums = f.sums;
  float* consts = f.consts;
  const float* small = f.small;
  const int k = threadIdx.x;
  if (do_reduce) {
    double t = fold_rows(f.partials, f.n_partials, f.row_stride, fin_ncols(stage));
    if (k < SUMS) {
      if (stage == MPN_STAGE_ENC0 && f.fixed != nullptr && k < 5)
        t += (double)(long long)__ldcg(f.fixed + k) * (1.0 / 1099511627776.0);
      sums[k] = t;
    }
  }
  __syncthreads();
  if (!do_consts) return;
  const double inv_n = 1.0 / (f.n_total_dev ? *f.n_total_dev : f.n_total);
  if (stage == MPN_STAGE_ENC0) {
    // static constants
    // step 1 of reattach_initial_edges sees e_in = [e0 | e0]: one folded 4x4 block (We0 + We1)
    if (k < 16) consts[FC_EDGE_WE + k] = small[MPN_W_EDGE_W + (k >> 2) * 68 + 64 + (k & 3)] +
                                         (f.re_e ? small[MPN_W_EDGE_W0 + (k >> 2) * 68 + 64 + (k & 3)] : 0.f);
    if (k < 16) consts[FC_EDGE_WE0 + k] = 0.f;
    if (k < 8) consts[FC_CLS_W + k] = small[MPN_W_CLS_W + k];
    if (k < 2) consts[FC_CLS_B + k] = small[MPN_W_CLS_B + k];
    if (k < 4) {
      const double ma = sums[0] * inv_n, mb = sums[1] * inv_n;
      const double caa = sums[2] * inv_n - ma * ma, cab = sums[3] * inv_n - ma * mb, cbb = sums[4] * inv_n - mb * mb;
      const double w0 = small[MPN_W_ENC1_W + 2 * k], w1 = small[MPN_W_ENC1_W + 2 * k + 1], b = small[MPN_W_ENC1_B + k];
      const double mean = w0 * ma + w1 * mb + b;
      double var = w0 * w0 * caa + 2.0 * w0 * w1 * cab + w1 * w1 * cbb;
      if (var < 0.0) var = 0.0;
      const double s = (double)small[MPN_W_ENC1_G + k] / sqrt(var + (double)BN_EPS);
      const double t = (double)small[MPN_W_ENC1_BETA + k] - s * mean;
      consts[FC_ENC1_W + 2 * k] = (float)(s * w0);
      consts[FC_ENC1_W + 2 * k + 1] = (float)(s * w1);
      consts[FC_ENC1_C + k] = (float)(s * b + t);
    }
  } else if (stage == MPN_STAGE_ENC1 || stage == MPN_STAGE_EDGE) {
    if (k < 4) {
      const double mean = sums[k] * inv_n;
      double var = sums[4 + k] * inv_n - mean * mean;
      if (var < 0.0) var = 0.0;
      const int G = (stage == MPN_STAGE_ENC1) ? MPN_W_ENC2_G : MPN_W_EDGE_G;
      const int B = (stage == MPN_STAGE_ENC1) ? MPN_W_ENC2_BETA : MPN_W_EDGE_BETA;
      const double s = (double)small[G + k] / sqrt(var + (double)BN_EPS);
      const double t = (double)small[B + k] - s * mean;
      if (stage == MPN_STAGE_ENC1) {
        for (int j = 0; j < 4; ++j) consts[FC_ENC2_W + 4 * k + j] = (float)(s * small[MPN_W_ENC2_W + 4 * k + j]);
        consts[FC_ENC2_C + k] = (float)(s * small[MPN_W_ENC2_B + k] + t);
      } else {
        consts[FC_BN3_S + k] = (float)s;
        consts[FC_BN3_T + k] = (float)t;
      }
    }
    if (stage == MPN_STAGE_EDGE && f.re_e == 2 && k < 16) {
      // every later edge update sees e_in = [e0 | e]: the two 4x4 blocks separately (idempotent after the first step)
      consts[FC_EDGE_WE + k] = small[MPN_W_EDGE_W + (k >> 2) * 68 + 64 + (k & 3)];
      consts[FC_EDGE_WE0 + k] = small[MPN_W_EDGE_W0 + (k >> 2) * 68 + 64 + (k & 3)];
    }
  } else if (stage == MPN_STAGE_NODE) {
    if (k < 32) {
      double w[4];
      for (int j = 0; j < 4; ++j) w[j] = small[MPN_W_NODE_W + k * 36 + 32 + j];
      double quad = 0.0;
      int idx = 0;
      for (int a = 0; a < 4; ++a)
        for (int b = a; b < 4; ++b) quad += (a == b ? 1.0 : 2.0) * w[a] * w[b] * sums[64 + idx++];
      const double mean = sums[k] * inv_n;
      double var = (sums[32 + k] + quad) * inv_n - mean * mean;
      if (var < 0.0) var = 0.0;
      const double s = (double)small[MPN_W_NODE_G + k] / sqrt(var + (double)BN_EPS);
      const double t = (double)small[MPN_W_NODE_BETA + k] - s * mean;
      consts[FC_BN4_S + k] = (float)s;
      consts[FC_BN4_T + k] = (float)t;
      for (int j = 0; j < 4; ++j) consts[FC_NODE_WE + 4 * k + j] = (float)(s * w[j]);
    }
  }
}

constexpr int FIN_THREADS = 1024;
__global__ void __launch_bounds__(FIN_THREADS) finalize_kernel(const FinArgs f, int do_reduce, int do_consts) {
  pdl_wait();
  finalize_body(f, do_reduce, do_consts);
}

// ---- collectives fused over NVLink peer memory (sharded runs) ---------------------------------------------------
constexpr int KPEERS = MPN_MAX_PEERS;
struct PeerArgs {
  int rank, world;
  double* sums[KPEERS];
  unsigned long long* flags[KPEERS];
  float* h[KPEERS];
  double* cstats[KPEERS];
};
// moment all-reduce + constant folding: local partials -> my slot -> flag; wait for every rank; add the slots in rank order (the
// same order on every rank => bit-identical totals); fold.  Runs as its own one-block kernel, or inside the last block of the
// sweep that produced the partials (FinArgs::peers): no extra launch, and the partial rows are still hot in L2.
__device__ __forceinline__ void finalize_peer_body(const FinArgs& f, const PeerArgs& P, unsigned long long seq) {
  finalize_body(f, 1, 0);                                   // local block partials -> f.sums
  __syncthreads();
  const int k = threadIdx.x;
  const int slot = (int)(seq & 1ull);
  // the first all-reduce of a forward also carries the edge counts (last, otherwise unused, slot entry)
  if (k == SUMS - 1 && f.stage == MPN_STAGE_ENC0 && f.n_total_dev) f.sums[SUMS - 1] = f.local_edges;
  __syncthreads();
  // PUSH: every rank stores its sums into each peer's memory (slot of this exchange, row = my rank), then raises my flag word IN
  // THE PEER'S memory; a rank polls and reads only its own memory (remote loads cost a NVLink round trip each, remote stores
  // are fire-and-forget).  Double-buffered by the parity of seq: a rank can be at most one exchange ahead of a peer.
  if (k < SUMS) {
    const double v = f.sums[k];
    for (int r = 0; r < P.world; ++r) P.sums[r][((size_t)slot * KPEERS + P.rank) * SUMS + k] = v;
  }
  __threadfence_system();
  __syncthreads();
  if (k < P.world) st_release_sys(P.flags[k] + P.rank, seq);               // flag word [0][my rank] of peer k
  if (k < P.world) wait_flag(P.flags[P.rank] + k, seq);                    // my own memory: word [0][k] raised by rank k
  __syncthreads();
  if (k < SUMS) {
    double t = 0.0;
    for (int r = 0; r < P.world; ++r) {                                     // rank order: the same on every rank
      double v;
      asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(P.sums[P.rank] + ((size_t)slot * KPEERS + r) * SUMS + k));
      t += v;
    }
    f.sums[k] = t;
    if (k == SUMS - 1 && f.stage == MPN_STAGE_ENC0 && f.n_total_dev) *f.n_total_dev = t;
  }
  __syncthreads();
  finalize_body(f, 0, 1);
}
__global__ void __launch_bounds__(1024) finalize_peer_kernel(const FinArgs f, const PeerArgs P, unsigned long long seq) {
  pdl_wait();
  finalize_peer_body(f, P, seq);
}

// h all-gather: publish / wait on the second flag word
__global__ void peer_publish_h_kernel(const PeerArgs P, unsigned long long seq) {
  pdl_wait();
  if (blockIdx.x == 0 && threadIdx.x < P.world) {                         // flag word [1][my rank] of every peer (pushed)
    __threadfence_system();
    st_release_sys(P.flags[threadIdx.x] + KPEERS + P.rank, seq);
  }
}
__global__ void peer_wait_h_kernel(const PeerArgs P, unsigned long long seq) {
  pdl_wait();
  if (blockIdx.x == 0 && threadIdx.x < P.world) wait_flag(P.flags[P.rank] + KPEERS + threadIdx.x, seq);     // own memory
}

// Called by every block at the end of a sweep kernel, after its partial row has been written.  Two-level ticket: the last block of
// each group of FOLD_GROUP consecutive blocks folds the group's rows into the group's first row, and the last of those folds the
// group rows and the constants.  One block folding all 444-592 rows was a serial tail of ~18 us for the 74 live columns of the
// node BatchNorm; two short folds take a few L2 round trips each.  Counters: [0] groups done, [1 + g] blocks of group g done.
constexpr int FOLD_GROUP = 16;
constexpr int FIN_COUNTERS = 1 + (SWEEP_GRID + FOLD_GROUP - 1) / FOLD_GROUP;
__device__ __forceinline__ void finalize_in_last_block(const FinArgs& f) {
  if (f.counter == nullptr) return;
  __shared__ unsigned int s_ticket;
  const int grp = blockIdx.x / FOLD_GROUP, n_groups = (gridDim.x + FOLD_GROUP - 1) / FOLD_GROUP;
  const int grp_blocks = min(FOLD_GROUP, (int)gridDim.x - grp * FOLD_GROUP);
  __threadfence();                                   // publish this block's partials
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(f.counter + 1 + grp, 1u);
  __syncthreads();
  if (s_ticket != (unsigned)grp_blocks - 1) return;
  __threadfence();
  double* grp_row = const_cast<double*>(f.partials) + (size_t)grp * FOLD_GROUP * SUMS;
  const int ncols = fin_ncols(f.stage);
  const double t = fold_rows(grp_row, grp_blocks, 1, ncols);
  if (threadIdx.x < ncols) grp_row[threadIdx.x] = t;
  if (threadIdx.x == 0) f.counter[1 + grp] = 0u;     // ready for the next sweep
  __threadfence();                                   // publish the group row
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(f.counter, 1u);
  __syncthreads();
  if (s_ticket != (unsigned)n_groups - 1) return;
  __threadfence();
  FinArgs g = f;
  g.n_partials = n_groups;
  g.row_stride = FOLD_GROUP;
  if (g.peers != nullptr) finalize_peer_body(g, *g.peers, g.seq);
  else finalize_body(g, 1, 1);
  if (threadIdx.x == 0) *f.counter = 0u;             // ready for the next sweep
}

// ------------------------------------------------------------------------------------------------
// flat sweeps over edge_attr for the two encoder BatchNorms
// ------------------------------------------------------------------------------------------------
// STAGE 0: sums of (a, b, aa, ab, bb);  STAGE 1: sums of u[4], u^2[4] with u = W2·relu(BN1(W1·ea+b1)) + b2
template <int STAGE>
__global__ void __launch_bounds__(SWEEP_THREADS) enc_moments_kernel(const float2* __restrict__ edge_attr, long long E,
                                                                    const float* __restrict__ consts,
                                                                    const float* __restrict__ small,
                                                                    double* __restrict__ partials, const FinArgs fin,
                                                                    const int* __restrict__ run_flag) {
  pdl_wait();
  if (run_flag != nullptr && *run_flag == 0) return;       // the fused edge-feature kernel has taken these sums already
  __shared__ EdgeConsts sc;
  __shared__ double red[(SWEEP_THREADS / 32) * 8];
  __shared__ float w2raw[20];
  load_consts(sc, consts);
  if (STAGE == 1) {
    if (threadIdx.x < 16) w2raw[threadIdx.x] = small[MPN_W_ENC2_W + threadIdx.x];
    else if (threadIdx.x < 20) w2raw[threadIdx.x] = small[MPN_W_ENC2_B + threadIdx.x - 16];
    __syncthreads();
  }
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  constexpr int U = 4;                                  // independent loads in flight per thread
  // Sums run in fp32 over RUN x U edges of this thread, then join the fp64 accumulators: the fp32 -> fp64 conversions and the
  // double-precision adds per edge were what bounded this sweep (8 of each per edge), not the 8 B/edge it reads.  A run of 32
  // terms of similar size loses ~1e-7 relative with random sign; over E / 32 runs the totals keep ~1e-9.
  constexpr int RUN = 8;
  float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  int in_run = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; e0 < E; e0 += stride * U) {
    float2 eav[U];
    bool ok[U];
#pragma unroll
    for (int j = 0; j < U; ++j) {
      const long long e = e0 + stride * j;
      ok[j] = e < E;
      eav[j] = ldg_stream2(edge_attr + (ok[j] ? e : E - 1));
    }
#pragma unroll
    for (int j = 0; j < U; ++j) {
      if (!ok[j]) continue;
      const float2 ea = eav[j];
      if (STAGE == 0) {
        f[0] += ea.x; f[1] += ea.y; f[2] = fmaf(ea.x, ea.x, f[2]); f[3] = fmaf(ea.x, ea.y, f[3]); f[4] = fmaf(ea.y, ea.y, f[4]);
      } else {
        float a1[4], u[4];
        enc_layer1(sc, ea, a1);
        enc_layer2_pre(w2raw, w2raw + 16, a1, u);
#pragma unroll
        for (int k = 0; k < 4; ++k) { f[k] += u[k]; f[4 + k] = fmaf(u[k], u[k], f[4 + k]); }
      }
    }
    if (++in_run == RUN) {
#pragma unroll
      for (int k = 0; k < 8; ++k) { acc[k] += (double)f[k]; f[k] = 0.f; }
      in_run = 0;
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] += (double)f[k];
  block_sum_doubles<8, SWEEP_THREADS>(acc, red, partials + (size_t)blockIdx.x * SUMS);
  finalize_in_last_block(fin);
}

// ------------------------------------------------------------------------------------------------
// Edge sweeps.  One warp per task (<= chunk consecutive edges of one row), lane = edge.  Every lane handles U edges per
// iteration and issues all of their loads (col, edge_attr | y) before the dependent Pd[col] gathers and the math: the
// sweeps are latency-bound on the col -> Pd[col] chain otherwise (ncu: long_scoreboard 14-17 warps per issue).
// Out-of-range lanes read a clamped (valid) edge and are masked out of every sum / store.
// ------------------------------------------------------------------------------------------------
template <int U>
struct EdgeLoad {
  int e[U];
  bool ok[U];
  float2 ea[U];
  float4 pd[U];
  float4 y[U];
};

// YSRC 0: (edge_attr, col, Pd) -> y recomputed;  YSRC 1: y read from ybuf.  NEED_PD: SA with SRC 1 needs Pd AND ybuf.
template <int U, bool LOAD_EA, bool LOAD_PD, bool LOAD_Y>
__device__ __forceinline__ void load_edges(EdgeLoad<U>& L, const mpn_graph& g, int base, int end, int lane,
                                           const float2* __restrict__ edge_attr, const float4* __restrict__ Pd,
                                           const float4* __restrict__ ybuf) {
  int c[U];
#pragma unroll
  for (int j = 0; j < U; ++j) {
    const int e = base + 32 * j + lane;
    L.ok[j] = e < end;
    L.e[j] = L.ok[j] ? e : end - 1;
    if (LOAD_PD) c[j] = ldg_stream_i32(g.col + L.e[j]);
    if (LOAD_EA) L.ea[j] = ldg_stream2(edge_attr + L.e[j]);
    if (LOAD_Y) L.y[j] = ybuf[L.e[j]];
  }
  if (LOAD_PD) {
#pragma unroll
    for (int j = 0; j < U; ++j) L.pd[j] = __ldg(Pd + c[j]);
  }
}

// SA: moments of the edge-update pre-activation y (and optionally materialise y)
//   SRC 0: e_in = encoder(edge_attr[e])            (step 1)
//   SRC 1: e_in = relu(BN3_prev(ybuf[e]))          (step >= 2; ybuf updated in place)
//   RE_E (reattach_initial_edges, steps >= 2): e_in = [e0 | e] with e0 = encoder(edge_attr[e]) recomputed: y += We0 . e0
// A warp walks its tasks from the last to the first: the sweep before it (ENC1 over edge_attr, or the apply sweep of the previous
// step) ends at the high edges, which are then still in L2; the node-moment sweep after it walks forwards for the same reason.
template <int SRC, bool WRITE_Y, bool BATCHED, bool RE_E = false>
__global__ void __launch_bounds__(SWEEP_THREADS, 2) edge_moments_kernel(const mpn_graph g, const float2* __restrict__ edge_attr,
                                                                     const float4* __restrict__ Ps, const float4* __restrict__ Pd,
                                                                     float4* __restrict__ ybuf, const float* __restrict__ consts,
                                                                     double* __restrict__ partials, const FinArgs fin) {
  pdl_wait();
  constexpr int U = 4;
  __shared__ EdgeConsts scs[BATCHED ? SWEEP_THREADS / 32 : 1];
  __shared__ double red[(SWEEP_THREADS / 32) * 8];
  const int lane = threadIdx.x & 31;
  EdgeConsts& sc = scs[BATCHED ? (threadIdx.x >> 5) : 0];
  if (!BATCHED) load_consts(sc, consts);
  const int gwarp = (blockIdx.x * SWEEP_THREADS + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * SWEEP_THREADS) >> 5;
  const int n_tasks = *g.n_tasks;
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int cur_gid = -1;
  const int t_last = gwarp + max(n_tasks - 1 - gwarp, 0) / nwarps * nwarps;
  TaskPrefetch tp;
  tp.start(g, t_last, -nwarps, n_tasks);
  for (int t = t_last; task_in(t, n_tasks); t -= nwarps) {
    const int row_nn = tp.issue(g, t, -nwarps, n_tasks);
    const TaskRange tr = tp.cur;
    if (BATCHED) {
      const int gid = g.node_gid[tr.row];
      if (gid != cur_gid) { warp_load_consts(sc, consts + (size_t)gid * FC_TOTAL, lane); cur_gid = gid; }
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = 0.0;
    }
    const float4 ps = Ps[tr.row];
    float ft[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int base = tr.beg; base < tr.end; base += 32 * U) {
      EdgeLoad<U> L;
      load_edges<U, SRC == 0 || RE_E, true, SRC == 1>(L, g, base, tr.end, lane, edge_attr, Pd, ybuf);
#pragma unroll
      for (int j = 0; j < U; ++j) {
        float ein[4], y[4];
        if (SRC == 0) {
          enc_full(sc, L.ea[j], ein);
        } else {
          const float ypv[4] = {L.y[j].x, L.y[j].y, L.y[j].z, L.y[j].w};
          bn3_relu(sc, ypv, ein);
        }
        edge_pre(sc, ps, L.pd[j], ein, y);
        if (RE_E) {
          float e0[4];
          enc_full(sc, L.ea[j], e0);
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) y[a] = fmaf(sc.v[FC_EDGE_WE0 + 4 * a + b], e0[b], y[a]);
        }
        if (L.ok[j]) {
          if (WRITE_Y) ybuf[L.e[j]] = make_float4(y[0], y[1], y[2], y[3]);
#pragma unroll
          for (int k = 0; k < 4; ++k) { ft[k] += y[k]; ft[4 + k] = fmaf(y[k], y[k], ft[4 + k]); }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] += (double)ft[k];      // one task (<= chunk / 32 edges per lane) in fp32, the running sums in fp64
    if (BATCHED) {                                         // per-task partial, reduced per graph in fixed task order
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const double v = warp_sum(acc[k]);
        if (lane == 0) partials[(size_t)t * TASK_PART + k] = v;
      }
    }
    tp.rotate(row_nn);
  }
  if (!BATCHED) {
    block_sum_doubles<8, SWEEP_THREADS>(acc, red, partials + (size_t)blockIdx.x * SUMS);
    finalize_in_last_block(fin);
  }
}

// e' = relu(BN3(y)) for one loaded edge
template <int YSRC>
__device__ __forceinline__ void eprime_of(const EdgeConsts& sc, const float4 ps, const float2 ea, const float4 pd, const float4 yv,
                                          float (&ep)[4]) {
  float y[4];
  if (YSRC == 0) {
    float ein[4];
    enc_full(sc, ea, ein);
    edge_pre(sc, ps, pd, ein, y);
  } else {
    y[0] = yv.x; y[1] = yv.y; y[2] = yv.z; y[3] = yv.w;
  }
  bn3_relu(sc, y, ep);
}

// SB: per-task S1 = sum e' (for the closed-form node-BN moments), global T2 = sum e' e'^T.
// A warp walks its tasks from the first to the last: the edge update before it (SA) walks them backwards, so the y lines it wrote
// last, still in L2, are the first ones read here.
template <int YSRC, bool BATCHED>
__global__ void __launch_bounds__(SWEEP_THREADS, YSRC == 1 ? SWEEP_RESIDENT_BLOCKS : 2) node_moments_sweep_kernel(const mpn_graph g, const float2* __restrict__ edge_attr,
                                                                           const float4* __restrict__ Ps, const float4* __restrict__ Pd,
                                                                           const float4* __restrict__ ybuf, const float* __restrict__ consts,
                                                                           float4* __restrict__ s1_task, double* __restrict__ partials,
                                                                           const float* __restrict__ A, const float* __restrict__ small,
                                                                           const FinArgs fin) {
  pdl_wait();
  constexpr int U = (YSRC == 1 && !BATCHED) ? 8 : 4;     // stored y: 8 x 16 B in flight per lane (the sweep is bound by bytes in flight)
  __shared__ EdgeConsts scs[BATCHED ? SWEEP_THREADS / 32 : 1];
  __shared__ double red[(SWEEP_THREADS / 32) * 10];
  __shared__ double red_m[BATCHED ? 1 : SWEEP_THREADS / 32][64];
  const int lane = threadIdx.x & 31;
  EdgeConsts& sc = scs[BATCHED ? (threadIdx.x >> 5) : 0];
  if (!BATCHED) load_consts(sc, consts);
  const int gwarp = (blockIdx.x * SWEEP_THREADS + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * SWEEP_THREADS) >> 5;
  const int n_tasks = *g.n_tasks;
  double t2 = 0.0;                                         // lane i < 10: running sum of T2 entry i over this warp's tasks
  // per-node part of the closed-form node-BN moments, taken per task (it is linear in the task's edge count and S1):
  //   m1[c] += n_t A[row,c] + w_c.S1_t ;  m2[c] += n_t A[row,c]^2 + 2 A[row,c] (w_c.S1_t)      (w_c = W_node[c, 32:36]; lane = c)
  double m1 = 0.0, m2 = 0.0;
  int cur_gid = -1;
  TaskPrefetch tp;
  tp.start(g, gwarp, nwarps, n_tasks);
  for (int t = gwarp; t < n_tasks; t += nwarps) {
    const int row_nn = tp.issue(g, t, nwarps, n_tasks);
    const TaskRange tr = tp.cur;
    if (BATCHED) {
      const int gid = g.node_gid[tr.row];
      if (gid != cur_gid) { warp_load_consts(sc, consts + (size_t)gid * FC_TOTAL, lane); cur_gid = gid; }
    }
    const float a_row = BATCHED ? 0.f : A[(size_t)tr.row * MPN_DH + lane];
    const float4 ps = (YSRC == 0) ? Ps[tr.row] : make_float4(0.f, 0.f, 0.f, 0.f);
    float s1[4] = {0.f, 0.f, 0.f, 0.f};
    float q[10] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int base = tr.beg; base < tr.end; base += 32 * U) {
      EdgeLoad<U> L;
      load_edges<U, YSRC == 0, YSRC == 0, YSRC == 1>(L, g, base, tr.end, lane, edge_attr, Pd, ybuf);
#pragma unroll
      for (int j = 0; j < U; ++j) {
        float ep[4];
        eprime_of<YSRC>(sc, ps, L.ea[j], L.pd[j], L.y[j], ep);
        if (!L.ok[j]) { ep[0] = ep[1] = ep[2] = ep[3] = 0.f; }
        int idx = 0;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          s1[a] += ep[a];
#pragma unroll
          for (int b = a; b < 4; ++b) { q[idx] = fmaf(ep[a], ep[b], q[idx]); ++idx; }
        }
      }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) s1[a] = warp_sum(s1[a]);
    if (lane == 0) s1_task[t] = make_float4(s1[0], s1[1], s1[2], s1[3]);
    if (!BATCHED) {                                        // one task's term in fp32 (<= chunk edges), the running sums in fp64
      const float nt = (float)(tr.end - tr.beg);
      const float4 wn = *reinterpret_cast<const float4*>(small + MPN_W_NODE_W + lane * 36 + 32);      // L1-resident, once per task
      const float qd = fmaf(wn.x, s1[0], fmaf(wn.y, s1[1], fmaf(wn.z, s1[2], wn.w * s1[3])));
      m1 += (double)fmaf(nt, a_row, qd);
      m2 += (double)(a_row * fmaf(nt, a_row, 2.0f * qd));
    }
#pragma unroll
    for (int i = 0; i < 10; ++i) {                          // <= chunk/32 fp32 terms per lane, folded across the warp in fp64
      const double v = warp_sum((double)q[i]);
      if (BATCHED) { if (lane == 0) partials[(size_t)t * TASK_PART + i] = v; }
      else if (lane == i) t2 += v;
    }
    tp.rotate(row_nn);
  }
  if (!BATCHED) {
    const int warp = threadIdx.x >> 5;
    red_m[warp][lane] = m1;
    red_m[warp][32 + lane] = m2;
    block_sum_lane_columns<10, SWEEP_THREADS>(t2, red, partials + (size_t)blockIdx.x * SUMS + 64);   // (has the barriers)
    if (threadIdx.x < 64) {
      double sm = 0.0;
      for (int wv = 0; wv < SWEEP_THREADS / 32; ++wv) sm += red_m[wv][threadIdx.x];
      partials[(size_t)blockIdx.x * SUMS + threadIdx.x] = sm;
    }
    finalize_in_last_block(fin);
  }
}

// ------------------------------------------------------------------------------------------------
// SC: apply.  messages m = relu(BN4(A[row] + Wn·e')), per-task segment sums, logits, decisions.
// Lane = edge, two edges per lane per iteration (the folded weights are read once from shared memory for both), the
// loads of the NEXT iteration are issued before the math of the current one.  The 32-channel message is computed on
// packed channel pairs with fma.rn.f32x2 / add.f32x2 (sm_100 packed fp32).  32 fp32 accumulators per lane; a 31-shuffle
// transpose-reduce per task leaves channel c's sum in lane c (deterministic: fixed shuffle tree, fixed task order in
// node_finalize).
// ------------------------------------------------------------------------------------------------
template <bool MAXOP = false>
__device__ __forceinline__ float transpose_reduce32(float (&acc)[32], int lane) {
  // after the step with offset o the live values per lane halve; the lane keeps the half selected by bit o of its id
#pragma unroll
  for (int o = 16, n = 16; o > 0; o >>= 1, n >>= 1) {
    const bool upper = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (i < n) {
        const float send = upper ? acc[i] : acc[i + n];
        const float keep = upper ? acc[i + n] : acc[i];
        const float other = __shfl_xor_sync(0xffffffffu, send, o);
        acc[i] = MAXOP ? fmaxf(keep, other) : keep + other;
      }
    }
  }
  return acc[0];
}

typedef unsigned long long f32x2;        // two packed fp32 in one 64-bit register
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 relu2(f32x2 v) {
  float lo, hi;
  unpack2(v, lo, hi);
  return pack2(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
}

// ENC1 moments on packed fp32: the sweep over edge_attr for the second encoder BatchNorm is issue bound (ncu: 2.1 warp
// instructions per edge, issue slots 64 % busy, DRAM 28 %), so a thread takes TWO edges per 16-byte load and runs both through the
// 2 -> 4 -> 4 edge encoder with fma.rn.f32x2 (one instruction per channel for both edges); the folded weights sit in registers as
// broadcast pairs.  Sums in fp32 runs (RUN x U x 2 edges), then fp64, as enc_moments_kernel<1>.
__global__ void __launch_bounds__(SWEEP_THREADS, 2) enc_moments1_packed_kernel(const float4* __restrict__ edge_attr2, long long n_pairs,
                                                                             const float2* __restrict__ edge_attr, long long E,
                                                                             const float* __restrict__ consts, const float* __restrict__ small,
                                                                             double* __restrict__ partials, const FinArgs fin) {
  pdl_wait();
  __shared__ EdgeConsts sc;
  __shared__ double red[(SWEEP_THREADS / 32) * 8];
  load_consts(sc, consts);
  f32x2 w1x[4], w1y[4], c1[4], w2[16], c2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    w1x[j] = pack2(sc.v[FC_ENC1_W + 2 * j], sc.v[FC_ENC1_W + 2 * j]);
    w1y[j] = pack2(sc.v[FC_ENC1_W + 2 * j + 1], sc.v[FC_ENC1_W + 2 * j + 1]);
    c1[j] = pack2(sc.v[FC_ENC1_C + j], sc.v[FC_ENC1_C + j]);
    const float b = small[MPN_W_ENC2_B + j];
    c2[j] = pack2(b, b);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float w = small[MPN_W_ENC2_W + 4 * j + k]; w2[4 * j + k] = pack2(w, w); }
  }
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  f32x2 f[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) f[k] = 0ull;
  constexpr int U = 4, RUN = 4;
  int in_run = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n_pairs; i0 += stride * U) {
    float4 v[U];
    bool ok[U];
#pragma unroll
    for (int j = 0; j < U; ++j) {
      const long long i = i0 + stride * j;
      ok[j] = i < n_pairs;
      v[j] = ldg_stream4(edge_attr2 + (ok[j] ? i : n_pairs - 1));
    }
#pragma unroll
    for (int j = 0; j < U; ++j) {
      if (!ok[j]) continue;
      const f32x2 x2 = pack2(v[j].x, v[j].z), y2 = pack2(v[j].y, v[j].w);
      f32x2 a1[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) a1[c] = relu2(fma2(w1x[c], x2, fma2(w1y[c], y2, c1[c])));
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        f32x2 u = c2[c];
#pragma unroll
        for (int k = 0; k < 4; ++k) u = fma2(w2[4 * c + k], a1[k], u);
        f[c] = add2(f[c], u);
        f[4 + c] = fma2(u, u, f[4 + c]);
      }
    }
    if (++in_run == RUN) {
#pragma unroll
      for (int k = 0; k < 8; ++k) { float lo, hi; unpack2(f[k], lo, hi); acc[k] += (double)lo + (double)hi; f[k] = 0ull; }
      in_run = 0;
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) { float lo, hi; unpack2(f[k], lo, hi); acc[k] += (double)lo + (double)hi; }
  if ((E & 1) && blockIdx.x == 0 && threadIdx.x == 0) {          // odd edge count: the last edge on its own
    float a1[4], u[4];
    enc_layer1(sc, edge_attr[E - 1], a1);
    float w2raw[20];
#pragma unroll
    for (int k = 0; k < 16; ++k) w2raw[k] = small[MPN_W_ENC2_W + k];
#pragma unroll
    for (int k = 0; k < 4; ++k) w2raw[16 + k] = small[MPN_W_ENC2_B + k];
    enc_layer2_pre(w2raw, w2raw + 16, a1, u);
#pragma unroll
    for (int k = 0; k < 4; ++k) { acc[k] += (double)u[k]; acc[4 + k] += (double)u[k] * (double)u[k]; }
  }
  block_sum_doubles<8, SWEEP_THREADS>(acc, red, partials + (size_t)blockIdx.x * SUMS);
  finalize_in_last_block(fin);
}

// softmax([l0,l1])[1] (inference.py:475-477) with ATen's own arithmetic (softmax_warp_forward: exp(x - max) / sum, IEEE
// division, full-precision expf), so that the value is bit-identical to torch.softmax(logits, dim=1)[:, 1] on the device:
// PRUNING takes an argmin over it and SPLITTING compares it with float == (utils.py:96-98, 288-289).  exp(0) = 1 exactly, so
// one expf suffices:  l1 >= l0: 1 / (e + 1);  l1 < l0: e / (1 + e),  e = expf(-|l0 - l1|).
__device__ __forceinline__ float softmax1(float l0, float l1) {
  const float e = expf(-fabsf(l0 - l1));
  const float sum = e + 1.0f;
  return __fdiv_rn((l1 >= l0) ? 1.0f : e, sum);
}

template <bool CLASSIFY>
__device__ __forceinline__ void classify_store(const EdgeConsts& sc, const float (&ep)[4], int e, float2* __restrict__ logits,
                                               uint8_t* __restrict__ pred, float* __restrict__ prob1) {
  if (!CLASSIFY) return;
  float l0 = sc.v[FC_CLS_B + 0], l1 = sc.v[FC_CLS_B + 1];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    l0 = fmaf(sc.v[FC_CLS_W + k], ep[k], l0);
    l1 = fmaf(sc.v[FC_CLS_W + 4 + k], ep[k], l1);
  }
  logits[e] = make_float2(l0, l1);
  if (pred) pred[e] = (l1 > l0) ? 1 : 0;                  // argmax, tie -> class 0 (inference.py:479)
  if (prob1) prob1[e] = softmax1(l0, l1);
}

template <int YSRC, bool CLASSIFY, bool BATCHED, bool AGGMAX>
__global__ void __launch_bounds__(SWEEP_THREADS, 2) apply_kernel(const mpn_graph g, const float2* __restrict__ edge_attr,
                                                              const float4* __restrict__ Ps, const float4* __restrict__ Pd,
                                                              const float4* __restrict__ ybuf, const float* __restrict__ A,
                                                              const float* __restrict__ consts, float* __restrict__ msg_task,
                                                              float2* __restrict__ logits, uint8_t* __restrict__ pred,
                                                              float* __restrict__ prob1) {
  pdl_wait();
  constexpr int U = 2;
  constexpr int NW = BATCHED ? SWEEP_THREADS / 32 : 1;
  __shared__ EdgeConsts scs[NW];
  __shared__ __align__(16) f32x2 w2s_all[NW][16][4];          // folded node weights as channel pairs: (w[2p][k], w[2p+1][k])
  const int lane = threadIdx.x & 31;
  EdgeConsts& sc = scs[BATCHED ? (threadIdx.x >> 5) : 0];
  f32x2 (*w2s)[4] = w2s_all[BATCHED ? (threadIdx.x >> 5) : 0];
  if (!BATCHED) {
    load_consts(sc, consts);
    if (threadIdx.x < 64) {
      const int p = threadIdx.x >> 2, k = threadIdx.x & 3;
      w2s[p][k] = pack2(sc.v[FC_NODE_WE + 4 * (2 * p) + k], sc.v[FC_NODE_WE + 4 * (2 * p + 1) + k]);
    }
    __syncthreads();
  }
  const uint32_t w2_addr = (uint32_t)__cvta_generic_to_shared(&w2s[0][0]);
  const int gwarp = (blockIdx.x * SWEEP_THREADS + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * SWEEP_THREADS) >> 5;
  const int n_tasks = *g.n_tasks;
  int cur_gid = -1;
  for (int t = gwarp; t < n_tasks; t += nwarps) {
    const TaskRange tr = task_range(g, t);
    if (BATCHED) {
      const int gid = g.node_gid[tr.row];
      if (gid != cur_gid) {
        warp_load_consts(sc, consts + (size_t)gid * FC_TOTAL, lane);
#pragma unroll
        for (int i = lane; i < 64; i += 32) {
          const int p = i >> 2, k = i & 3;
          w2s[p][k] = pack2(sc.v[FC_NODE_WE + 4 * (2 * p) + k], sc.v[FC_NODE_WE + 4 * (2 * p + 1) + k]);
        }
        __syncwarp();
        cur_gid = gid;
      }
    }
    const float4 ps = (YSRC == 0) ? Ps[tr.row] : make_float4(0.f, 0.f, 0.f, 0.f);
    // folded A'[c] = s4[c]*A[row,c] + t4[c]; lane c computes it, every lane needs all 32 (as 16 packed pairs)
    const float a_mine = fmaf(sc.v[FC_BN4_S + lane], A[(size_t)tr.row * MPN_DH + lane], sc.v[FC_BN4_T + lane]);
    f32x2 ap[16], acc[16];
#pragma unroll
    for (int p = 0; p < 16; ++p) {
      ap[p] = pack2(__shfl_sync(0xffffffffu, a_mine, 2 * p), __shfl_sync(0xffffffffu, a_mine, 2 * p + 1));
      acc[p] = 0ull;
    }
    EdgeLoad<U> cur, nxt;
    load_edges<U, YSRC == 0, YSRC == 0, YSRC == 1>(cur, g, tr.beg, tr.end, lane, edge_attr, Pd, ybuf);
    for (int base = tr.beg; base < tr.end; base += 32 * U) {
      const int nbase = base + 32 * U;
      if (nbase < tr.end) load_edges<U, YSRC == 0, YSRC == 0, YSRC == 1>(nxt, g, nbase, tr.end, lane, edge_attr, Pd, ybuf);
      float ep[U][4];
      f32x2 ed[U][4];
#pragma unroll
      for (int j = 0; j < U; ++j) {
        eprime_of<YSRC>(sc, ps, cur.ea[j], cur.pd[j], cur.y[j], ep[j]);
#pragma unroll
        for (int k = 0; k < 4; ++k) ed[j][k] = pack2(ep[j][k], ep[j][k]);
      }
#pragma unroll
      for (int p = 0; p < 16; ++p) {
        // volatile: keep the 32 weight loads inside the loop (hoisting them costs 128 registers and spills)
        ulonglong2 wa, wb;
        asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(wa.x), "=l"(wa.y) : "r"(w2_addr + p * 32));
        asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(wb.x), "=l"(wb.y) : "r"(w2_addr + p * 32 + 16));
#pragma unroll
        for (int j = 0; j < U; ++j) {
          f32x2 z = fma2(wa.x, ed[j][0], ap[p]);
          z = fma2(wa.y, ed[j][1], z);
          z = fma2(wb.x, ed[j][2], z);
          z = fma2(wb.y, ed[j][3], z);
          z = relu2(z);
          if (cur.ok[j]) {
            if (AGGMAX) {                                  // scatter_max (models/mpn.py:199): messages are >= 0, so 0 is neutral
              float zl, zh, al, ah;
              unpack2(z, zl, zh);
              unpack2(acc[p], al, ah);
              acc[p] = pack2(fmaxf(al, zl), fmaxf(ah, zh));
            } else {
              acc[p] = add2(acc[p], z);
            }
          }
        }
      }
#pragma unroll
      for (int j = 0; j < U; ++j)
        if (cur.ok[j]) classify_store<CLASSIFY>(sc, ep[j], cur.e[j], logits, pred, prob1);
#pragma unroll
      for (int j = 0; j < U; ++j) {                       // rotate only the fields this variant loads
        cur.e[j] = nxt.e[j];
        cur.ok[j] = nxt.ok[j];
        if (YSRC == 0) { cur.ea[j] = nxt.ea[j]; cur.pd[j] = nxt.pd[j]; }
        else cur.y[j] = nxt.y[j];
      }
    }
    float accf[32];
#pragma unroll
    for (int p = 0; p < 16; ++p) unpack2(acc[p], accf[2 * p], accf[2 * p + 1]);
    const float total = transpose_reduce32<AGGMAX>(accf, lane);
    msg_task[(size_t)t * MPN_DH + lane] = total;
  }
}

// ------------------------------------------------------------------------------------------------
// SC on the 5th-generation tensor cores (stored-y mode).  The packed-fp32 kernel above is issue bound: ~10 warp
// instructions per edge, most of them the 32 x 4 message FMAs and the ReLU+add.  Here, for a batch of 128 edges of one row,
//   Z[128 edges x 32 channels] = E1 (128 x 8) W1^T  +  E2 (128 x 8) W2^T
//       E1[e] = [ e'_hi (4) | e'_lo (4) ]        W1[c] = [ W'_hi[c] (4) | W'_hi[c] (4) ]
//       E2[e] = [ e'_hi (4) | 1 1 0 0   ]        W2[c] = [ W'_lo[c] (4) | A'_hi[c] A'_lo[c] 0 0 ]
// is two tcgen05.mma (M=128, N=32, K=8, kind::tf32; hi.hi + lo.hi + hi.lo = 3xTF32, the row's folded A' enters through two
// exact "1" columns) into 32 TMEM columns.  Thread i owns TMEM lane i = its own edge and adds |z| of the 32 channels
// into 32 registers (one FADD each, the absolute value is an operand modifier):
//     sum relu(z) = ( sum |z| + sum z ) / 2,      sum z = deg A' + W' . S1      (S1 = sum e' is already known from sweep SB),
// so node_finalize adds the closed-form half.  A masked edge has an all-zero operand row -> z = 0.
// The 31-shuffle transpose-reduce runs once per RUN of consecutive tasks of one row (the block walks a contiguous task range);
// the run's sum goes to its last task, zeros to the others (node_finalize adds a row's tasks in order: same result).
// Pipeline: y streams through a per-thread cp.async ring D batches ahead; operand tiles are double buffered so the MMA of
// batch k runs while the CUDA cores prepare batch k+1; one __syncthreads per batch.  Deterministic (fixed edge -> lane
// map, fixed shuffle tree, fixed task order).
// ------------------------------------------------------------------------------------------------
constexpr int ATC_THREADS = 128;
constexpr int ATC_CTAS_PER_SM = 5;                       // 40.6 KB shared memory, 89 registers, 64 TMEM columns per block
constexpr int ATC_SEG = 128;                             // task ranges staged in shared memory per segment
constexpr int ATC_BATCHES = 512;                         // 128-edge batches per segment (the segment is shortened to fit)
constexpr int ATC_NB = 2;                                // 128-edge batches per iteration (one barrier / fence / commit for both)
constexpr int ATC_D = 4;                                 // y runs D batches ahead
constexpr int ATC_RL = ATC_D + 1;                        // ring slots
constexpr int ATC_SLOT_BYTES = 128 * 16;
// canonical K-major no-swizzle operand tile: [rows/8 groups][2 K-cores][8 rows][4 floats]
__device__ __forceinline__ int tile_off(int row, int kcore) { return (row >> 3) * 64 + kcore * 32 + (row & 7) * 4; }
// edge-operand tile of the apply sweep: THREE K-core blocks per 8-row group, [e'_lo | e'_hi | 1 1 0 0].  E1 = [e'_lo | e'_hi]
// starts at block 0, E2 = [e'_hi | 1 1 0 0] at block 1 (same LBO = 128 B, SBO = 384 B): e'_hi is stored once and read by both
// MMAs (2 instead of 3 shared-memory stores per edge, 6 instead of 8 KB per 128-edge batch -> a 5th block per SM fits).
constexpr int ATC_GROUP_BYTES = 3 * 128;
constexpr int ATC_TILE_BYTES = 16 * ATC_GROUP_BYTES;
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
  // round-to-nearest (ties away) to 10 mantissa bits without cvt.rna.tf32 (which ptxas expands to 4 instructions with an
  // inf/nan guard): finite inputs only.  The tensor core reads the top 19 bits of lo: error ~2^-22 |v|.
  hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
  lo = v - hi;
}
// per-thread asynchronous copies global -> shared (LDGSTS): the landing ring is private to the thread that issued them, so
// cp.async.wait_group is the only synchronisation needed
template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// shared-memory accesses through explicit 32-bit addresses that the compiler must keep in registers (opaque): ptxas otherwise
// rebuilds every tile / ring address from threadIdx in each iteration of the batch loop (~15 instructions per batch)
__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) {
  asm volatile("" : "+r"(v));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

template <bool CLASSIFY, bool DECIDE, bool AGGMAX, int CTAS>
__global__ void __launch_bounds__(ATC_THREADS, CTAS) apply_tc_kernel(
    const mpn_graph g, const float4* __restrict__ ybuf, const float* __restrict__ A, const float* __restrict__ consts,
    float* __restrict__ msg_task, float2* __restrict__ logits, uint8_t* __restrict__ pred, float* __restrict__ prob1) {
  pdl_wait();
  __shared__ EdgeConsts sc;
  __shared__ __align__(128) float et[2 * ATC_NB][ATC_TILE_BYTES / 4];  // [buffer][half]: [e'_lo | e'_hi | 1 1 0 0] per 8-row group
  __shared__ __align__(128) float w1[32 * 8];
  __shared__ __align__(128) float w2[32 * 8];
  __shared__ __align__(16) float4 ring[ATC_RL][ATC_THREADS];
  __shared__ int s_row[ATC_SEG], s_beg[ATC_SEG], s_end[ATC_SEG];
  __shared__ int s_bstart[ATC_BATCHES], s_nbatch;
  __shared__ float red[2][ATC_THREADS / 32][32];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_slot;
  load_consts(sc, consts);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (warp == 0) tmem_alloc(&tmem_slot, 32 * ATC_NB);
  if (tid == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 32) {                                        // static parts of the weight tiles (channel = tid)
    float wh[4], wl[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      split_tf32(sc.v[FC_NODE_WE + 4 * tid + k], wh[k], wl[k]);
      uint32_t lb;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(wl[k]));
      wl[k] = __uint_as_float(lb);
    }
    *reinterpret_cast<float4*>(&w1[tile_off(tid, 0)]) = make_float4(wh[0], wh[1], wh[2], wh[3]);
    *reinterpret_cast<float4*>(&w1[tile_off(tid, 1)]) = make_float4(wh[0], wh[1], wh[2], wh[3]);
    *reinterpret_cast<float4*>(&w2[tile_off(tid, 0)]) = make_float4(wl[0], wl[1], wl[2], wl[3]);
    *reinterpret_cast<float4*>(&w2[tile_off(tid, 1)]) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  constexpr uint32_t IDESC = make_idesc_tf32(128, 32);
  const uint64_t d_w1 = make_smem_desc_noswizzle(smem_u32(w1), 128, 256), d_w2 = make_smem_desc_noswizzle(smem_u32(w2), 128, 256);
  const uint64_t d_e1 = make_smem_desc_noswizzle(smem_u32(et[0]), 128, ATC_GROUP_BYTES);            // [e'_lo | e'_hi]
  const uint64_t d_e2 = make_smem_desc_noswizzle(smem_u32(et[0]) + 128, 128, ATC_GROUP_BYTES);      // [e'_hi | 1 1 0 0]
  constexpr uint64_t BUF_STEP = ATC_TILE_BYTES >> 4;                     // next operand buffer, in descriptor address units
  const uint32_t my_tmem = opaque_u32(tmem + ((uint32_t)(warp * 32) << 16));
  const uint32_t et_addr = opaque_u32(smem_u32(et[0]) + (uint32_t)((tid >> 3) * ATC_GROUP_BYTES + (tid & 7) * 16));   // this edge's row of block 0
  const uint32_t ring_addr = opaque_u32(smem_u32(&ring[0][tid]));
  constexpr uint32_t TILE_BYTES = ATC_TILE_BYTES;
#pragma unroll
  for (int i = 0; i < 2 * ATC_NB; ++i)                   // the two "1" columns never change
    sts128(et_addr + (uint32_t)i * TILE_BYTES + 256, 1.f, 1.f, 0.f, 0.f);
  uint32_t phase = 0;
  const int n_tasks = *g.n_tasks;
  const int per = (n_tasks + (int)gridDim.x - 1) / (int)gridDim.x;
  const int t_first = blockIdx.x * per, t_last = min(n_tasks, t_first + per);
  const float bn_s = sc.v[FC_BN4_S + lane], bn_t = sc.v[FC_BN4_T + lane];
  const float s3[4] = {sc.v[FC_BN3_S], sc.v[FC_BN3_S + 1], sc.v[FC_BN3_S + 2], sc.v[FC_BN3_S + 3]};
  const float t3[4] = {sc.v[FC_BN3_T], sc.v[FC_BN3_T + 1], sc.v[FC_BN3_T + 2], sc.v[FC_BN3_T + 3]};
  int flushes = 0;

  const int seg_tasks = min(ATC_SEG, ATC_BATCHES / max(1, g.chunk / ATC_THREADS));   // a task has at most chunk / 128 batches
  for (int s0 = t_first; s0 < t_last; s0 += seg_tasks) {
    const int ns = min(seg_tasks, t_last - s0);
    __syncthreads();                                     // the previous segment's ranges are no longer read
    for (int i = tid; i < ns; i += ATC_THREADS) {
      const TaskRange tr = task_range(g, s0 + i);
      s_row[i] = tr.row; s_beg[i] = tr.beg; s_end[i] = tr.end;
    }
    __syncthreads();
    // first edge of every 128-edge batch of the segment, in processing order (a task's batches restart at the task's first edge):
    // the stream iterator below is then one shared-memory load per batch instead of a walk over the task ranges
    for (int i = tid; i < ns; i += ATC_THREADS) {
      int first = 0;
      for (int k = 0; k < i; ++k) first += (s_end[k] - s_beg[k] + ATC_THREADS - 1) / ATC_THREADS;
      const int nb_i = (s_end[i] - s_beg[i] + ATC_THREADS - 1) / ATC_THREADS;
      for (int k = 0; k < nb_i; ++k) s_bstart[first + k] = s_beg[i] + k * ATC_THREADS;
      if (i == ns - 1) s_nbatch = first + nb_i;
    }
    __syncthreads();
    // stream iterator (block-uniform): the batch whose y is copied next.  A lane past the end of its task reads on into the next
    // task's edges (clamped to the segment's last edge): valid memory, and a masked lane's result is never added.
    const int n_batch = s_nbatch, seg_last = s_end[ns - 1] - 1;
    int st_j = 0, st_off = 0;
    auto issue_stream = [&]() {
      if (st_j < n_batch) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(ring_addr + (uint32_t)st_off), "l"(ybuf + min(s_bstart[st_j] + tid, seg_last)) : "memory");
        ++st_j;
        st_off = (st_off == (ATC_RL - 1) * ATC_SLOT_BYTES) ? 0 : st_off + ATC_SLOT_BYTES;
      }
      cp_async_commit();
    };
#pragma unroll
    for (int j = 0; j < ATC_D; ++j) issue_stream();
    float acc[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) acc[c] = 0.f;
    int pending = 0;                                     // batches of the MMA group in flight whose result has not been accumulated
    int run_first = 0;                                   // first task (segment index) of the current run of one row
    int c_off = 0, buf = 0, issuer = 0;
    bool ok_prev[ATC_NB];
#pragma unroll
    for (int h = 0; h < ATC_NB; ++h) ok_prev[h] = false;
    float a_next = __ldg(A + (size_t)s_row[0] * MPN_DH + lane);
    auto drain = [&]() {                                 // accumulate the finished batches (only lanes whose edge was real)
      mbar_wait(&bar, phase);
      phase ^= 1;
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < ATC_NB; ++h) {
        if (h < pending) {
          float v[32];
          tmem_ld32(my_tmem + 32 * h, v);
          if (ok_prev[h]) {
#pragma unroll
            for (int c = 0; c < 32; ++c) acc[c] = AGGMAX ? fmaxf(acc[c], v[c]) : acc[c] + fabsf(v[c]);   // max relu(z) = max(0, max z)
          }
        }
      }
      tc_fence_before();
    };
    auto flush_to_red = [&]() {                          // this run's sum |z| per channel: lane c of every warp
      const float total = transpose_reduce32<AGGMAX>(acc, lane);
      red[flushes & 1][warp][lane] = total;
#pragma unroll
      for (int c = 0; c < 32; ++c) acc[c] = 0.f;
    };
    auto store_run = [&](int first, int last_t) {        // after the barrier that follows flush_to_red; warp 0 only
      const float (*r)[32] = red[flushes & 1];
      msg_task[(size_t)(s0 + last_t) * MPN_DH + lane] = AGGMAX ? fmaxf(fmaxf(r[0][lane], r[1][lane]), fmaxf(r[2][lane], r[3][lane]))
                                                               : (r[0][lane] + r[1][lane]) + (r[2][lane] + r[3][lane]);
      for (int t = first; t < last_t; ++t) msg_task[(size_t)(s0 + t) * MPN_DH + lane] = 0.f;
    };
    for (int ti = 0; ti < ns; ++ti) {
      const int row = s_row[ti], t_beg = s_beg[ti], t_end = s_end[ti];
      const bool new_run = ti == 0 || row != s_row[ti - 1];
      const float a_cur = a_next;
      if (ti + 1 < ns) a_next = __ldg(A + (size_t)s_row[ti + 1] * MPN_DH + lane);
      for (int pos = t_beg; pos < t_end; pos += ATC_NB * ATC_THREADS) {
        const int nb = (pos + ATC_THREADS < t_end) ? ATC_NB : 1;      // batches of this iteration (block-uniform)
        bool ok[ATC_NB];
        float ep[ATC_NB][4];
#pragma unroll
        for (int h = 0; h < ATC_NB; ++h) {
          ok[h] = false;
          if (h < nb) {
            cp_async_wait<ATC_D - 1>();                  // this batch's y has landed
            const float4 yv = lds128(ring_addr + (uint32_t)c_off);
            c_off = (c_off == (ATC_RL - 1) * ATC_SLOT_BYTES) ? 0 : c_off + ATC_SLOT_BYTES;
            issue_stream();
            const int e = pos + h * ATC_THREADS + tid;
            ok[h] = e < t_end;                           // a masked lane computes on a clamped edge; its TMEM row is never added
            ep[h][0] = fmaxf(fmaf(s3[0], yv.x, t3[0]), 0.f);
            ep[h][1] = fmaxf(fmaf(s3[1], yv.y, t3[1]), 0.f);
            ep[h][2] = fmaxf(fmaf(s3[2], yv.z, t3[2]), 0.f);
            ep[h][3] = fmaxf(fmaf(s3[3], yv.w, t3[3]), 0.f);
            if (CLASSIFY && ok[h]) {
              float l0 = sc.v[FC_CLS_B + 0], l1 = sc.v[FC_CLS_B + 1];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                l0 = fmaf(sc.v[FC_CLS_W + k], ep[h][k], l0);
                l1 = fmaf(sc.v[FC_CLS_W + 4 + k], ep[h][k], l1);
              }
              logits[e] = make_float2(l0, l1);
              if (DECIDE) {
                pred[e] = (l1 > l0) ? 1 : 0;                                      // argmax, tie -> class 0 (inference.py:479)
                prob1[e] = softmax1(l0, l1);                                      // softmax(.)[1] (inference.py:475-477), ATen-exact
              }
            }
            float eh[4], el[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) split_tf32(ep[h][k], eh[k], el[k]);
            const uint32_t boff = (uint32_t)(buf * ATC_NB + h) * TILE_BYTES;
            sts128(et_addr + boff, el[0], el[1], el[2], el[3]);
            sts128(et_addr + boff + 128, eh[0], eh[1], eh[2], eh[3]);
          }
        }
        if (pending) drain();                            // the previous iteration's MMAs finished while this one was being prepared
#pragma unroll
        for (int h = 0; h < ATC_NB; ++h) ok_prev[h] = ok[h];
        const bool first_batch = pos == t_beg;
        const bool flushed = first_batch && new_run && ti > 0;
        if (first_batch && new_run) {
          if (ti > 0) flush_to_red();
          if (tid < 32) {                                // the new row's folded A' (the previous MMA has completed)
            float ah, al, al_hi, al_lo;
            split_tf32(fmaf(bn_s, a_cur, bn_t), ah, al);
            split_tf32(al, al_hi, al_lo);
            *reinterpret_cast<float4*>(&w2[tile_off(tid, 1)]) = make_float4(ah, al_hi, 0.f, 0.f);
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == issuer) {                             // the issuing duty (~75 instructions) rotates over the four warps: no warp is
          tc_fence_after();                              // the one the block barrier always waits for
#pragma unroll
          for (int h = 0; h < ATC_NB; ++h) {
            if (h < nb) {
              umma_tf32(tmem + 32 * h, d_e1 + (uint64_t)(buf * ATC_NB + h) * BUF_STEP, d_w1, IDESC, 0);
              umma_tf32(tmem + 32 * h, d_e2 + (uint64_t)(buf * ATC_NB + h) * BUF_STEP, d_w2, IDESC, 1);
            }
          }
          umma_commit(&bar);
        }
        issuer = (issuer + 32) & (ATC_THREADS - 1);
        pending = nb;
        buf ^= 1;
        if (flushed) {
          if (warp == 0) store_run(run_first, ti - 1);
          ++flushes;
          run_first = ti;
        }
      }
    }
    if (pending) drain();
    flush_to_red();
    __syncthreads();
    if (warp == 0) store_run(run_first, ns - 1);
    ++flushes;
    cp_async_wait<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 32 * ATC_NB);
  }
}

// ------------------------------------------------------------------------------------------------
// Batched small graphs (BASELINE configs[2]): one launch over all graphs, BatchNorm statistics per graph.
// Moment sweeps write one partial per task; a block per graph adds its tasks in task order (deterministic) and folds
// that graph's constants.  Graphs are contiguous in node, task and edge order.
// ------------------------------------------------------------------------------------------------
template <int STAGE>
__global__ void __launch_bounds__(SWEEP_THREADS) enc_moments_task_kernel(const mpn_graph g, const float2* __restrict__ edge_attr,
                                                                         const float* __restrict__ consts, const float* __restrict__ small,
                                                                         double* __restrict__ task_part) {
  pdl_wait();
  __shared__ EdgeConsts scs[SWEEP_THREADS / 32];
  __shared__ float w2raw[20];
  if (threadIdx.x < 16) w2raw[threadIdx.x] = small[MPN_W_ENC2_W + threadIdx.x];
  else if (threadIdx.x < 20) w2raw[threadIdx.x] = small[MPN_W_ENC2_B + threadIdx.x - 16];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  EdgeConsts& sc = scs[threadIdx.x >> 5];
  const int gwarp = (blockIdx.x * SWEEP_THREADS + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * SWEEP_THREADS) >> 5;
  const int n_tasks = *g.n_tasks;
  int cur_gid = -1;
  for (int t = gwarp; t < n_tasks; t += nwarps) {
    const TaskRange tr = task_range(g, t);
    if (STAGE == 1) {
      const int gid = g.node_gid[tr.row];
      if (gid != cur_gid) { warp_load_consts(sc, consts + (size_t)gid * FC_TOTAL, lane); cur_gid = gid; }
    }
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int e = tr.beg + lane; e < tr.end; e += 32) {
      const float2 ea = ldg_stream2(edge_attr + e);
      if (STAGE == 0) {
        const double a = ea.x, b = ea.y;
        acc[0] += a; acc[1] += b; acc[2] += a * a; acc[3] += a * b; acc[4] += b * b;
      } else {
        float a1[4], u[4];
        enc_layer1(sc, ea, a1);
        enc_layer2_pre(w2raw, w2raw + 16, a1, u);
#pragma unroll
        for (int k = 0; k < 4; ++k) { const double d = u[k]; acc[k] += d; acc[4 + k] += d * d; }
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const double v = warp_sum(acc[k]);
      if (lane == 0) task_part[(size_t)t * TASK_PART + k] = v;
    }
  }
}

// one block (128 threads) per graph: task partials -> sums[g] -> consts[g]
__global__ void __launch_bounds__(128) graph_finalize_kernel(int stage, const mpn_graph g, const double* __restrict__ task_part,
                                                             const float* __restrict__ A, const float4* __restrict__ s1_task,
                                                             const float* __restrict__ small, double* __restrict__ sums_all,
                                                             float* __restrict__ consts_all, int re_e) {
  pdl_wait();
  __shared__ double red[4][64];
  const int gi = blockIdx.x;
  const int n0 = g.graph_nptr[gi], n1 = g.graph_nptr[gi + 1];
  const int t0 = g.taskptr[n0], t1 = g.taskptr[n1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* sums = sums_all + (size_t)gi * SUMS;
  const int ncols = (stage == MPN_STAGE_NODE) ? 10 : 8;
  const int cbase = (stage == MPN_STAGE_NODE) ? 64 : 0;
  for (int col = warp; col < ncols; col += 4) {                 // warp per column, lanes stride the graph's tasks
    double v = 0.0;
    for (int t = t0 + lane; t < t1; t += 32) v += task_part[(size_t)t * TASK_PART + col];
    v = warp_sum(v);
    if (lane == 0) sums[cbase + col] = v;
  }
  if (stage == MPN_STAGE_NODE) {                                // closed-form per-node part (lane = channel)
    float w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = small[MPN_W_NODE_W + lane * 36 + 32 + k];
    double m1 = 0.0, m2 = 0.0;
    for (int n = n0 + warp; n < n1; n += 4) {
      const int deg = g.rowptr[n + 1] - g.rowptr[n];
      if (deg == 0) continue;
      double sv[4] = {0, 0, 0, 0};
      for (int t = g.taskptr[n]; t < g.taskptr[n + 1]; ++t) {
        const float4 v = s1_task[t];
        sv[0] += v.x; sv[1] += v.y; sv[2] += v.z; sv[3] += v.w;
      }
      const double a = A[(size_t)n * MPN_DH + lane];
      const double qd = w[0] * sv[0] + w[1] * sv[1] + w[2] * sv[2] + w[3] * sv[3];
      m1 += deg * a + qd;
      m2 += deg * a * a + 2.0 * a * qd;
    }
    red[warp][lane] = m1;
    red[warp][32 + lane] = m2;
    __syncthreads();
    if (threadIdx.x < 64) sums[threadIdx.x] = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
  }
  __syncthreads();
  FinArgs f;
  f.stage = stage;
  f.partials = nullptr; f.n_partials = 0; f.row_stride = 1; f.partials2 = nullptr; f.n_partials2 = 0;
  f.sums = sums;
  f.consts = consts_all + (size_t)gi * FC_TOTAL;
  f.small = small;
  f.n_total = (double)(g.rowptr[n1] - g.rowptr[n0]);
  f.counter = nullptr;
  f.n_total_dev = nullptr;
  f.local_edges = 0.0;
  f.fixed = nullptr;
  f.peers = nullptr;
  f.seq = 0;
  f.re_e = re_e;
  finalize_body(f, 0, 1);
}

// per-graph column statistics of the node-encoder activations: grid (32-column tiles, graphs) -> scale/shift [G][Nc]
__global__ void __launch_bounds__(256) colstats_graph_kernel(const float* __restrict__ Y, int Nc, const int* __restrict__ graph_nptr,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             float* __restrict__ scale, float* __restrict__ shift) {
  pdl_wait();
  __shared__ double ssum[8][33], ssq[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  const int gi = blockIdx.y;
  const int r0 = graph_nptr[gi], r1 = graph_nptr[gi + 1];
  double s = 0.0, q = 0.0;
  if (col < Nc)
    for (int r = r0 + ry; r < r1; r += 8) {
      const double v = Y[(size_t)r * Nc + col];
      s += v;
      q += v * v;
    }
  ssum[ry][cx] = s;
  ssq[ry][cx] = q;
  __syncthreads();
  if (ry == 0 && col < Nc) {
    for (int i = 1; i < 8; ++i) { s += ssum[i][cx]; q += ssq[i][cx]; }
    const int M = r1 - r0;
    const double mean = s / M;
    double var = q / M - mean * mean;
    if (var < 0.0) var = 0.0;
    const double sc = (double)gamma[col] / sqrt(var + (double)BN_EPS);
    scale[(size_t)gi * Nc + col] = (float)sc;
    shift[(size_t)gi * Nc + col] = (float)((double)beta[col] - sc * mean);
  }
}

// L == 0 special case (models/mpn.py:295-297): classify the encoder output directly
__global__ void __launch_bounds__(SWEEP_THREADS) classify_encoded_kernel(const float2* __restrict__ edge_attr, long long E,
                                                                         const float* __restrict__ consts,
                                                                         float2* __restrict__ logits, uint8_t* __restrict__ pred,
                                                                         float* __restrict__ prob1) {
  pdl_wait();
  __shared__ EdgeConsts sc;
  load_consts(sc, consts);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    float ep[4];
    enc_full(sc, ldg_stream2(edge_attr + e), ep);
    float l0 = sc.v[FC_CLS_B + 0], l1 = sc.v[FC_CLS_B + 1];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      l0 = fmaf(sc.v[FC_CLS_W + k], ep[k], l0);
      l1 = fmaf(sc.v[FC_CLS_W + 4 + k], ep[k], l1);
    }
    logits[e] = make_float2(l0, l1);
    if (pred) pred[e] = (l1 > l0) ? 1 : 0;
    if (prob1) prob1[e] = softmax1(l0, l1);
  }
}

// decisions as a bit mask: bit (e & 31) of word e >> 5 (= np.unpackbits(bytes, bitorder="little")); 1/8 of the D2H bytes
__global__ void __launch_bounds__(256) pack_decisions_kernel(const uint8_t* __restrict__ pred, long long E, uint32_t* __restrict__ words) {
  pdl_wait();
  const long long n_words = (E + 31) >> 5;
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long w = warp0; w < n_words; w += nwarps) {
    const long long e = (w << 5) + lane;
    const unsigned int bits = __ballot_sync(0xffffffffu, e < E && pred[e] != 0);
    if (lane == 0) words[w] = bits;
  }
}

__global__ void decide_kernel(const float2* __restrict__ logits, long long E, uint8_t* __restrict__ pred, float* __restrict__ prob1) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    const float2 l = logits[e];
    if (pred) pred[e] = (l.y > l.x) ? 1 : 0;
    if (prob1) prob1[e] = softmax1(l.x, l.y);
  }
}

// ------------------------------------------------------------------------------------------------
// finalize: fixed-order reduction of block partials -> sums; sums -> folded constants
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// node encoder pieces: column statistics of a [M, Nc] activation, BN+ReLU apply
// ------------------------------------------------------------------------------------------------
constexpr int CS_ROWSPLIT_MAX = 64;
// grid (32-column tiles, row splits): fp64 partial sums per split; the LAST split block of a column tile (ticket counter)
// adds the partials in split order and folds them into the BatchNorm scale/shift of that tile's columns.
__global__ void __launch_bounds__(256) colstats_kernel(const float* __restrict__ Y, int M, int Nc, int rows_per_split,
                                                       double* __restrict__ part /*[splits][Nc][2]*/, unsigned int* __restrict__ tile_counter,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       float* __restrict__ scale, float* __restrict__ shift) {
  pdl_wait();
  __shared__ double ssum[8][33], ssq[8][33];
  __shared__ unsigned int s_ticket;
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  const int r0 = blockIdx.y * rows_per_split, r1 = min(r0 + rows_per_split, M);
  double s = 0.0, q = 0.0;
  if (col < Nc)
    for (int r = r0 + ry; r < r1; r += 8) {
      const double v = Y[(size_t)r * Nc + col];
      s += v;
      q += v * v;
    }
  ssum[ry][cx] = s;
  ssq[ry][cx] = q;
  __syncthreads();
  if (ry == 0 && col < Nc) {
    for (int i = 1; i < 8; ++i) { s += ssum[i][cx]; q += ssq[i][cx]; }
    part[((size_t)blockIdx.y * Nc + col) * 2 + 0] = s;
    part[((size_t)blockIdx.y * Nc + col) * 2 + 1] = q;
  }
  if (tile_counter == nullptr) return;                    // partials only (sharded encoder: reduced across ranks next)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(&tile_counter[blockIdx.x], 1u);
  __syncthreads();
  if (s_ticket != gridDim.y - 1) return;
  __threadfence();
  if (ry == 0 && col < Nc) {
    double ts = 0.0, tq = 0.0;
    for (int i = 0; i < (int)gridDim.y; ++i) {
      ts += __ldcg(&part[((size_t)i * Nc + col) * 2 + 0]);
      tq += __ldcg(&part[((size_t)i * Nc + col) * 2 + 1]);
    }
    const double mean = ts / M;
    double var = tq / M - mean * mean;
    if (var < 0.0) var = 0.0;
    const double sc = (double)gamma[col] / sqrt(var + (double)BN_EPS);
    scale[col] = (float)sc;
    shift[col] = (float)((double)beta[col] - sc * mean);
  }
  if (threadIdx.x == 0) tile_counter[blockIdx.x] = 0u;
}

// sharded node encoder: column sums of this rank's rows -> my slot -> flag; wait; add all ranks' slots in rank order;
// fold into the BatchNorm scale/shift over ALL M_total rows.  One block, one thread per column (Nc <= 1024).
__global__ void __launch_bounds__(1024) colstats_peer_kernel(const double* __restrict__ part, int splits, int Nc, int M_total,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             float* __restrict__ scale, float* __restrict__ shift,
                                                             const PeerArgs P, unsigned long long seq) {
  pdl_wait();
  const int col = threadIdx.x;
  const int slot = (int)(seq & 1ull);
  double* mine = P.cstats[P.rank] + (size_t)slot * MPN_PEER_CSTAT_COLS * 2;
  if (col < Nc) {
    double s = 0.0, q = 0.0;
    for (int i = 0; i < splits; ++i) {
      s += part[((size_t)i * Nc + col) * 2 + 0];
      q += part[((size_t)i * Nc + col) * 2 + 1];
    }
    mine[2 * col] = s;
    mine[2 * col + 1] = q;
  }
  __threadfence_system();
  __syncthreads();
  if (col == 0) st_release_sys(P.flags[P.rank] + 2 * KPEERS, seq);
  if (col < P.world) wait_flag(P.flags[col] + 2 * KPEERS, seq);
  __syncthreads();
  if (col < Nc) {
    double s = 0.0, q = 0.0;
    for (int r = 0; r < P.world; ++r) {
      const double* src = P.cstats[r] + (size_t)slot * MPN_PEER_CSTAT_COLS * 2 + 2 * col;
      double a, b;
      asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(a) : "l"(src));
      asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(b) : "l"(src + 1));
      s += a;
      q += b;
    }
    const double mean = s / M_total;
    double var = q / M_total - mean * mean;
    if (var < 0.0) var = 0.0;
    const double sc = (double)gamma[col] / sqrt(var + (double)BN_EPS);
    scale[col] = (float)sc;
    shift[col] = (float)((double)beta[col] - sc * mean);
  }
}

// final BatchNorm+ReLU of the sharded encoder: this rank's rows of h, stored locally and into every peer's h buffer
__global__ void bn_relu_apply_peer_kernel(const float* __restrict__ Y, int rows, int row_offset, const float* __restrict__ scale,
                                          const float* __restrict__ shift, const PeerArgs P) {
  pdl_wait();
  const long long total = (long long)rows * MPN_DH;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % MPN_DH);
    const float v = fmaxf(fmaf(Y[i], scale[c], shift[c]), 0.f);
    const size_t o = (size_t)row_offset * MPN_DH + (size_t)i;
    for (int r = 0; r < P.world; ++r) P.h[r][o] = v;
  }
}

__global__ void bn_relu_apply_kernel(const float* __restrict__ Y, long long total, int Nc, const float* __restrict__ scale,
                                     const float* __restrict__ shift, const int* __restrict__ row_gid, float* __restrict__ out) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % Nc);
    const size_t o = row_gid ? (size_t)row_gid[i / Nc] * Nc + c : (size_t)c;
    out[i] = fmaxf(fmaf(Y[i], scale[o], shift[o]), 0.f);
  }
}

// ------------------------------------------------------------------------------------------------
// per-step node tables:  Ps = h·Ws^T + b_e, Pd = h·Wd^T, A = h·Wh^T + b_n
// ------------------------------------------------------------------------------------------------
constexpr int NT_NODES = 64, NT_THREADS = 256, NT_OUT = 40;
// reattach_initial_nodes (RE_N): h_in = [h0 | h], so every table gets a second term with the weight columns of the initial
// encoding h0 (MPN_W_EDGE_W0 / MPN_W_NODE_W0).  At step 1 h == h0: the kernel reads h for both and saves it as h0.
template <bool RE_N>
__global__ void __launch_bounds__(NT_THREADS) node_tables_kernel(const float* __restrict__ h_full, float* __restrict__ h0_full,
                                                                 int first_step, int n_cols, int row_offset,
                                                                 int n_rows, const float* __restrict__ small,
                                                                 float* __restrict__ Ps, float* __restrict__ Pd,
                                                                 float* __restrict__ A) {
  pdl_wait();
  __shared__ float hs[NT_NODES][33];
  __shared__ float ws[NT_OUT][33];
  __shared__ float hs0[RE_N ? NT_NODES : 1][33];
  __shared__ float ws0[RE_N ? NT_OUT : 1][33];
  __shared__ float bs[NT_OUT];
  const int n0 = blockIdx.x * NT_NODES;
  for (int i = threadIdx.x; i < NT_NODES * 32; i += NT_THREADS) {
    const int n = n0 + (i >> 5);
    const float v = (n < n_cols) ? h_full[(size_t)n * 32 + (i & 31)] : 0.f;
    hs[i >> 5][i & 31] = v;
    if (RE_N) {
      float v0 = v;
      if (n < n_cols) {
        if (first_step) h0_full[(size_t)n * 32 + (i & 31)] = v;
        else v0 = h0_full[(size_t)n * 32 + (i & 31)];
      }
      hs0[i >> 5][i & 31] = v0;
    }
  }
  for (int i = threadIdx.x; i < NT_OUT * 32; i += NT_THREADS) {
    const int o = i >> 5, c = i & 31;
    float v, v0 = 0.f;
    if (o < 4) v = small[MPN_W_EDGE_W + o * 68 + c];                 // Ws: columns 0..31 of the 68-wide weight
    else if (o < 8) v = small[MPN_W_EDGE_W + (o - 4) * 68 + 32 + c]; // Wd: columns 32..63
    else v = small[MPN_W_NODE_W + (o - 8) * 36 + c];                 // Wh: columns 0..31 of the 36-wide weight
    ws[o][c] = v;
    if (RE_N) {
      if (o < 4) v0 = small[MPN_W_EDGE_W0 + o * 68 + c];
      else if (o < 8) v0 = small[MPN_W_EDGE_W0 + (o - 4) * 68 + 32 + c];
      else v0 = small[MPN_W_NODE_W0 + (o - 8) * 32 + c];
      ws0[o][c] = v0;
    }
  }
  if (threadIdx.x < NT_OUT) {
    const int o = threadIdx.x;
    bs[o] = (o < 4) ? small[MPN_W_EDGE_B + o] : (o < 8 ? 0.f : small[MPN_W_NODE_B + o - 8]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NT_NODES * NT_OUT; i += NT_THREADS) {
    const int ln = i / NT_OUT, o = i % NT_OUT;
    const int n = n0 + ln;
    if (n >= n_cols) continue;
    float s = bs[o];
    if (RE_N) {                                           // the reference's concat order: initial features first
#pragma unroll
      for (int c = 0; c < 32; ++c) s = fmaf(ws0[o][c], hs0[ln][c], s);
    }
#pragma unroll
    for (int c = 0; c < 32; ++c) s = fmaf(ws[o][c], hs[ln][c], s);
    const int lr = n - row_offset;
    if (o >= 4 && o < 8) Pd[(size_t)n * 4 + (o - 4)] = s;
    else if (lr >= 0 && lr < n_rows) {
      if (o < 4) Ps[(size_t)lr * 4 + o] = s;
      else A[(size_t)lr * 32 + (o - 8)] = s;
    }
  }
}

// h'[row] = sum over the row's tasks of msg_task (fixed order)  — the deterministic segment sum of models/mpn.py:202.
// PEERS: the rows are also stored into every other rank's h buffer over NVLink (the per-step all-gather of h).
// ABS (tensor-core apply): msg_task holds sum |z|;  sum relu(z) = (sum |z| + deg A' + W' . S1) / 2 with S1 = the row's sum of e'.
struct AbsFix {
  int on;
  int agg;                    // MPN_AGG_SUM | MPN_AGG_MEAN | MPN_AGG_MAX
  const float* A;
  const float4* s1_task;
  const float* consts;
};
template <bool PEERS>
__global__ void __launch_bounds__(256) node_finalize_kernel(const mpn_graph g, const float* __restrict__ msg_task,
                                                            float* __restrict__ h_full, const PeerArgs P, const AbsFix fix) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int n = gwarp; n < g.n_nodes; n += nwarps) {
    float s = 0.f;
    const int tb = g.taskptr[n], te = g.taskptr[n + 1];
    if (fix.agg == MPN_AGG_MAX) {
      for (int t = tb; t < te; ++t) s = fmaxf(s, msg_task[(size_t)t * MPN_DH + lane]);     // rows without edges -> 0 (torch_scatter)
    } else {
      for (int t = tb; t < te; ++t) s += msg_task[(size_t)t * MPN_DH + lane];
    }
    if (fix.on && te > tb) {
      float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int t = tb; t < te; ++t) {
        const float4 v = fix.s1_task[t];
        s1.x += v.x; s1.y += v.y; s1.z += v.z; s1.w += v.w;
      }
      const float deg = (float)(g.rowptr[n + 1] - g.rowptr[n]);
      const float ap = fmaf(fix.consts[FC_BN4_S + lane], fix.A[(size_t)n * MPN_DH + lane], fix.consts[FC_BN4_T + lane]);
      const float* w = fix.consts + FC_NODE_WE + 4 * lane;
      const float lin = fmaf(deg, ap, fmaf(w[0], s1.x, fmaf(w[1], s1.y, fmaf(w[2], s1.z, w[3] * s1.w))));
      s = 0.5f * (s + lin);
    }
    if (fix.agg == MPN_AGG_MEAN) s /= fmaxf((float)(g.rowptr[n + 1] - g.rowptr[n]), 1.f);   // scatter_mean: count clamped to >= 1
    const size_t o = (size_t)(g.row_offset + n) * MPN_DH + lane;
    h_full[o] = s;
    if (PEERS)
      for (int r = 0; r < P.world; ++r)
        if (r != P.rank) P.h[r][o] = s;
  }
}

}  // namespace mpn

// ================================================================================================
// plan + C ABI
// ================================================================================================
using namespace mpn;

struct mpn_fwd_plan {
  mpn_graph g;
  mpn_weights w;
  int L, n_cls, use_tc, max_dim;
  int msg_abs;                // the last apply sweep wrote sum |z| (tensor-core kernel)
  long long total_edges;
  float *act0, *act1, *colscale, *colshift;
  double* colpart;
  float *h_full, *h0_full, *Ps, *Pd, *A, *consts, *s1_task, *msg_task, *ybuf;
  double *partials, *partials2, *sums;
  unsigned int* fin_counter;
  unsigned long long* fix_sums;  // [8] fixed-point moment sums of the refined edge features (fused K1)
  int seq_m_active;              // sharded runs: the sweeps' last blocks do the peer exchange
  PeerArgs* peers_dev;           // sharded runs: device copy of the peer table (exchange fused into the sweeps' last blocks)
  unsigned long long seq_m;      // sharded runs: last moment-exchange sequence number used
  unsigned int* col_counter;   // [max_dim/32 + 1] ticket counters of the column-statistics tiles
  int fuse_fin;               // single-GPU: the last block of each moment sweep folds the constants itself
  int n_graphs;               // > 1: batched small graphs, BatchNorm statistics per graph
  double* n_total_dev;        // total edge count of the whole (sharded) graph, filled by the first fused all-reduce
  int n_total_on_device;
  double* task_part;          // [max_tasks][TASK_PART] per-task moment partials (batched)
  void* gemm_ws;
  size_t gemm_ws_bytes;
};

// Is the edge-update pre-activation y materialised (16 B / edge) and re-read by the later sweeps, or recomputed by each of
// them from (col, edge_attr, Pd[col])?  Multi-step runs need it anyway; for a single large graph with L == 1 it trades
// 24 B / edge of extra traffic for ~2 x 65 fewer instructions per edge in sweeps that are issue bound (measured: 0.41 ->
// 0.35 ms on configs[1] with the packed-fp32 apply kernel) and feeds the tensor-core apply kernel.  MPN_STORE_Y=0 disables.
static bool stores_y(const mpn_fwd_plan& p) {
  static int opt = -1;
  if (opt < 0) { const char* e = getenv("MPN_STORE_Y"); opt = e ? atoi(e) : 1; }
  return p.L > 1 || (p.L == 1 && opt != 0 && p.n_graphs <= 1);
}

static mpn::AbsFix abs_fix(const mpn_fwd_plan* p) {
  mpn::AbsFix f;
  f.on = p->msg_abs;
  f.agg = p->w.node_agg;
  f.A = p->A;
  f.s1_task = (const float4*)p->s1_task;
  f.consts = p->consts;
  return f;
}

static int plan_layout(mpn_fwd_plan& p, void* ws, size_t ws_bytes, size_t* need) {
  Arena a(ws, ws_bytes);
  const mpn_graph& g = p.g;
  int max_dim = 0;
  for (int i = 1; i <= p.w.n_node_layers; ++i) max_dim = p.w.node_dims[i] > max_dim ? p.w.node_dims[i] : max_dim;
  p.max_dim = max_dim;
  p.act0 = a.take<float>((size_t)g.n_cols * max_dim);
  p.act1 = a.take<float>((size_t)g.n_cols * max_dim);
  const size_t G = (g.n_graphs > 1 && g.node_gid && g.graph_nptr) ? (size_t)g.n_graphs : 1;
  p.n_graphs = (int)G;
  p.colscale = a.take<float>(G * (max_dim > 0 ? max_dim : 1));      // [G][Nc] tables when batched
  p.colshift = a.take<float>(G * (max_dim > 0 ? max_dim : 1));
  p.colpart = a.take<double>((size_t)CS_ROWSPLIT_MAX * (max_dim > 0 ? max_dim : 1) * 2);
  p.h_full = a.take<float>((size_t)g.n_cols * MPN_DH);
  p.h0_full = p.w.reattach_nodes ? a.take<float>((size_t)g.n_cols * MPN_DH) : nullptr;     // initial node encodings (reattach_initial_nodes)
  p.Ps = a.take<float>((size_t)g.n_nodes * 4);
  p.Pd = a.take<float>((size_t)g.n_cols * 4);
  p.A = a.take<float>((size_t)g.n_nodes * MPN_DH);
  p.consts = a.take<float>(G * FC_TOTAL);
  p.task_part = (G > 1) ? a.take<double>((size_t)g.max_tasks * TASK_PART) : nullptr;
  p.s1_task = a.take<float>((size_t)g.max_tasks * 4);
  p.msg_task = a.take<float>((size_t)g.max_tasks * MPN_DH);
  p.sums = a.take<double>(G * SUMS);
  p.partials = a.take<double>((size_t)SWEEP_GRID * SUMS);      // partials | fin_counter | fix_sums are adjacent: one memset clears
  p.partials2 = nullptr;                                       // them (clear_moment_state); the per-node moment part lives in the
  p.fin_counter = a.take<unsigned int>(FIN_COUNTERS);          // sweep's own partial rows
  p.fix_sums = a.take<unsigned long long>(8);
  p.peers_dev = a.take<PeerArgs>(1);
  p.n_total_dev = a.take<double>(1);
  p.col_counter = a.take<unsigned int>((size_t)(max_dim > 0 ? max_dim : 1) / 32 + 1);
  p.ybuf = stores_y(p) ? a.take<float>((size_t)g.n_edges * 4) : nullptr;
  size_t gw = 0;
  if (p.use_tc) {
    int prev = p.w.node_dims[0];
    for (int i = 0; i < p.w.n_node_layers; ++i) {
      size_t b = gemm_tc_workspace_bytes(g.n_cols, p.w.node_dims[i + 1], prev);
      gw = b > gw ? b : gw;
      prev = p.w.node_dims[i + 1];
    }
  }
  p.gemm_ws_bytes = gw;
  p.gemm_ws = gw ? (void*)a.take<char>(gw) : nullptr;
  if (need) *need = a.off;
  if (!a.ok()) {
    set_error("forward workspace too small: need %zu bytes, have %zu", a.off, ws_bytes);
    return MPN_ERR_WORKSPACE;
  }
  return MPN_OK;
}

static int check_weights(const mpn_weights* w) {
  MPN_REQUIRE(w != nullptr, "weights is NULL");
  MPN_REQUIRE(w->n_node_layers >= 1 && w->n_node_layers <= MPN_MAX_NODE_LAYERS, "n_node_layers must be in [1,%d]", MPN_MAX_NODE_LAYERS);
  MPN_REQUIRE(w->node_dims[w->n_node_layers] == MPN_DH, "node_out_dim must be %d (got %d)", MPN_DH, w->node_dims[w->n_node_layers]);
  for (int i = 0; i < w->n_node_layers; ++i)
    MPN_REQUIRE(w->node_w[i] && w->node_b[i] && w->node_gamma[i] && w->node_beta[i] && w->node_dims[i] > 0, "node layer %d has NULL tensors", i);
  MPN_REQUIRE(w->small != nullptr, "small weight block is NULL");
  MPN_REQUIRE(w->node_agg >= MPN_AGG_SUM && w->node_agg <= MPN_AGG_MAX, "node_agg must be MPN_AGG_SUM, _MEAN or _MAX (got %d)", w->node_agg);
  return MPN_OK;
}

extern "C" {

size_t mpn_forward_workspace_bytes(const mpn_graph* g, const mpn_weights* w, int32_t num_enc_steps) {
  if (!g || !w) return 0;
  mpn_fwd_plan p;
  memset(&p, 0, sizeof(p));
  p.g = *g; p.w = *w; p.L = num_enc_steps; p.use_tc = 1;
  size_t need = 0;
  plan_layout(p, nullptr, 0, &need);
  return need + 256;
}

int mpn_plan_create(mpn_fwd_plan** plan_out, const mpn_graph* g, const mpn_weights* w, int32_t L, int32_t n_cls,
                    int64_t total_edges, int use_tc, void* ws, size_t ws_bytes) {
  MPN_REQUIRE(plan_out && g && ws, "plan_create: NULL argument");
  MPN_TRY(check_weights(w));
  MPN_REQUIRE(L >= 0 && n_cls >= 0 && n_cls <= (L > 0 ? L : 1), "need 0 <= num_class_steps <= max(num_enc_steps,1)");
  MPN_REQUIRE(total_edges >= g->n_edges, "total_edges smaller than this shard's edges");
  MPN_REQUIRE(total_edges > 1, "BatchNorm over edges needs more than 1 edge (reference raises ValueError)");
  MPN_REQUIRE(g->n_cols > 1, "BatchNorm over nodes needs more than 1 node (reference raises ValueError)");
  MPN_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  mpn_fwd_plan* p = new (std::nothrow) mpn_fwd_plan;
  MPN_REQUIRE(p != nullptr, "out of host memory");
  memset(p, 0, sizeof(*p));
  p->g = *g; p->w = *w; p->L = L; p->n_cls = n_cls; p->use_tc = use_tc; p->total_edges = total_edges;
  int rc = plan_layout(*p, ws, ws_bytes, nullptr);
  if (rc != MPN_OK) { delete p; return rc; }
  *plan_out = p;
  return MPN_OK;
}

void mpn_plan_destroy(mpn_fwd_plan* plan) { delete plan; }
double* mpn_plan_sums(mpn_fwd_plan* plan) { return plan ? plan->sums : nullptr; }
float* mpn_plan_h_full(mpn_fwd_plan* plan) { return plan ? plan->h_full : nullptr; }

// partial rows, the last-block ticket and the fixed-point sums of the fused edge-feature kernel in one memset (every driver call
// before the first long kernel of a step is on the host's critical path)
static cudaError_t clear_moment_state(const mpn_fwd_plan* p, cudaStream_t st) {
  return cudaMemsetAsync(p->partials, 0, (size_t)((const char*)(p->fix_sums + 8) - (const char*)p->partials), st);
}

static FinArgs make_fin(const mpn_fwd_plan* p, int stage, bool fused) {
  FinArgs f;
  f.stage = stage;
  f.partials = p->partials;
  f.n_partials = SWEEP_GRID;
  f.row_stride = 1;
  f.partials2 = p->partials;             // the node-BN sweep writes its per-node part into the same partial rows
  f.n_partials2 = SWEEP_GRID;
  f.sums = p->sums;
  f.consts = p->consts;
  f.small = p->w.small;
  f.n_total = (double)p->total_edges;
  f.counter = fused ? p->fin_counter : nullptr;
  f.n_total_dev = p->n_total_on_device ? p->n_total_dev : nullptr;
  f.local_edges = (double)p->g.n_edges;
  f.fixed = nullptr;
  f.peers = nullptr;
  f.seq = 0;
  if (fused && p->seq_m_active) { f.peers = p->peers_dev; f.seq = ++const_cast<mpn_fwd_plan*>(p)->seq_m; }
  f.re_e = p->w.reattach_edges ? (stores_y(*p) ? 2 : 1) : 0;
  return f;
}

// FinArgs of a moment sweep launched on grid <= SWEEP_GRID blocks: the fold reads that many partial rows.  A separate reduce
// (phase API) adds SWEEP_GRID rows, and the rows beyond this grid still hold the previous stage's partial sums: they are cleared.
static int sweep_fin(const mpn_fwd_plan* p, int stage, bool fused, int grid, cudaStream_t st, FinArgs& f) {
  f = make_fin(p, stage, fused);
  f.n_partials = f.n_partials2 = grid;
  if (!fused && grid < SWEEP_GRID)
    MPN_CUDA_OK(cudaMemsetAsync(p->partials + (size_t)grid * SUMS, 0, sizeof(double) * (size_t)(SWEEP_GRID - grid) * SUMS, st));
  return MPN_OK;
}

// 3xFP16 planes for encoder layer l: cached weight planes present, K a multiple of 8 (TMA row stride), not disabled
static bool encoder_f16(const mpn_fwd_plan* p, int l, int K) {
  static int opt = -1;                               // MPN_ENC_F16=0 keeps the TF32 planes (diagnostics)
  if (opt < 0) { const char* e = getenv("MPN_ENC_F16"); opt = e ? atoi(e) : 1; }
  return opt != 0 && (K % 8) == 0 && p->w.node_w_hi16[l] && p->w.node_w_lo16[l] && p->w.node_w_scale16[l] > 0.f;
}
// Upper bound of |input of layer l|.  Layer 0: unknown (-1: measured on the device).  Layer l > 0 reads relu(BN(y)) of layer
// l-1 over M_total rows: a z-score of M values is at most sqrt(M-1) in magnitude, so |.| <= max|beta| + max|gamma| sqrt(M-1).
static float encoder_input_bound(const mpn_fwd_plan* p, int l, int M_total) {
  if (l == 0) return -1.f;
  const float b = p->w.node_bn_bmax[l - 1] + p->w.node_bn_gmax[l - 1] * sqrtf((float)(M_total > 1 ? M_total - 1 : 1));
  return b > 0.f ? b * 1.0001f : 1.f;
}

// layers [l_begin, l_end) of the node encoder; l_end == n_node_layers also writes h.  The pieces of one forward are enqueued in
// order on one stream (layer l reads the activations, column scale and shift that layer l-1 left in the plan's buffers).
// x: node features of element kind x_kind (MPN_X_*), read in place by layer 0's operand split
static int node_encoder_layers(mpn_fwd_plan* p, const void* x, int x_kind, int l_begin, int l_end, cudaStream_t st) {
  MPN_REQUIRE(p && x, "node_encoder: NULL argument");
  MPN_X_KIND_OK(x_kind);
  const int M = p->g.n_cols;
  const bool batched = p->n_graphs > 1;
  if (l_begin == 0) MPN_CUDA_OK(cudaMemsetAsync(p->col_counter, 0, sizeof(unsigned int) * ((size_t)p->max_dim / 32 + 1), st));
  float* bufs[2] = {p->act0, p->act1};
  const void* in = l_begin == 0 ? x : bufs[(l_begin - 1) & 1];
  int in_kind = l_begin == 0 ? x_kind : MPN_X_F32;
  const float *sc = l_begin == 0 ? nullptr : p->colscale, *sh = l_begin == 0 ? nullptr : p->colshift;
  for (int l = l_begin; l < l_end; ++l) {
    const int K = p->w.node_dims[l], Nc = p->w.node_dims[l + 1];
    float* out = bufs[l & 1];
    bool done = false;
    const int* gid = batched ? p->g.node_gid : nullptr;        // per-graph BatchNorm tables [G][K] when batched
    // the operand splits read four elements at once; a layer-0 input that is not aligned to that takes the SIMT loader
    if (p->use_tc && gemm_tc_supported(M, Nc, K) && x_vec4_aligned(in, in_kind)) {
      // tensor-core path: BatchNorm+ReLU of the previous layer is applied while the operand is split into its two planes
      if (encoder_f16(p, l, K))
        MPN_TRY(gemm_nt_tc_f16(in, p->w.node_b[l], out, M, Nc, K, p->gemm_ws, p->gemm_ws_bytes, st, sc, sh, gid,
                               encoder_input_bound(p, l, M), p->w.node_w_hi16[l], p->w.node_w_lo16[l], p->w.node_w_scale16[l], in_kind));
      else
        MPN_TRY(gemm_nt_tc(in, p->w.node_w[l], p->w.node_b[l], out, M, Nc, K, p->gemm_ws, p->gemm_ws_bytes, st, sc, sh,
                           p->w.node_w_hi[l], p->w.node_w_lo[l], gid, in_kind));
      done = true;
    }
    if (!done) MPN_TRY(gemm_nt_simt(in, p->w.node_w[l], p->w.node_b[l], sc, sh, out, M, Nc, K, st, gid, in_kind));
    if (batched) {
      mpn::launch(colstats_graph_kernel, dim3(div_up(Nc, 32), p->n_graphs), 256, 0, st, out, Nc, p->g.graph_nptr, p->w.node_gamma[l],
                                                                              p->w.node_beta[l], p->colscale, p->colshift);
    } else {
      int splits = div_up(M, 256);
      splits = splits > CS_ROWSPLIT_MAX ? CS_ROWSPLIT_MAX : splits;
      const int rps = div_up(M, splits);
      mpn::launch(colstats_kernel, dim3(div_up(Nc, 32), splits), 256, 0, st, out, M, Nc, rps, p->colpart, p->col_counter, p->w.node_gamma[l],
                                                                    p->w.node_beta[l], p->colscale, p->colshift);
    }
    MPN_LAUNCH_OK();
    in = out;
    in_kind = MPN_X_F32;
    sc = p->colscale;
    sh = p->colshift;
  }
  if (l_end < p->w.n_node_layers) return MPN_OK;
  MPN_REQUIRE(in_kind == MPN_X_F32, "node_encoder: no encoder layer between x and h");
  mpn::launch(bn_relu_apply_kernel, min(kNumSMs * 4, div_up((long long)M * MPN_DH, 256)), 256, 0, st, (const float*)in, (long long)M * MPN_DH, MPN_DH, sc, sh, batched ? p->g.node_gid : nullptr, p->h_full);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_plan_node_encoder_x(mpn_fwd_plan* p, const void* x, int32_t x_kind, void* stream) {
  MPN_REQUIRE(p && x, "node_encoder: NULL argument");
  return node_encoder_layers(p, x, x_kind, 0, p->w.n_node_layers, (cudaStream_t)stream);
}

int mpn_plan_node_encoder(mpn_fwd_plan* p, const float* x, void* stream) { return mpn_plan_node_encoder_x(p, x, MPN_X_F32, stream); }

// node encoder over this rank's row block only; BatchNorm column sums all-reduced through peer memory per layer;
// the encoded rows land in every rank's h buffer (publish of the h flag is left to the caller)
static int node_encoder_sharded(mpn_fwd_plan* p, const void* x, int x_kind, const PeerArgs& P, unsigned long long& seq_c, cudaStream_t st,
                                int l_begin, int l_end) {                 // layers [l_begin, l_end), as node_encoder_layers
  const int M = p->g.n_nodes, off = p->g.row_offset;
  float* bufs[2] = {p->act0, p->act1};
  const void* in = l_begin == 0 ? (const void*)((const char*)x + (size_t)off * p->w.node_dims[0] * x_elem_bytes(x_kind))
                                 : (const void*)bufs[(l_begin - 1) & 1];
  int in_kind = l_begin == 0 ? x_kind : MPN_X_F32;
  const float *sc = l_begin == 0 ? nullptr : p->colscale, *sh = l_begin == 0 ? nullptr : p->colshift;
  for (int l = l_begin; l < l_end; ++l) {
    const int K = p->w.node_dims[l], Nc = p->w.node_dims[l + 1];
    MPN_REQUIRE(Nc <= MPN_PEER_CSTAT_COLS, "sharded node encoder: layer width %d > %d", Nc, MPN_PEER_CSTAT_COLS);
    float* out = bufs[l & 1];
    // a 16-bit row block at offset off*K is aligned to four elements only when off*K % 4 == 0: else the SIMT loader
    const bool tc = p->use_tc && gemm_tc_supported(M, Nc, K) && x_vec4_aligned(in, in_kind);
    if (tc && encoder_f16(p, l, K))
      MPN_TRY(gemm_nt_tc_f16(in, p->w.node_b[l], out, M, Nc, K, p->gemm_ws, p->gemm_ws_bytes, st, sc, sh, nullptr,
                             encoder_input_bound(p, l, p->g.n_cols), p->w.node_w_hi16[l], p->w.node_w_lo16[l], p->w.node_w_scale16[l],
                             in_kind));
    else if (tc)
      MPN_TRY(gemm_nt_tc(in, p->w.node_w[l], p->w.node_b[l], out, M, Nc, K, p->gemm_ws, p->gemm_ws_bytes, st, sc, sh,
                         p->w.node_w_hi[l], p->w.node_w_lo[l], nullptr, in_kind));
    else
      MPN_TRY(gemm_nt_simt(in, p->w.node_w[l], p->w.node_b[l], sc, sh, out, M, Nc, K, st, nullptr, in_kind));
    int splits = div_up(M, 256);
    splits = splits > CS_ROWSPLIT_MAX ? CS_ROWSPLIT_MAX : splits;
    const int rps = div_up(M, splits);
    mpn::launch(colstats_kernel, dim3(div_up(Nc, 32), splits), 256, 0, st, out, M, Nc, rps, p->colpart, nullptr, p->w.node_gamma[l],
                                                                  p->w.node_beta[l], p->colscale, p->colshift);
    MPN_LAUNCH_OK();
    mpn::launch(colstats_peer_kernel, 1, 1024, 0, st, p->colpart, splits, Nc, p->g.n_cols, p->w.node_gamma[l], p->w.node_beta[l], p->colscale,
                                            p->colshift, P, ++seq_c);
    MPN_LAUNCH_OK();
    in = out;
    in_kind = MPN_X_F32;
    sc = p->colscale;
    sh = p->colshift;
  }
  if (l_end < p->w.n_node_layers) return MPN_OK;
  MPN_REQUIRE(in_kind == MPN_X_F32, "node_encoder: no encoder layer between x and h");
  mpn::launch(bn_relu_apply_peer_kernel, min(kNumSMs * 4, div_up((long long)M * MPN_DH, 256)), 256, 0, st, (const float*)in, M, off, sc, sh, P);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_plan_node_tables(mpn_fwd_plan* p, int32_t step, void* stream) {
  MPN_REQUIRE(p, "node_tables: NULL plan");
  if (p->w.reattach_nodes)
    mpn::launch(node_tables_kernel<true>, div_up(p->g.n_cols, NT_NODES), NT_THREADS, 0, (cudaStream_t)stream, 
        p->h_full, p->h0_full, step <= 1, p->g.n_cols, p->g.row_offset, p->g.n_nodes, p->w.small, p->Ps, p->Pd, p->A);
  else
    mpn::launch(node_tables_kernel<false>, div_up(p->g.n_cols, NT_NODES), NT_THREADS, 0, (cudaStream_t)stream, 
        p->h_full, nullptr, step <= 1, p->g.n_cols, p->g.row_offset, p->g.n_nodes, p->w.small, p->Ps, p->Pd, p->A);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_plan_sweep(mpn_fwd_plan* p, int32_t step, int32_t stage, const float* edge_attr, float* logits_out,
                   uint8_t* pred_out, float* prob1_out, void* stream) {
  MPN_REQUIRE(p && edge_attr, "sweep: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  const mpn_graph& g = p->g;
  const float2* ea = (const float2*)edge_attr;
  const bool stored = stores_y(*p);       // y materialised in ybuf
  const bool fused = p->fuse_fin != 0;
  const int flat_grid = (int)min((long long)SWEEP_GRID, (long long)div_up(g.n_edges > 0 ? g.n_edges : 1, SWEEP_THREADS));
  const bool batched = p->n_graphs > 1;
  const float4 *Ps4 = (const float4*)p->Ps, *Pd4 = (const float4*)p->Pd;
  float4* yb = (float4*)p->ybuf;
  if (batched) {
    // per-graph statistics: task-partial moments, then one block per graph reduces + folds (graph_finalize_kernel)
    double* tp = p->task_part;
    switch (stage) {
      case MPN_STAGE_ENC0:
        mpn::launch(enc_moments_task_kernel<0>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, p->consts, p->w.small, tp);
        break;
      case MPN_STAGE_ENC1:
        mpn::launch(enc_moments_task_kernel<1>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, p->consts, p->w.small, tp);
        break;
      case MPN_STAGE_EDGE:
        if (step == 1) {
          if (stored) mpn::launch(edge_moments_kernel<0, true, true>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, tp, make_fin(p, stage, false));
          else mpn::launch(edge_moments_kernel<0, false, true>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, nullptr, p->consts, tp, make_fin(p, stage, false));
        } else {
          if (p->w.reattach_edges) mpn::launch(edge_moments_kernel<1, true, true, true>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, tp, make_fin(p, stage, false));
          else mpn::launch(edge_moments_kernel<1, true, true>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, tp, make_fin(p, stage, false));
        }
        break;
      case MPN_STAGE_NODE:
        if (stored) mpn::launch(node_moments_sweep_kernel<1, true>, SWEEP_RESIDENT_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, (float4*)p->s1_task, tp, p->A, p->w.small, make_fin(p, stage, false));
        else mpn::launch(node_moments_sweep_kernel<0, true>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, nullptr, p->consts, (float4*)p->s1_task, tp, p->A, p->w.small, make_fin(p, stage, false));
        break;
      case MPN_STAGE_APPLY: {
        const bool classify = logits_out != nullptr;
        float2* lg = (float2*)logits_out;
        MPN_REQUIRE(p->L > 0, "batched graphs need num_enc_steps >= 1");
#define MPN_APPLY_B2(YS, CL, MX) mpn::launch(apply_kernel<YS, CL, true, MX>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->A, p->consts, p->msg_task, lg, pred_out, prob1_out)
#define MPN_APPLY_B(YS, CL) do { if (p->w.node_agg == MPN_AGG_MAX) MPN_APPLY_B2(YS, CL, true); else MPN_APPLY_B2(YS, CL, false); } while (0)
        if (stored) { if (classify) MPN_APPLY_B(1, true); else MPN_APPLY_B(1, false); }
        else        { if (classify) MPN_APPLY_B(0, true); else MPN_APPLY_B(0, false); }
#undef MPN_APPLY_B
#undef MPN_APPLY_B2
        break;
      }
      default:
        MPN_REQUIRE(false, "unknown stage %d", stage);
    }
    MPN_LAUNCH_OK();
    if (stage != MPN_STAGE_APPLY) {
      mpn::launch(graph_finalize_kernel, p->n_graphs, 128, 0, st, stage, g, tp, p->A, (const float4*)p->s1_task, p->w.small, p->sums, p->consts,
                                                         p->w.reattach_edges ? (stored ? 2 : 1) : 0);
      MPN_LAUNCH_OK();
    }
    return MPN_OK;
  }
  switch (stage) {
    case MPN_STAGE_ENC0:
      MPN_CUDA_OK(clear_moment_state(p, st));
      mpn::launch(enc_moments_kernel<0>, flat_grid, SWEEP_THREADS, 0, st, ea, g.n_edges, p->consts, p->w.small, p->partials, make_fin(p, stage, fused),
                  (const int*)nullptr);
      break;
    case MPN_STAGE_ENC1:
      if ((((uintptr_t)ea) & 15) == 0 && g.n_edges >= 2) {
        const long long n_pairs = g.n_edges >> 1;
        const int pgrid = (int)min((long long)kNumSMs * 2, (long long)div_up(n_pairs, SWEEP_THREADS));
        FinArgs pf;
        MPN_TRY(sweep_fin(p, stage, fused, pgrid, st, pf));
        mpn::launch(enc_moments1_packed_kernel, pgrid, SWEEP_THREADS, 0, st, (const float4*)ea, n_pairs, ea, g.n_edges, p->consts, p->w.small,
                    p->partials, pf);
      } else {
        mpn::launch(enc_moments_kernel<1>, flat_grid, SWEEP_THREADS, 0, st, ea, g.n_edges, p->consts, p->w.small, p->partials, make_fin(p, stage, fused),
                    (const int*)nullptr);
      }
      break;
    case MPN_STAGE_EDGE:
      if (step == 1) {
        if (stored) mpn::launch(edge_moments_kernel<0, true, false>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, p->partials, make_fin(p, stage, fused));
        else mpn::launch(edge_moments_kernel<0, false, false>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, nullptr, p->consts, p->partials, make_fin(p, stage, fused));
      } else {
        if (p->w.reattach_edges) mpn::launch(edge_moments_kernel<1, true, false, true>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, p->partials, make_fin(p, stage, fused));
        else mpn::launch(edge_moments_kernel<1, true, false>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, p->partials, make_fin(p, stage, fused));
      }
      break;
    case MPN_STAGE_NODE: {
      FinArgs nf;
      MPN_TRY(sweep_fin(p, stage, fused, stored ? SWEEP_RESIDENT_GRID : SWEEP_GRID, st, nf));
      if (stored) mpn::launch(node_moments_sweep_kernel<1, false>, SWEEP_RESIDENT_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->consts, (float4*)p->s1_task, p->partials, p->A, p->w.small, nf);
      else mpn::launch(node_moments_sweep_kernel<0, false>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, nullptr, p->consts, (float4*)p->s1_task, p->partials, p->A, p->w.small, nf);
      break;
    }
    case MPN_STAGE_APPLY: {
      const bool classify = logits_out != nullptr;
      float2* lg = (float2*)logits_out;
      if (p->L == 0) {
        MPN_REQUIRE(classify, "L == 0 needs a logits buffer");
        mpn::launch(classify_encoded_kernel, flat_grid, SWEEP_THREADS, 0, st, ea, g.n_edges, p->consts, lg, pred_out, prob1_out);
        break;
      }
      // tensor-core variant: stored-y runs on graphs with >= 128-edge tasks (MPN_APPLY_TC=0 selects the packed-fp32 kernel)
      static int apply_tc = -1;
      if (apply_tc < 0) { const char* e = getenv("MPN_APPLY_TC"); apply_tc = e ? atoi(e) : 1; }
      p->msg_abs = 0;
      if (p->use_tc && apply_tc && stored && g.chunk >= ATC_THREADS && (!classify || (pred_out != nullptr) == (prob1_out != nullptr))) {
        const bool agg_max = p->w.node_agg == MPN_AGG_MAX;
        p->msg_abs = agg_max ? 0 : 1;                      // msg_task holds sum |z|: node_finalize adds the closed-form half
#define MPN_ATC3(CL, DE, MX, NC) mpn::launch(apply_tc_kernel<CL, DE, MX, NC>, kNumSMs * NC, ATC_THREADS, 0, st, g, yb, p->A, p->consts, p->msg_task, lg, pred_out, prob1_out)
#define MPN_ATC2(CL, DE, MX) MPN_ATC3(CL, DE, MX, ATC_CTAS_PER_SM)
#define MPN_ATC(CL, DE) do { if (agg_max) MPN_ATC2(CL, DE, true); else MPN_ATC2(CL, DE, false); } while (0)
        if (!classify) MPN_ATC(false, false);
        else if (pred_out && prob1_out) MPN_ATC(true, true);
        else MPN_ATC(true, false);
#undef MPN_ATC
#undef MPN_ATC2
#undef MPN_ATC3
        break;
      }
#define MPN_APPLY2(YS, CL, MX) mpn::launch(apply_kernel<YS, CL, false, MX>, SWEEP_GRID, SWEEP_THREADS, 0, st, g, ea, Ps4, Pd4, yb, p->A, p->consts, p->msg_task, lg, pred_out, prob1_out)
#define MPN_APPLY(YS, CL) do { if (p->w.node_agg == MPN_AGG_MAX) MPN_APPLY2(YS, CL, true); else MPN_APPLY2(YS, CL, false); } while (0)
      if (stored) { if (classify) MPN_APPLY(1, true); else MPN_APPLY(1, false); }
      else        { if (classify) MPN_APPLY(0, true); else MPN_APPLY(0, false); }
#undef MPN_APPLY
#undef MPN_APPLY2
      break;
    }
    default:
      MPN_REQUIRE(false, "unknown stage %d", stage);
  }
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_plan_finalize(mpn_fwd_plan* p, int32_t step, int32_t stage, void* stream) {
  MPN_REQUIRE(p, "finalize: NULL plan");
  (void)step;
  if (p->n_graphs > 1) return MPN_OK;     // batched: graph_finalize_kernel already ran after the sweep
  // sums already reduced (and possibly all-reduced by the host): constants only
  mpn::launch(finalize_kernel, 1, FIN_THREADS, 0, (cudaStream_t)stream, make_fin(p, stage, false), 0, 1);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

// reduce this rank's block partials into the sums vector (phase API: host all-reduces it afterwards)
int mpn_plan_reduce(mpn_fwd_plan* p, int32_t stage, int with_consts, void* stream) {
  MPN_REQUIRE(p, "reduce: NULL plan");
  if (p->n_graphs > 1) return MPN_OK;     // batched: graph_finalize_kernel already ran after the sweep
  mpn::launch(finalize_kernel, 1, FIN_THREADS, 0, (cudaStream_t)stream, make_fin(p, stage, false), 1, with_consts);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_plan_node_finalize(mpn_fwd_plan* p, int32_t step, void* stream) {
  MPN_REQUIRE(p, "node_finalize: NULL plan");
  (void)step;
  mpn::launch(node_finalize_kernel<false>, min(kNumSMs * 8, div_up((long long)p->g.n_nodes * 32, 256)), 256, 0, (cudaStream_t)stream, p->g, p->msg_task, p->h_full, PeerArgs(), abs_fix(p));
  MPN_LAUNCH_OK();
  return MPN_OK;
}

// per-device side stream + fork/join events (created once, never destroyed)
struct SideStream {
  cudaStream_t stream;
  cudaEvent_t fork, join;
};
static SideStream* side_stream() {
  static SideStream table[64];
  static int state[64];                 // 0 = not tried, 1 = ok, -1 = failed
  static std::mutex init_lock;          // (the library is used by one host thread per device; creation is guarded all the same)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> hold(init_lock);
  if (state[dev] == 0) {
    SideStream& s = table[dev];
    const bool ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess &&
                    cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) == cudaSuccess &&
                    cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) == cudaSuccess;
    state[dev] = ok ? 1 : -1;
  }
  return state[dev] == 1 ? &table[dev] : nullptr;
}

// Timeline of one forward (bench.py / tools): events at the phase boundaries of the caller's stream and at the end of the
// side-stream encoder.  Off by default (an event record between two kernels ends their programmatic overlap).
constexpr int TL_MAX = 24;
static bool g_tl_on = false;
static cudaEvent_t g_tl_ev[TL_MAX];
static const char* g_tl_name[TL_MAX];
static int g_tl_n = 0;
static void tl_mark(const char* name, cudaStream_t st, bool first = false) {
  if (!g_tl_on) return;
  if (first) g_tl_n = 0;
  if (g_tl_n >= TL_MAX) return;
  if (!g_tl_ev[g_tl_n] && cudaEventCreate(&g_tl_ev[g_tl_n]) != cudaSuccess) return;
  if (cudaEventRecord(g_tl_ev[g_tl_n], st) != cudaSuccess) return;
  g_tl_name[g_tl_n++] = name;
}

// ef_ws != NULL: edge_attr is an OUTPUT, produced here by mpn_edge_features on the main stream while the node encoder runs on
// the side stream (both only read x)
static int forward_impl(const mpn_graph* g, const mpn_weights* w, const void* x, int x_kind, float* edge_attr_rw, int32_t L,
                        int32_t n_cls, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out, int use_tc, void* ws,
                        size_t ws_bytes, void* ef_ws, size_t ef_ws_bytes, void* stream) {
  const float* edge_attr = edge_attr_rw;
  MPN_REQUIRE(g && x && edge_attr && logits_out, "forward: NULL argument");
  MPN_X_KIND_OK(x_kind);
  MPN_REQUIRE(g->row_offset == 0 && g->n_cols == g->n_nodes, "mpn_forward runs an unsharded graph; use the plan API for row blocks");
  cudaStream_t st = (cudaStream_t)stream;
  mpn_fwd_plan* p = nullptr;
  MPN_TRY(mpn_plan_create(&p, g, w, L, n_cls, g->n_edges, use_tc, ws, ws_bytes));
  int rc = MPN_OK;
  const size_t lstride = (size_t)g->n_edges * 2;
#define STEP_TRY(expr) do { rc = (expr); if (rc != MPN_OK) goto done; } while (0)
  p->fuse_fin = (p->n_graphs > 1) ? 0 : 1;
  {
    // the node encoder (tensor-core GEMM chain) depends neither on the edge features nor on the edge-encoder sweeps: it runs
    // on a side stream while the caller's stream does the edge chain
    SideStream* ss = side_stream();
    tl_mark("start", st, true);
    const bool fork = ss != nullptr && cudaEventRecord(ss->fork, st) == cudaSuccess && cudaStreamWaitEvent(ss->stream, ss->fork, 0) == cudaSuccess;
    // Enqueue order (measured, profiles/r2_05_enqueue_order.md): first encoder layer (the big GEMM, on the idle device), then the
    // edge-feature kernels (they head the critical path), then the small later encoder layers, which fit beside the Gram kernel
    // (it leaves SMs free, gram_ef.cu) and are wanted only at the join after the second sweep.  Without a side stream (or without
    // fused features) the whole encoder is enqueued first, as stream order then demands.
    bool encoder_enqueued = false;
    int enc_done_layers = 0;
#define ENQUEUE_ENCODER() do { if (!encoder_enqueued) { encoder_enqueued = true; \
      STEP_TRY(node_encoder_layers(p, x, x_kind, enc_done_layers, p->w.n_node_layers, fork ? ss->stream : st)); \
      tl_mark("node_encoder_end(side stream)", fork ? ss->stream : st); \
      if (fork && cudaEventRecord(ss->join, ss->stream) != cudaSuccess) { set_error("event record failed"); rc = MPN_ERR_CUDA; goto done; } } } while (0)
    if (!fork || ef_ws == nullptr) ENQUEUE_ENCODER();
    else if (p->w.n_node_layers > 1) {
      // the first (largest) encoder layer starts on the idle device; the later, small ones fit beside the Gram kernel
      STEP_TRY(node_encoder_layers(p, x, x_kind, 0, 1, ss->stream));
      enc_done_layers = 1;
    }
    bool enc0_done = false;
    if (ef_ws != nullptr && p->n_graphs <= 1) {
      // K1 with the first encoder BatchNorm's moment sums taken in the GEMM epilogue (dense cross-camera graphs): the ENC0 sweep
      // over edge_attr is replaced by one finalize block; for a graph whose layout is decided on the device the sweep is
      // enqueued behind a flag test and returns at once when the fused kernel ran
      if (clear_moment_state(p, st) != cudaSuccess) { set_error("memset failed"); rc = MPN_ERR_CUDA; goto done; }
      EfMoments mom;
      mom.partials = p->partials; mom.fixed_sums = p->fix_sums; mom.handled_flag = nullptr; mom.known_fused = 0;
      STEP_TRY(edge_features_impl(g, x, x_kind, w->node_dims[0], edge_attr_rw, use_tc, ef_ws, ef_ws_bytes, st, &mom));
      ENQUEUE_ENCODER();
      if (mom.handled_flag != nullptr) {
        if (!mom.known_fused) {
          const int flat_grid = (int)min((long long)SWEEP_GRID, (long long)div_up(g->n_edges > 0 ? g->n_edges : 1, SWEEP_THREADS));
          mpn::launch(enc_moments_kernel<0>, flat_grid, SWEEP_THREADS, 0, st, (const float2*)edge_attr, g->n_edges, p->consts, p->w.small,
                      p->partials, make_fin(p, MPN_STAGE_ENC0, false), mom.handled_flag);
          ++mpn::g_kernel_launches;
        }
        FinArgs f = make_fin(p, MPN_STAGE_ENC0, false);
        f.fixed = p->fix_sums;
        mpn::launch(finalize_kernel, 1, FIN_THREADS, 0, st, f, 1, 1);
        ++mpn::g_kernel_launches;
        if (cudaGetLastError() != cudaSuccess) { set_error("ENC0 finalize launch failed"); rc = MPN_ERR_CUDA; goto done; }
        // the later sweeps reduce SWEEP_GRID partial rows and write only their own grid's: rows the fused kernel may have
        // written beyond that grid must read zero again (never the case for a dense graph: E / 256 >= tiles)
        if ((long long)kNumSMs > (long long)div_up(g->n_edges > 0 ? g->n_edges : 1, SWEEP_THREADS) &&
            cudaMemsetAsync(p->partials, 0, sizeof(double) * SWEEP_GRID * SUMS, st) != cudaSuccess) { set_error("memset failed"); rc = MPN_ERR_CUDA; goto done; }
        enc0_done = true;
      }
    } else if (ef_ws != nullptr) {
      STEP_TRY(edge_features_impl(g, x, x_kind, w->node_dims[0], edge_attr_rw, use_tc, ef_ws, ef_ws_bytes, st, nullptr));
    }
    ENQUEUE_ENCODER();
#undef ENQUEUE_ENCODER
    if (!enc0_done) STEP_TRY(mpn_plan_sweep(p, 0, MPN_STAGE_ENC0, edge_attr, nullptr, nullptr, nullptr, st));
    tl_mark("edge_features+enc0_end", st);
    STEP_TRY(mpn_plan_sweep(p, 0, MPN_STAGE_ENC1, edge_attr, nullptr, nullptr, nullptr, st));
    tl_mark("enc1_end", st);
    if (fork && cudaStreamWaitEvent(st, ss->join, 0) != cudaSuccess) { set_error("stream wait failed"); rc = MPN_ERR_CUDA; goto done; }
    tl_mark("joined", st);
  }
  if (L == 0) {
    STEP_TRY(mpn_plan_sweep(p, 0, MPN_STAGE_APPLY, edge_attr, logits_out, pred_out, prob1_out, st));
  }
  {
    const int first_class_step = L - n_cls + 1;
    int k = 0;
    for (int step = 1; step <= L; ++step) {
      STEP_TRY(mpn_plan_node_tables(p, step, st));
      tl_mark("node_tables_end", st);
      STEP_TRY(mpn_plan_sweep(p, step, MPN_STAGE_EDGE, edge_attr, nullptr, nullptr, nullptr, st));
      tl_mark("edge_update_end", st);
      STEP_TRY(mpn_plan_sweep(p, step, MPN_STAGE_NODE, edge_attr, nullptr, nullptr, nullptr, st));
      tl_mark("node_moments_end", st);
      const bool cls = step >= first_class_step;
      const bool last = step == L;
      STEP_TRY(mpn_plan_sweep(p, step, MPN_STAGE_APPLY, edge_attr, cls ? logits_out + lstride * k : nullptr,
                              (cls && last) ? pred_out : nullptr, (cls && last) ? prob1_out : nullptr, st));
      if (cls) ++k;
      tl_mark("node_apply_end", st);
      STEP_TRY(mpn_plan_node_finalize(p, step, st));
      tl_mark("node_finalize_end", st);
    }
  }
  if (h_out) {
    cudaError_t e = cudaMemcpyAsync(h_out, p->h_full, sizeof(float) * (size_t)g->n_nodes * MPN_DH, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { set_error("h copy failed: %s", cudaGetErrorString(e)); rc = MPN_ERR_CUDA; }
  }
#undef STEP_TRY
done:
  mpn_plan_destroy(p);
  return rc;
}

int mpn_forward_x(const mpn_graph* g, const mpn_weights* w, const void* x, int32_t x_kind, const float* edge_attr, int32_t L,
                  int32_t n_cls, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out, int use_tc, void* ws,
                  size_t ws_bytes, void* stream) {
  return forward_impl(g, w, x, x_kind, const_cast<float*>(edge_attr), L, n_cls, logits_out, h_out, pred_out, prob1_out, use_tc, ws,
                      ws_bytes, nullptr, 0, stream);
}

int mpn_forward(const mpn_graph* g, const mpn_weights* w, const float* x, const float* edge_attr, int32_t L, int32_t n_cls,
                float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out, int use_tc, void* ws, size_t ws_bytes,
                void* stream) {
  return mpn_forward_x(g, w, x, MPN_X_F32, edge_attr, L, n_cls, logits_out, h_out, pred_out, prob1_out, use_tc, ws, ws_bytes, stream);
}

int mpn_forward_with_edge_features_x(const mpn_graph* g, const mpn_weights* w, const void* x, int32_t x_kind, float* edge_attr_out,
                                     int32_t L, int32_t n_cls, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out,
                                     int use_tc, void* ws, size_t ws_bytes, void* ef_ws, size_t ef_ws_bytes, void* stream) {
  MPN_REQUIRE(ef_ws != nullptr && edge_attr_out != nullptr, "forward_with_edge_features: NULL edge-feature buffer / workspace");
  return forward_impl(g, w, x, x_kind, edge_attr_out, L, n_cls, logits_out, h_out, pred_out, prob1_out, use_tc, ws, ws_bytes, ef_ws,
                      ef_ws_bytes, stream);
}

int mpn_forward_with_edge_features(const mpn_graph* g, const mpn_weights* w, const float* x, float* edge_attr_out, int32_t L,
                                   int32_t n_cls, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out, int use_tc,
                                   void* ws, size_t ws_bytes, void* ef_ws, size_t ef_ws_bytes, void* stream) {
  return mpn_forward_with_edge_features_x(g, w, x, MPN_X_F32, edge_attr_out, L, n_cls, logits_out, h_out, pred_out, prob1_out, use_tc,
                                          ws, ws_bytes, ef_ws, ef_ws_bytes, stream);
}

// ef_ws != NULL: edge_attr is an OUTPUT, produced here by the fused edge-feature kernel on the caller's stream (it overlaps the
// node encoder on the side stream and hands over the first encoder BatchNorm's moment sums: no ENC0 sweep)
static int forward_sharded_impl(const mpn_graph* g, const mpn_weights* w, const void* x, int x_kind, float* edge_attr_rw, int32_t L,
                                int32_t n_cls, int64_t total_edges, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out,
                                int use_tc, const mpn_peer_ctx* peers, void* ws, size_t ws_bytes, void* ef_ws, size_t ef_ws_bytes,
                                void* stream) {
  const float* edge_attr = edge_attr_rw;
  MPN_REQUIRE(g && x && edge_attr && logits_out && peers, "forward_sharded: NULL argument");
  MPN_X_KIND_OK(x_kind);
  MPN_REQUIRE(peers->world >= 1 && peers->world <= MPN_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world, "forward_sharded: bad rank/world");
  MPN_REQUIRE(g->n_graphs <= 1, "forward_sharded: batched graphs cannot be row-sharded");
  MPN_REQUIRE(L >= 1, "forward_sharded needs num_enc_steps >= 1");
  PeerArgs P;
  P.rank = peers->rank;
  P.world = peers->world;
  for (int r = 0; r < peers->world; ++r) {
    MPN_REQUIRE(peers->sums[r] && peers->flags[r] && (L <= 1 || peers->h[r]), "forward_sharded: NULL peer buffer for rank %d", r);
    MPN_REQUIRE(!peers->shard_node_encoder || (peers->h[r] && peers->cstats[r]), "forward_sharded: sharded encoder needs h and cstats buffers");
    P.sums[r] = peers->sums[r];
    P.flags[r] = (unsigned long long*)peers->flags[r];
    P.h[r] = peers->h[r];
    P.cstats[r] = peers->cstats[r];
  }
  const bool shard_enc = peers->shard_node_encoder != 0;
  cudaStream_t st = (cudaStream_t)stream;
  mpn_fwd_plan* p = nullptr;
  // total_edges <= 0: the ranks' edge counts travel with the first fused all-reduce (no host collective at all)
  MPN_TRY(mpn_plan_create(&p, g, w, L, n_cls, total_edges > 0 ? total_edges : (int64_t)1 << 40, use_tc, ws, ws_bytes));
  p->n_total_on_device = total_edges > 0 ? 0 : 1;
  if (L > 1 || shard_enc) p->h_full = peers->h[peers->rank];            // node tables read the peer-visible buffer
  // the moment exchange of every BatchNorm runs in the last block of the sweep that produced the partial sums
  p->fuse_fin = 1;
  p->seq_m_active = 1;
  p->seq_m = peers->seq_moments;
  int rc = MPN_OK;
  unsigned long long& seq_m = p->seq_m;
  unsigned long long seq_h = peers->seq_h, seq_c = peers->seq_c;
  if (cudaMemcpyAsync(p->peers_dev, &P, sizeof(PeerArgs), cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemsetAsync(p->fin_counter, 0, sizeof(unsigned int) * FIN_COUNTERS, st) != cudaSuccess) {
    set_error("peer table upload failed");
    mpn_plan_destroy(p);
    return MPN_ERR_CUDA;
  }
  bool h_pending = false;                                   // an h exchange has been published and not yet awaited
  const size_t lstride = (size_t)g->n_edges * 2;
  // shared symmetric Gram: every pair of nodes computed by one rank, the mirrored entry stored into its owner's edge_attr
  GeShare share;
  const GeShare* share_ptr = nullptr;
  if (ef_ws != nullptr && peers->world >= 2 && peers->edge_attr[0] != nullptr) {
    memset(&share, 0, sizeof(share));
    share.rank = peers->rank; share.world = peers->world; share.seq = peers->seq_t + 1;
    for (int r = 0; r < peers->world; ++r) {
      if (!(peers->edge_attr[r] && peers->node_tables[r])) { set_error("forward_sharded: NULL shared-Gram buffer for rank %d", r); mpn_plan_destroy(p); return MPN_ERR_INVALID; }
      share.ea[r] = (float2*)peers->edge_attr[r];
      share.tab[r] = (int4*)peers->node_tables[r];
      share.flags[r] = (unsigned long long*)peers->flags[r];
      share.blk[r] = peers->block_start[r];
    }
    share.blk[peers->world] = peers->block_start[peers->world];
    share_ptr = &share;
  }
#define STEP_TRY(expr) do { rc = (expr); if (rc != MPN_OK) goto done; } while (0)
#define PEER_FINALIZE(stage) do { mpn::launch(finalize_peer_kernel, 1, FIN_THREADS, 0, st, make_fin(p, stage, false), P, ++seq_m); \
    ++mpn::g_kernel_launches; if (cudaGetLastError() != cudaSuccess) { set_error("finalize_peer launch failed"); rc = MPN_ERR_CUDA; goto done; } } while (0)
  // first encoder BatchNorm: a sweep over edge_attr, or (features computed here by the fused kernel) the partial rows of its epilogue
#define ENC0_STAGE() do { \
    bool enc0_done_ = false; \
    if (ef_ws != nullptr) { \
      if (clear_moment_state(p, st) != cudaSuccess) { set_error("memset failed"); rc = MPN_ERR_CUDA; goto done; } \
      EfMoments mom_; \
      mom_.partials = p->partials; mom_.fixed_sums = p->fix_sums; mom_.handled_flag = nullptr; mom_.known_fused = 0; \
      STEP_TRY(edge_features_impl(g, x, x_kind, w->node_dims[0], edge_attr_rw, use_tc, ef_ws, ef_ws_bytes, st, &mom_, share_ptr)); \
      if (mom_.handled_flag != nullptr) { \
        if (!mom_.known_fused) {   /* layout decided on the device: the sweep runs only if the fused kernel did not */ \
          const int fg_ = (int)min((long long)SWEEP_GRID, (long long)div_up(g->n_edges > 0 ? g->n_edges : 1, SWEEP_THREADS)); \
          mpn::launch(enc_moments_kernel<0>, fg_, SWEEP_THREADS, 0, st, (const float2*)edge_attr, g->n_edges, p->consts, p->w.small, \
                      p->partials, make_fin(p, MPN_STAGE_ENC0, false), mom_.handled_flag); \
          ++mpn::g_kernel_launches; \
        } \
        FinArgs f_ = make_fin(p, MPN_STAGE_ENC0, false); \
        f_.fixed = p->fix_sums; \
        mpn::launch(finalize_peer_kernel, 1, FIN_THREADS, 0, st, f_, P, ++seq_m); \
        ++mpn::g_kernel_launches; \
        if (cudaGetLastError() != cudaSuccess) { set_error("finalize_peer launch failed"); rc = MPN_ERR_CUDA; goto done; } \
        enc0_done_ = true; \
      } \
    } \
    if (!enc0_done_) STEP_TRY(mpn_plan_sweep(p, 0, MPN_STAGE_ENC0, edge_attr, nullptr, nullptr, nullptr, st)); \
    } while (0)
  if (shard_enc) {
    // every rank encodes its own rows; column statistics and the encoded rows travel over NVLink inside the kernels.  The
    // encoder chain (GEMMs + column-statistics exchanges, flag word 2, then the h publish, flag word 1) runs on the side stream
    // while the caller's stream does the two encoder sweeps over edge_attr and their moment exchanges (flag word 0): the two
    // chains touch different exchange slots and meet again before the first node tables.
    SideStream* ss = side_stream();
    tl_mark("start", st, true);
    const bool fork = ss != nullptr && cudaEventRecord(ss->fork, st) == cudaSuccess && cudaStreamWaitEvent(ss->stream, ss->fork, 0) == cudaSuccess;
    cudaStream_t es = fork ? ss->stream : st;
    // enqueue order as in forward_impl: first encoder layer, edge features (they head the critical path), later layers
    const int n_first = (fork && ef_ws != nullptr && p->w.n_node_layers > 1) ? 1 : p->w.n_node_layers;
    STEP_TRY(node_encoder_sharded(p, x, x_kind, P, seq_c, es, 0, n_first));
    if (n_first < p->w.n_node_layers) {
      ENC0_STAGE();
      tl_mark("edge_features+enc0_end", st);
      STEP_TRY(node_encoder_sharded(p, x, x_kind, P, seq_c, es, n_first, p->w.n_node_layers));
    }
    mpn::launch(peer_publish_h_kernel, 1, 32, 0, es, P, ++seq_h);
    ++mpn::g_kernel_launches;
    h_pending = true;
    tl_mark("node_encoder_end(side stream)", es);
    if (fork && cudaEventRecord(ss->join, ss->stream) != cudaSuccess) { set_error("event record failed"); rc = MPN_ERR_CUDA; goto done; }
    if (n_first == p->w.n_node_layers) {
      ENC0_STAGE();
      tl_mark("edge_features+enc0_end", st);
    }
    STEP_TRY(mpn_plan_sweep(p, 0, MPN_STAGE_ENC1, edge_attr, nullptr, nullptr, nullptr, st));
    tl_mark("enc1_end", st);
    if (fork && cudaStreamWaitEvent(st, ss->join, 0) != cudaSuccess) { set_error("stream wait failed"); rc = MPN_ERR_CUDA; goto done; }
    tl_mark("joined", st);
  } else {
    SideStream* ss = side_stream();
    const bool fork = ss != nullptr && cudaEventRecord(ss->fork, st) == cudaSuccess && cudaStreamWaitEvent(ss->stream, ss->fork, 0) == cudaSuccess;
    STEP_TRY(mpn_plan_node_encoder_x(p, x, x_kind, fork ? ss->stream : st));
    if (fork && cudaEventRecord(ss->join, ss->stream) != cudaSuccess) { set_error("event record failed"); rc = MPN_ERR_CUDA; goto done; }
    ENC0_STAGE();
    STEP_TRY(mpn_plan_sweep(p, 0, MPN_STAGE_ENC1, edge_attr, nullptr, nullptr, nullptr, st));
    if (fork && cudaStreamWaitEvent(st, ss->join, 0) != cudaSuccess) { set_error("stream wait failed"); rc = MPN_ERR_CUDA; goto done; }
  }
  {
    const int first_class_step = L - n_cls + 1;
    int k = 0;
    for (int step = 1; step <= L; ++step) {
      if (h_pending) {                                      // every rank's rows of h must have landed in my buffer
        mpn::launch(peer_wait_h_kernel, 1, 32, 0, st, P, seq_h);
        ++mpn::g_kernel_launches;
        h_pending = false;
        tl_mark("h_arrived", st);
      }
      STEP_TRY(mpn_plan_node_tables(p, step, st));
      tl_mark("node_tables_end", st);
      STEP_TRY(mpn_plan_sweep(p, step, MPN_STAGE_EDGE, edge_attr, nullptr, nullptr, nullptr, st));
      tl_mark("edge_update_end", st);
      STEP_TRY(mpn_plan_sweep(p, step, MPN_STAGE_NODE, edge_attr, nullptr, nullptr, nullptr, st));
      tl_mark("node_moments_end", st);
      const bool cls = step >= first_class_step;
      const bool last = step == L;
      STEP_TRY(mpn_plan_sweep(p, step, MPN_STAGE_APPLY, edge_attr, cls ? logits_out + lstride * k : nullptr,
                              (cls && last) ? pred_out : nullptr, (cls && last) ? prob1_out : nullptr, st));
      if (cls) ++k;
      tl_mark("node_apply_end", st);
      const int grid = min(kNumSMs * 8, div_up((long long)g->n_nodes * 32, 256));
      if (!last) {
        mpn::launch(node_finalize_kernel<true>, grid, 256, 0, st, p->g, p->msg_task, p->h_full, P, abs_fix(p));
        mpn::launch(peer_publish_h_kernel, 1, 32, 0, st, P, ++seq_h);
        mpn::g_kernel_launches += 2;
        h_pending = true;
      } else {
        mpn::launch(node_finalize_kernel<false>, grid, 256, 0, st, p->g, p->msg_task, p->h_full, P, abs_fix(p));
        ++mpn::g_kernel_launches;
      }
      if (cudaGetLastError() != cudaSuccess) { set_error("node_finalize launch failed"); rc = MPN_ERR_CUDA; goto done; }
      tl_mark("node_finalize_end", st);
    }
  }
  if (h_out) {
    cudaError_t e = cudaMemcpyAsync(h_out, p->h_full + (size_t)g->row_offset * MPN_DH, sizeof(float) * (size_t)g->n_nodes * MPN_DH,
                                    cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { set_error("h copy failed: %s", cudaGetErrorString(e)); rc = MPN_ERR_CUDA; }
  }
#undef ENC0_STAGE
#undef PEER_FINALIZE
#undef STEP_TRY
done:
  mpn_plan_destroy(p);
  return rc;
}

int mpn_forward_sharded_x(const mpn_graph* g, const mpn_weights* w, const void* x, int32_t x_kind, const float* edge_attr, int32_t L,
                          int32_t n_cls, int64_t total_edges, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out,
                          int use_tc, const mpn_peer_ctx* peers, void* ws, size_t ws_bytes, void* stream) {
  return forward_sharded_impl(g, w, x, x_kind, const_cast<float*>(edge_attr), L, n_cls, total_edges, logits_out, h_out, pred_out,
                              prob1_out, use_tc, peers, ws, ws_bytes, nullptr, 0, stream);
}

int mpn_forward_sharded(const mpn_graph* g, const mpn_weights* w, const float* x, const float* edge_attr, int32_t L, int32_t n_cls,
                        int64_t total_edges, float* logits_out, float* h_out, uint8_t* pred_out, float* prob1_out, int use_tc,
                        const mpn_peer_ctx* peers, void* ws, size_t ws_bytes, void* stream) {
  return mpn_forward_sharded_x(g, w, x, MPN_X_F32, edge_attr, L, n_cls, total_edges, logits_out, h_out, pred_out, prob1_out, use_tc,
                               peers, ws, ws_bytes, stream);
}

int mpn_forward_sharded_with_edge_features_x(const mpn_graph* g, const mpn_weights* w, const void* x, int32_t x_kind,
                                             float* edge_attr_out, int32_t L, int32_t n_cls, int64_t total_edges, float* logits_out,
                                             float* h_out, uint8_t* pred_out, float* prob1_out, int use_tc, const mpn_peer_ctx* peers,
                                             void* ws, size_t ws_bytes, void* ef_ws, size_t ef_ws_bytes, void* stream) {
  MPN_REQUIRE(ef_ws != nullptr && edge_attr_out != nullptr, "forward_sharded_with_edge_features: NULL edge-feature buffer / workspace");
  return forward_sharded_impl(g, w, x, x_kind, edge_attr_out, L, n_cls, total_edges, logits_out, h_out, pred_out, prob1_out, use_tc,
                              peers, ws, ws_bytes, ef_ws, ef_ws_bytes, stream);
}

int mpn_forward_sharded_with_edge_features(const mpn_graph* g, const mpn_weights* w, const float* x, float* edge_attr_out, int32_t L,
                                           int32_t n_cls, int64_t total_edges, float* logits_out, float* h_out, uint8_t* pred_out,
                                           float* prob1_out, int use_tc, const mpn_peer_ctx* peers, void* ws, size_t ws_bytes,
                                           void* ef_ws, size_t ef_ws_bytes, void* stream) {
  return mpn_forward_sharded_with_edge_features_x(g, w, x, MPN_X_F32, edge_attr_out, L, n_cls, total_edges, logits_out, h_out, pred_out,
                                                  prob1_out, use_tc, peers, ws, ws_bytes, ef_ws, ef_ws_bytes, stream);
}

int mpn_pack_decisions(const uint8_t* pred, int64_t E, uint32_t* words_out, void* stream) {
  MPN_REQUIRE((pred && words_out) || E == 0, "pack_decisions: NULL argument");
  if (E == 0) return MPN_OK;
  const long long n_words = (E + 31) >> 5;
  mpn::launch(pack_decisions_kernel, (int)min((long long)kNumSMs * 8, (long long)div_up(n_words * 32, 256)), 256, 0, (cudaStream_t)stream, pred,
              (long long)E, words_out);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

int mpn_profile_timeline(int enable) {
  g_tl_on = enable != 0;
  g_tl_n = 0;
  return g_tl_on;
}

int mpn_profile_timeline_read(float* ms_out, char* names_out, int names_bytes) {

  if (g_tl_n == 0) return 0;
  for (int i = 0; i < g_tl_n; ++i)
    if (cudaEventSynchronize(g_tl_ev[i]) != cudaSuccess) return -1;
  int used = 0;
  for (int i = 0; i < g_tl_n; ++i) {
    float ms = 0.f;
    if (i > 0 && cudaEventElapsedTime(&ms, g_tl_ev[0], g_tl_ev[i]) != cudaSuccess) return -1;
    if (ms_out) ms_out[i] = ms;
    if (names_out) {
      const int len = (int)strlen(g_tl_name[i]);
      if (used + len + 2 > names_bytes) return -1;
      memcpy(names_out + used, g_tl_name[i], len);
      used += len;
      names_out[used++] = i + 1 < g_tl_n ? '|' : '\0';
    }
  }
  if (names_out && used == 0 && names_bytes > 0) names_out[0] = '\0';
  return g_tl_n;
}

int mpn_decide(const float* logits, int64_t E, uint8_t* pred, float* prob1, void* stream) {
  MPN_REQUIRE(logits || E == 0, "decide: NULL logits");
  if (E == 0) return MPN_OK;
  mpn::launch(decide_kernel, (int)min((long long)kNumSMs * 8, (long long)div_up(E, 256)), 256, 0, (cudaStream_t)stream, 
      (const float2*)logits, E, pred, prob1);
  MPN_LAUNCH_OK();
  return MPN_OK;
}

}  // extern "C"
