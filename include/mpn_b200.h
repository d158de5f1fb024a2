/*
 * mpn_b200.h — C ABI of the B200-native tracklet-graph message-passing path.
 *
 * Drop-in boundary for the reference's hot path.  The reference has no FFI layer (it is pure
 * Python on ATen / torch_scatter / networkx); each entry point below names the reference code it
 * replaces (paths relative to the upstream repository root).  The Python host in
 * graph-convolutional-network-for-multi-camera-vehicle-tracking_b200/ binds these with ctypes and
 * mirrors the reference classes/functions (MOTMPNet, post_processing, pruning, splitting, ...).
 *
 * Conventions
 *   - plain pointers and sizes only; every `dev` pointer is CUDA device memory owned by the caller;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it.  Functions documented as
 *     "synchronises" wait for the stream internally because they return host-side results;
 *   - workspaces are caller-allocated device memory; the *_workspace_bytes functions size them;
 *   - return value: 0 = ok, otherwise an MPN_ERR_* code; mpn_last_error() gives a thread-local message;
 *   - floating point is IEEE fp32 with fp64 accumulation of all BatchNorm moments; indices int32 on
 *     device (edge ids < 2^31 per shard), int64 accepted at the boundary as the reference delivers them.
 */
#ifndef MPN_B200_H
#define MPN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPN_B200_ABI_VERSION 6

enum {
  MPN_OK = 0,
  MPN_ERR_INVALID = 1,      /* bad argument / unsupported configuration */
  MPN_ERR_CUDA = 2,         /* a CUDA runtime call or kernel launch failed */
  MPN_ERR_UNSORTED = 3,     /* edge_index is not lexicographically (row, col) sorted */
  MPN_ERR_WORKSPACE = 4,    /* workspace too small */
  MPN_ERR_NO_DEVICE = 5     /* no sm_100 device / kernels not loadable */
};

/* fixed widths of the supported model family (config/config_training.yaml:68-111) */
#define MPN_DE 4            /* edge embedding width  (encoder edge_out_dim, edge_model fc_dims[-1]) */
#define MPN_DH 32           /* node embedding width  (encoder node_out_dim, node_model fc_dims[-1]) */
#define MPN_MAX_NODE_LAYERS 8

/* Threading contract: one host thread and one CUDA stream per device use the library at a time.  Work is enqueued on the caller's
 * stream (plus one library-owned side stream per device, forked from and joined to it with events); scratch memory is the
 * caller's (workspace arguments); the error string and the SPLITTING statistics are thread-local. */
int mpn_abi_version(void);
const char* mpn_last_error(void);
/* number of CUDA kernels this library has launched so far in this process (monotonic) */
uint64_t mpn_kernel_launches(void);
/* Programmatic dependent launch of the graph-build / edge-feature / forward kernels (on by default): the launch latency of
 * kernel n+1 overlaps the tail of kernel n (every kernel starts with griddepcontrol.wait, so results are bit-identical).
 * enable > 0 / == 0 switches it on / off (A/B measurements), enable < 0 only queries.  Returns 1 = off, 2 = on. */
int mpn_set_pdl(int enable);
/* 0 if device `dev` exists and is sm_100; error otherwise.  Never falls back to CPU. */
int mpn_check_device(int dev);

/* ------------------------------------------------------------------------------------------------
 * Graph tables (K0).  Replaces the implicit `row, col = edge_index` indexing of
 * models/mpn.py:44,82 and the tuple-list scans of utils.py:125-142 with an int32 CSR.
 * `edge_index` is the reference layout: int64 [2,E] row-major (row = edge_index[0], aggregated-at node).
 * Must be lexicographically sorted by (row, col) and free of duplicates — true for inference graphs
 * (inference.py:407-413); MPN_ERR_UNSORTED otherwise (the Python host then sorts and permutes).
 * A task is a run of <= `chunk` consecutive edges of one row; max_tasks = E / chunk + N.
 * ---------------------------------------------------------------------------------------------- */
typedef struct mpn_graph {
  int32_t n_nodes;          /* nodes whose rows this table holds (all nodes of the graph, or a row block) */
  int32_t n_cols;           /* size of the column (neighbour) id space: total nodes of the graph */
  int32_t row_offset;       /* global id of local row 0 (0 for an unsharded graph) */
  int32_t chunk;            /* edges per task (power of two, 32..4096) */
  int64_t n_edges;
  int32_t max_tasks;        /* capacity of task_row / task_beg */
  int32_t layout_hint;      /* MPN_LAYOUT_UNKNOWN, or MPN_LAYOUT_ONE_GAP when the builder of the tables vouches that every row lists
                             * all columns but one contiguous gap (mpn_graph_build_cross_camera sets it): mpn_edge_features then
                             * skips the launches of the Gram + gather path, which an unknown layout enqueues as the alternative */
  int32_t* rowptr;          /* dev [n_nodes+1]  */
  int32_t* col;             /* dev [n_edges]    global column ids */
  int32_t* taskptr;         /* dev [n_nodes+1]  first task of each row */
  int32_t* task_row;        /* dev [max_tasks]  local row of each task */
  int32_t* n_tasks;         /* dev [1]          */
  /* batched small graphs (block-diagonal edge set, nodes of a graph contiguous): BatchNorm statistics are taken
   * per graph, exactly as if each graph had been passed to the reference on its own (inference.py:375,469).
   * n_graphs <= 1 (or NULL pointers): one graph. */
  int32_t n_graphs;
  int32_t max_graph_nodes;  /* largest graph of the batch (sizes the block-diagonal Gram tiles) */
  int32_t* node_gid;        /* dev [n_nodes]     graph id of each node            */
  int32_t* graph_nptr;      /* dev [n_graphs+1]  first node of each graph         */
} mpn_graph;

enum { MPN_LAYOUT_UNKNOWN = 0, MPN_LAYOUT_ONE_GAP = 1 };
/* Fills the tables of `g` (pointers and sizes pre-set by the caller).  Synchronises (reads the sorted flag). */
int mpn_graph_build(mpn_graph* g, const int64_t* edge_index_dev, void* stream);
/* Same from int32 row/col arrays already split (used for row-block shards). */
int mpn_graph_build_i32(mpn_graph* g, const int32_t* row_dev, const int32_t* col_dev, void* stream);
/* Same tables without the host round trip: the validity flags (bit 0: not strictly (row,col)-sorted, bit 1: node id out of
 * range) are copied to *flags_host_pinned (page-locked host int) behind the scan and the call returns without synchronising;
 * an invalid edge list leaves an EMPTY graph on the device (no task, so later sweeps touch nothing).  The caller reads the
 * flag word after its next synchronisation of `stream`.  flags_dev: one device int of scratch that must stay alive until then. */
int mpn_graph_build_deferred(mpn_graph* g, const int64_t* edge_index_dev, int32_t* flags_dev, int32_t* flags_host_pinned,
                             void* stream);

/* Graph construction on the device (SURVEY.md section 8 row f1).  Replaces inference.py:407-414: for every camera
 * ascending, cartesian_prod(nodes in the camera, nodes not in it).  Nodes must be grouped by camera (dataset.py:279-281);
 * cam_ptr_host[k] = first node of camera k, cam_ptr_host[n_cams] = n_nodes (HOST array, n_cams <= 64).  Fills the tables
 * of `g` (g->n_edges must equal the number of cross-camera edges of its rows) directly from the camera layout: the int64 edge_index (16 B/edge) is
 * never read, and only written when edge_index_out_dev != NULL ([2,E] int64, reference layout).  Does not synchronise.
 * A row-block shard (g->row_offset, g->n_nodes inside g->n_cols nodes) builds just its own rows; its edge count is
 * mpn_cross_camera_block_edges(). */
#define MPN_MAX_CAMERAS 64
int64_t mpn_cross_camera_edges(const int32_t* cam_ptr_host, int32_t n_cams);
int64_t mpn_cross_camera_block_edges(const int32_t* cam_ptr_host, int32_t n_cams, int32_t row0, int32_t n_rows);
int mpn_graph_build_cross_camera(mpn_graph* g, const int32_t* cam_ptr_host, int32_t n_cams, int64_t* edge_index_out_dev,
                                 void* stream);
/* The same for a batch of graphs (inference.py:407-414 for every graph of the loop at inference.py:375): block-diagonal tables in
 * which row r of graph g = [gs, ge), camera segment [ss, se), lists the columns [gs, ss) and [se, ge) in ascending order.  The
 * layout is given by segments, one per (graph, camera): seg_ptr[s] = first node of segment s (seg_ptr[n_segs] = n_nodes), and
 * graph_seg[g] = first segment of graph g (graph_seg[n_graphs] = n_segs).  Camera ids need not be contiguous or shared by the
 * graphs; nodes are grouped by camera within each graph.
 *   mpn_cross_camera_batched_layout   HOST: validates the layout (segments and graphs non-empty, offsets from 0) and fills
 *                 seg_ebase_host[n_segs+1] (optional) with the first edge of each segment's row block; returns E, -1 if malformed.
 *   mpn_graph_build_cross_camera_batched   fills rowptr / col / taskptr / task_row / n_tasks and node_gid / graph_nptr of `g`
 *                 (g->n_graphs, g->max_graph_nodes and all table pointers set by the caller, g->n_edges = the layout's E, no row
 *                 block) from the SAME arrays in device memory (seg_ebase_dev from the helper above); edge_index_out_dev: optional
 *                 [2,E] int64, the per-graph reference edge_index offset by the graph's first node and concatenated.  Leaves
 *                 layout_hint = MPN_LAYOUT_UNKNOWN (a row does not span all columns).  Does not synchronise. */
int64_t mpn_cross_camera_batched_layout(const int32_t* seg_ptr_host, int32_t n_segs, const int32_t* graph_seg_host, int32_t n_graphs,
                                        int64_t* seg_ebase_host);
int mpn_graph_build_cross_camera_batched(mpn_graph* g, const int32_t* seg_ptr_dev, int32_t n_segs, const int32_t* graph_seg_dev,
                                         const int64_t* seg_ebase_dev, int64_t* edge_index_out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Edge features (K1).  Replaces inference.py:453-456:
 *   edge_attr[e] = [ ||x_r - x_c + 1e-6||_2 , 1 - cos(x_r, x_c) ]
 * computed from the Gram matrix X X^T of the centred features (fp32-accurate: three fp16-plane products on the tensor
 * cores, or the fp32 SIMT GEMM when `use_tensor_cores` is 0); the [E,D] gathers of the reference are never materialised.
 * Dense cross-camera graphs (every row = all columns but one contiguous gap, inference.py:407-413; checked on the device
 * unless g->layout_hint says so) with D % 64 == 0: ONE persistent tcgen05 kernel whose epilogue turns the TMEM accumulator
 * straight into edge_attr rows (csrc/gram_ef.cu) — no Gram matrix in HBM, no gather pass.  Any other graph: Gram block in
 * HBM + a gather pass.  x: dev [n_cols, D] fp32 row-major.  edge_attr: dev [E,2].
 * ---------------------------------------------------------------------------------------------- */
/* Measurement hook (bench.py): with enable != 0 every later mpn_edge_features call records a CUDA event on its stream before and
 * after the Gram GEMM + distance epilogue launch (csrc/gram_ef.cu); mpn_profile_gram_ms waits for the second event and returns
 * the duration of the last such launch in milliseconds (-1 if none).  Off by default: the events break the launch overlap. */
int mpn_profile_gram(int enable);
float mpn_profile_gram_ms(void);
/* Measurement hook (bench.py, tools/): while enabled, mpn_forward / mpn_forward_with_edge_features / mpn_forward_sharded* record a CUDA
 * event at every phase boundary of the caller's stream (edge features + first BatchNorm, second encoder sweep, join with the
 * side-stream node encoder, arrival of the peers' rows, node tables, the three sweeps of every step, node finalize) and one at the
 * end of the side-stream encoder.  mpn_profile_timeline_read waits for the last forward's events and returns their number n;
 * ms_out[i] = time from the first event to event i, names_out = the n names joined by '|'.  Off by default: an event between
 * two kernels ends their programmatic overlap.  Not thread safe. */
/* Tests / bench: how the last mpn_forward_sharded_with_edge_features that used `ef_workspace_dev` computed the edge features
 * (synchronises the stream): 2 = shared symmetric Gram (mpn_peer_ctx.edge_attr), 0 = every rank its own rows, -1 = error. */
int mpn_shared_gram_mode(const mpn_graph* g, int32_t feature_dim, const void* ef_workspace_dev, size_t ef_workspace_bytes, void* stream);
/* Tests: the pair-ownership rule of the shared Gram exactly as the kernels evaluate it.  Rows [out[0], out[1]) (global node ids,
 * intersected with rank's own block by the caller) of rank `rank` compute their pair with column c; returns the owner rank of
 * node c, or -1 on bad arguments.  Host only. */
int mpn_shared_gram_row_range(int32_t rank, int32_t world, const int32_t* block_start, int32_t c, int32_t* out_host);
int mpn_profile_timeline(int enable);
int mpn_profile_timeline_read(float* ms_out, char* names_out, int names_bytes);
size_t mpn_edge_features_workspace_bytes(const mpn_graph* g, int32_t D);
int mpn_edge_features(const mpn_graph* g, const float* x_dev, int32_t D, float* edge_attr_dev,
                      int use_tensor_cores, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * MPN weights.  Same tensors, names and shapes as the reference state_dict (models/mpn.py:166-247,
 * models/mlp.py:11-30); `small` is one packed fp32 block (offsets below) so the sweeps stage it once.
 * ---------------------------------------------------------------------------------------------- */
enum {                                   /* offsets (in floats) inside mpn_weights.small */
  MPN_W_ENC1_W = 0,                      /* encoder.edge_mlp.fc_layers.0.weight [4,2]  */
  MPN_W_ENC1_B = 8,                      /* ...0.bias [4] */
  MPN_W_ENC1_G = 12,                     /* ...1.weight (BN gamma) [4] */
  MPN_W_ENC1_BETA = 16,                  /* ...1.bias   (BN beta)  [4] */
  MPN_W_ENC2_W = 20,                     /* encoder.edge_mlp.fc_layers.4.weight [4,4]  */
  MPN_W_ENC2_B = 36,
  MPN_W_ENC2_G = 40,
  MPN_W_ENC2_BETA = 44,
  MPN_W_EDGE_W = 48,                     /* MPNet.edge_model.edge_mlp.fc_layers.0.weight [4,68] = [h_row|h_col|e] */
  MPN_W_EDGE_B = 320,
  MPN_W_EDGE_G = 324,
  MPN_W_EDGE_BETA = 328,
  MPN_W_NODE_W = 332,                    /* MPNet.node_model.node_mlp.fc_layers.0.weight [32,36] = [h_row|e] */
  MPN_W_NODE_B = 1484,
  MPN_W_NODE_G = 1516,
  MPN_W_NODE_BETA = 1548,
  MPN_W_CLS_W = 1580,                    /* classifier.edge_mlp.fc_layers.0.weight [2,4] */
  MPN_W_CLS_B = 1588,
  /* reattach_initial_nodes / reattach_initial_edges (models/mpn.py:207-215, 283-287): the columns of the two MPNet weights
   * that multiply the INITIAL encodings, split off by the host; all zero when the option is off.
   *   EDGE_W0 [4,68]  = [h0_row | h0_col | e0]   (the [4,68] block above then holds [h_row | h_col | e])
   *   NODE_W0 [32,32] = [h0_row]                 (the [32,36] block above holds [h_row | e]) */
  MPN_W_EDGE_W0 = 1592,
  MPN_W_NODE_W0 = 1864,
  MPN_W_SMALL_FLOATS = 2888
};

typedef struct mpn_weights {
  int32_t n_node_layers;                          /* encoder.node_mlp: number of Linear+BN+ReLU blocks */
  int32_t node_dims[MPN_MAX_NODE_LAYERS + 1];     /* in, hidden..., out (out must equal MPN_DH) */
  const float* node_w[MPN_MAX_NODE_LAYERS];       /* dev [out,in] row-major (nn.Linear.weight) */
  const float* node_b[MPN_MAX_NODE_LAYERS];       /* dev [out] */
  const float* node_gamma[MPN_MAX_NODE_LAYERS];   /* dev [out] BatchNorm weight */
  const float* node_beta[MPN_MAX_NODE_LAYERS];    /* dev [out] BatchNorm bias */
  const float* small;                             /* dev [MPN_W_SMALL_FLOATS] */
  /* optional cache: TF32 hi/lo planes of node_w[i] made by mpn_split_tf32 (NULL -> split on every forward) */
  const float* node_w_hi[MPN_MAX_NODE_LAYERS];
  const float* node_w_lo[MPN_MAX_NODE_LAYERS];
  /* optional cache: fp16 planes of node_w[i] * node_w_scale16[i] made by mpn_split_f16 ("3xFP16" GEMM, used when K % 8 == 0),
   * and max|gamma|, max|beta| of the layer's BatchNorm (bound of the next layer's input: |relu(BN(y))| <= bmax + gmax*sqrt(M-1)) */
  const void* node_w_hi16[MPN_MAX_NODE_LAYERS];
  const void* node_w_lo16[MPN_MAX_NODE_LAYERS];
  float node_w_scale16[MPN_MAX_NODE_LAYERS];
  float node_bn_gmax[MPN_MAX_NODE_LAYERS];
  float node_bn_bmax[MPN_MAX_NODE_LAYERS];
  /* node aggregation of the messages (models/mpn.py:193-202): scatter_add / scatter_mean / scatter_max over row */
  int32_t node_agg;                               /* MPN_AGG_SUM (shipped config) | MPN_AGG_MEAN | MPN_AGG_MAX */
  int32_t reattach_nodes;                         /* reattach_initial_nodes: h_in = [h0 | h] before every step */
  int32_t reattach_edges;                         /* reattach_initial_edges: e_in = [e0 | e] before every step */
  int32_t reserved;
} mpn_weights;
enum { MPN_AGG_SUM = 0, MPN_AGG_MEAN = 1, MPN_AGG_MAX = 2 };

/* x = hi + lo with hi = rna_tf32(x), lo = rna_tf32(x - hi): the operand planes of the 3xTF32 tensor-core GEMM.
 * n must be a multiple of 4, pointers 16-byte aligned. */
int mpn_split_tf32(const float* x_dev, int64_t n, float* hi_dev, float* lo_dev, void* stream);
/* x * s = hi + lo in fp16 with s = the power of two that puts amax (= max |x|, given by the caller) in [2^13, 2^14);
 * *scale_out_host receives s.  hi/lo: dev fp16 [n]. */
int mpn_split_f16(const float* x_dev, int64_t n, float amax, void* hi_dev, void* lo_dev, float* scale_out_host, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Forward (K1b-K4).  Replaces MOTMPNet.forward (models/mpn.py:250-299) for the supported family:
 * encoder (MLPGraphIndependent, mpn.py:128-142), `num_enc_steps` x MetaLayer (mpn.py:32-54: EdgeModel
 * mpn.py:67-69, NodeModel mpn.py:97-99 with scatter_add mpn.py:202) and the edge classifier on the last
 * `num_class_steps` steps (mpn.py:277,290-297).  BatchNorm uses batch statistics (models/mlp.py:16).
 *   x          dev [n_cols, node_dims[0]]
 *   edge_attr  dev [E,2]
 *   logits_out dev [n_out, E, 2], n_out = max(num_class_steps,1) if L==0 else num_class_steps
 *   h_out      dev [n_nodes, 32]   latent node features after the last step
 *   pred_out   dev [E] uint8 or NULL: argmax of the LAST logits (ties -> 0)      (inference.py:479)
 *   prob1_out  dev [E] fp32  or NULL: softmax(last logits)[:,1]                  (inference.py:475-477)
 * ---------------------------------------------------------------------------------------------- */
size_t mpn_forward_workspace_bytes(const mpn_graph* g, const mpn_weights* w, int32_t num_enc_steps);
int mpn_forward(const mpn_graph* g, const mpn_weights* w, const float* x_dev, const float* edge_attr_dev,
                int32_t num_enc_steps, int32_t num_class_steps, float* logits_out_dev, float* h_out_dev,
                uint8_t* pred_out_dev, float* prob1_out_dev, int use_tensor_cores,
                void* workspace_dev, size_t workspace_bytes, void* stream);

/* K1 + forward in one call: edge_attr_out (dev [E,2]) is PRODUCED here by mpn_edge_features (inference.py:453-456) on `stream`
 * while the node encoder runs on a side stream — the two only share the read-only x, so the encoder's GEMM chain hides behind the
 * Gram GEMM and the feature epilogue.  ef_workspace: mpn_edge_features_workspace_bytes(g, node_dims[0]).  Unsharded graphs. */
int mpn_forward_with_edge_features(const mpn_graph* g, const mpn_weights* w, const float* x_dev, float* edge_attr_out_dev,
                                   int32_t num_enc_steps, int32_t num_class_steps, float* logits_out_dev, float* h_out_dev,
                                   uint8_t* pred_out_dev, float* prob1_out_dev, int use_tensor_cores, void* workspace_dev,
                                   size_t workspace_bytes, void* ef_workspace_dev, size_t ef_workspace_bytes, void* stream);

/* Phase-level entry points of the same forward, for row-block sharded execution where the host inserts
 * the collectives (all-reduce of BatchNorm moment sums, all-gather of h) between phases.  See DESIGN.md. */
typedef struct mpn_fwd_plan mpn_fwd_plan;       /* opaque; lives inside the caller's workspace */
enum { MPN_SUMS_DOUBLES = 96 };                 /* size of the moment-sum vector exchanged between ranks */
enum {                                          /* sweep / stage ids */
  MPN_STAGE_ENC0 = 0,     /* moments of edge_attr                      -> BN of encoder layer 1 */
  MPN_STAGE_ENC1 = 1,     /* moments of encoder layer 2 pre-activation -> BN of encoder layer 2 */
  MPN_STAGE_EDGE = 2,     /* moments of the edge-update pre-activation y -> BN of edge model     */
  MPN_STAGE_NODE = 3,     /* moments of the node-update pre-activation z -> BN of node model     */
  MPN_STAGE_APPLY = 4     /* apply: messages, segment sum, logits, decisions                     */
};
int mpn_plan_create(mpn_fwd_plan** plan_out, const mpn_graph* g, const mpn_weights* w, int32_t num_enc_steps,
                    int32_t num_class_steps, int64_t total_edges, int use_tensor_cores,
                    void* workspace_dev, size_t workspace_bytes);
void mpn_plan_destroy(mpn_fwd_plan* plan);
/* node encoder over all n_cols nodes (replicated on every rank); h0 -> plan-internal buffer [n_cols,32] */
int mpn_plan_node_encoder(mpn_fwd_plan* plan, const float* x_dev, void* stream);
/* per-step node tables from the plan's full h buffer (after the host has all-gathered it) */
int mpn_plan_node_tables(mpn_fwd_plan* plan, int32_t step, void* stream);
/* run the sweep of `stage` for `step` (1-based); leaves local moment sums in plan sums buffer */
int mpn_plan_sweep(mpn_fwd_plan* plan, int32_t step, int32_t stage, const float* edge_attr_dev,
                   float* logits_out_dev, uint8_t* pred_out_dev, float* prob1_out_dev, void* stream);
/* device pointer to the MPN_SUMS_DOUBLES fp64 sums of the last sweep (all-reduce this across ranks) */
double* mpn_plan_sums(mpn_fwd_plan* plan);
/* reduce this rank's block partials of the last sweep into the sums vector (fixed order); with_consts != 0
 * also folds the constants right away (single-GPU shortcut for reduce + finalize) */
int mpn_plan_reduce(mpn_fwd_plan* plan, int32_t stage, int with_consts, void* stream);
/* turn (all-reduced) sums into folded BatchNorm constants for the next sweep */
int mpn_plan_finalize(mpn_fwd_plan* plan, int32_t step, int32_t stage, void* stream);
/* after MPN_STAGE_APPLY: reduce task partials into h rows of this shard; returns device pointers */
int mpn_plan_node_finalize(mpn_fwd_plan* plan, int32_t step, void* stream);
float* mpn_plan_h_full(mpn_fwd_plan* plan);     /* dev [n_cols,32]: row block [row_offset, +n_nodes) is this rank's */

/* ------------------------------------------------------------------------------------------------
 * Sharded forward with the collectives fused into the kernels over NVLink peer memory (one launch sequence per rank,
 * no host round trips): every BatchNorm's moment all-reduce happens inside the finalize kernel (each rank publishes its
 * 96 fp64 sums in a peer-mapped slot, raises a sequence flag with st.release.sys, then adds all ranks' slots in rank
 * order — bit-identical totals on every rank), and for L > 1 the node-finalize kernel stores its rows of h straight into
 * every peer's h buffer (the all-gather).  `sums[r]`, `flags[r]`, `h[r]` are rank r's buffers as mapped into THIS
 * process (e.g. torch.distributed._symmetric_memory); layout per rank: sums = 2 slots x MPN_MAX_PEERS rows x 96 doubles (row s of
 * a slot is WRITTEN BY rank s: the exchange pushes, every rank polls and reads only its own memory), flags = 3 x MPN_MAX_PEERS
 * uint64 (word [0][s]: moment sequence raised by rank s, [1][s]: h sequence raised by rank s, [2][0]: this rank's column-stat
 * sequence; zero-initialised, monotonic across calls), h = [n_cols,32] fp32,
 * cstats = 2 slots x MPN_PEER_CSTAT_COLS x 2 doubles.  With shard_node_encoder != 0 every rank encodes only its own row
 * block of x: the per-column BatchNorm sums of each encoder layer are all-reduced through `cstats` inside a kernel and
 * the encoded rows are stored into every peer's h buffer (needs h != NULL and encoder widths <= MPN_PEER_CSTAT_COLS).
 * total_edges <= 0: the edge count of the whole graph is summed on the device with the first moment all-reduce.
 * All ranks must call with the same sequence numbers; the call consumes 2+2L moment numbers, L-1 (+1 with a sharded
 * encoder) h numbers and, with a sharded encoder, one column-stat number per encoder layer.
 * Every wait traps after 10 s instead of hanging the GPU.
 * ---------------------------------------------------------------------------------------------- */
#define MPN_MAX_PEERS 16
typedef struct mpn_peer_ctx {
  int32_t rank, world;
  double* sums[MPN_MAX_PEERS];
  uint64_t* flags[MPN_MAX_PEERS];
  float* h[MPN_MAX_PEERS];
  double* cstats[MPN_MAX_PEERS];
  uint64_t seq_moments;     /* last moment sequence number already used (this call uses seq_moments+1 ...) */
  uint64_t seq_h;           /* last h sequence number already used */
  uint64_t seq_c;           /* last column-stat sequence number already used */
  int32_t shard_node_encoder;
  int32_t reserved;
  /* Shared symmetric Gram of mpn_forward_sharded_with_edge_features (optional: edge_attr[0] == NULL -> every rank computes all
   * pairs of its own rows).  edge_attr[r]: rank r's peer-visible edge_attr buffer ([E_r,2] fp32; edge_attr[rank] must be the
   * edge_attr_out_dev of the call); node_tables[r]: rank r's peer-visible [n_cols][4] int32 table (filled by the call);
   * block_start: rank r owns nodes [block_start[r], block_start[r+1]).  Every unordered pair of nodes is then computed by one
   * rank only, which stores the mirrored entry into the owner's edge_attr over NVLink (csrc/kernels.h GeShare for the rule);
   * flag word [3][src] of `flags` carries seq_t.  If any rank's rows are not dense cross-camera rows, all ranks fall back. */
  float* edge_attr[MPN_MAX_PEERS];
  int32_t* node_tables[MPN_MAX_PEERS];
  int32_t block_start[MPN_MAX_PEERS + 1];
  int32_t reserved2;
  uint64_t seq_t;           /* last node-table sequence number already used */
} mpn_peer_ctx;
#define MPN_PEER_CSTAT_COLS 1024
int mpn_forward_sharded(const mpn_graph* g, const mpn_weights* w, const float* x_dev, const float* edge_attr_dev,
                        int32_t num_enc_steps, int32_t num_class_steps, int64_t total_edges, float* logits_out_dev,
                        float* h_out_dev /* [g->n_nodes,32] local rows */, uint8_t* pred_out_dev, float* prob1_out_dev,
                        int use_tensor_cores, const mpn_peer_ctx* peers, void* workspace_dev, size_t workspace_bytes, void* stream);
/* K1 + the sharded forward in one call (the row-block variant of mpn_forward_with_edge_features): edge_attr_out_dev [E_local,2] is
 * PRODUCED here by the fused edge-feature kernel (this rank's rows of the Gram matrix) on `stream` while the node encoder runs on
 * the side stream; the first encoder BatchNorm's moment sums come from that kernel's epilogue (no sweep over edge_attr), the
 * ranks' sums still meet in the same peer-memory exchange.  ef_workspace: mpn_edge_features_workspace_bytes(g, node_dims[0]). */
int mpn_forward_sharded_with_edge_features(const mpn_graph* g, const mpn_weights* w, const float* x_dev, float* edge_attr_out_dev,
                                           int32_t num_enc_steps, int32_t num_class_steps, int64_t total_edges, float* logits_out_dev,
                                           float* h_out_dev, uint8_t* pred_out_dev, float* prob1_out_dev, int use_tensor_cores,
                                           const mpn_peer_ctx* peers, void* workspace_dev, size_t workspace_bytes,
                                           void* ef_workspace_dev, size_t ef_workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decisions.  Replaces inference.py:475-479 when the caller owns the logits.
 * ---------------------------------------------------------------------------------------------- */
int mpn_decide(const float* logits_dev, int64_t n_edges, uint8_t* pred_out_dev, float* prob1_out_dev, void* stream);
/* The decisions (inference.py:479) as a bit mask for the trip to the host: bit (e & 31) of words_out_dev[e >> 5] = pred[e] != 0,
 * ceil(n_edges / 32) uint32 words (bytes in np.unpackbits(..., bitorder="little") order); 1/8 of the D2H bytes of pred. */
int mpn_pack_decisions(const uint8_t* pred_dev, int64_t n_edges, uint32_t* words_out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Post-processing (K5).  `act` is dev uint8 [E] (1 = active edge), updated in place; `prob1` dev fp32
 * with element stride `prob_stride` (2 when pointing at column 1 of the caller's [E,2] softmax).
 * All of these synchronise the stream (they iterate to a fixed point with host-visible flags).
 *   mpn_cut     remove_edges_single_direction      utils.py:125-142
 *   mpn_prune   pruning                            utils.py:144-339 (live 161-188,277-317); *changed_host = 0
 *               is the reference's "return []" case
 *   mpn_split   splitting                          utils.py:54-123.  Exact under probability ties: when no value that an
 *               oversized cluster can drop is shared with a second active edge, all oversized clusters drop their minimum in
 *               the same round on the device (the clusters are independent); otherwise the weakly connected components that
 *               SPLITTING can touch go through the reference's own one-cluster-at-a-time order (mpn_split_exact_host).
 *               mpn_split_last_stats reports which of the two ran.
 *   mpn_scc_labels  partition of compute_SCC_and_Clusters (utils.py:30-52); labels_dev[n] = smallest node
 *               id of n's strongly connected component ("canonical" numbering)
 *   mpn_post_processing  inference.post_processing inference.py:70-169 (CUT, PRUNE, CUT, SPLIT)
 * ---------------------------------------------------------------------------------------------- */
enum { MPN_POST_CUT = 1, MPN_POST_PRUNE = 2, MPN_POST_SPLIT = 4 };
size_t mpn_post_workspace_bytes(const mpn_graph* g);
int mpn_cut(const mpn_graph* g, uint8_t* act_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_prune(const mpn_graph* g, uint8_t* act_dev, const float* prob1_dev, int32_t prob_stride, int32_t num_cameras,
              int32_t* changed_host, int32_t* rounds_host, void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_split(const mpn_graph* g, uint8_t* act_dev, const float* prob1_dev, int32_t prob_stride, int32_t num_cameras,
              int32_t* rounds_host, void* workspace_dev, size_t workspace_bytes, void* stream);
/* SPLITTING of the calling thread's last mpn_split / mpn_post_processing: out[0] = active edges carrying a probability value
 * that is tied with an edge touching an oversized cluster (-1: not counted, every active edge went to the host),
 * out[1] = rounds (device) or dropped values (host order), out[2] = host-order steps taken on a label other than the lowest
 * oversized one (utils.py:112), out[3] = 0 device rounds | 1 reference order on the host.  After mpn_post_processing_batched:
 * out[0] and out[2] summed over the graphs, out[1] = device rounds + the dropped values of the host-order graphs, out[3] = the
 * number of graphs that took the reference order on the host. */
void mpn_split_last_stats(int64_t out_host[4]);
int mpn_scc_labels(const mpn_graph* g, const uint8_t* act_dev, int32_t* labels_dev, int32_t* n_components_host,
                   void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_post_processing(const mpn_graph* g, uint8_t* act_dev, const float* prob1_dev, int32_t prob_stride,
                        int32_t num_cameras, int32_t flags, int32_t* labels_dev, int32_t* n_components_host,
                        int32_t* prune_changed_host, void* workspace_dev, size_t workspace_bytes, void* stream);
/* inference.post_processing (inference.py:70-169, utils.py:30-52, 54-123, 125-142, 144-339) for EACH graph of a batched graph
 * (n_graphs > 1, node_gid / graph_nptr set) in one call, with the result a single-graph mpn_post_processing gives on every graph
 * alone.  num_cameras_dev: dev int32 [n_graphs], the camera count of each graph (PRUNE bounds degrees by num_cameras[g] - 1,
 * SPLIT cluster sizes by num_cameras[g]).  SPLITTING removes the edges of THE SAME graph whose probability equals a dropped
 * minimum (utils.py:96-98): its sets are keyed by (graph, value), and the mode (device rounds / reference order on the host) is
 * chosen per graph; mpn_split_last_stats then sums the counts over the graphs and out[3] is the number of graphs that took the
 * reference order.  labels_dev (optional): dev int32 [n_nodes], canonical graph-local labels (smallest node id of the SCC minus
 * the graph's first node); n_components_host: HOST int32 [n_graphs].  n_graphs <= 1: same as mpn_post_processing with
 * num_cameras_dev[0].  The workspace is mpn_post_workspace_bytes(g): the single-graph layout (whose SPLIT sets already hold
 * (graph, value) keys) plus three int32 per graph.  Synchronises. */
int mpn_post_processing_batched(const mpn_graph* g, uint8_t* act_dev, const float* prob1_dev, int32_t prob_stride,
                                const int32_t* num_cameras_dev, int32_t flags, int32_t* labels_dev, int32_t* n_components_host,
                                void* workspace_dev, size_t workspace_bytes, void* stream);
/* Active edges in edge order as (src, dst) int32 pairs, for the reference label numbering.
 * n_active_host receives the count; src_out/dst_out dev [capacity].  Synchronises. */
int mpn_active_edges(const mpn_graph* g, const uint8_t* act_dev, int32_t* src_out_dev, int32_t* dst_out_dev,
                     int64_t capacity, int64_t* n_active_host, void* workspace_dev, size_t workspace_bytes, void* stream);
/* Row-block sharded post-processing (new; the reference is single-GPU).  Only ACTIVE edges take part in any stage of
 * inference.post_processing (inference.py:93-166: CUT looks for an active reverse edge, PRUNE / SPLIT pick among active edges, the
 * labels are the SCCs of the active digraph), so a shard only has to contribute the order-preserving compaction of its own active
 * edges: the E-sized sweep stays sharded, the ranks exchange A << E entries once, and the fixed-point rounds run on the merged
 * active list (concatenated in rank order = global edge order, which keeps torch.argmin's lowest-edge-id tie rule).
 *   mpn_count_active     number of active edges of this shard (row-block graphs allowed); leaves the block offsets in the workspace
 *   mpn_compact_active   must follow mpn_count_active on the same workspace / stream with `act` unchanged: writes, in edge order,
 *                        src (GLOBAL row id = row_offset + local row), dst (global), the shard-local edge id and prob1 of every
 *                        active edge; outputs dev [n_active]
 *   mpn_clear_inactive   act[eid[i]] = 0 where keep[i] == 0 (the shard applies the merged result to its own decisions)
 * mpn_count_active synchronises the stream (the count is returned to the host); the other two do not. */
size_t mpn_compact_workspace_bytes(const mpn_graph* g);
int mpn_count_active(const mpn_graph* g, const uint8_t* act_dev, int64_t* n_active_host, void* workspace_dev,
                     size_t workspace_bytes, void* stream);
int mpn_compact_active(const mpn_graph* g, const uint8_t* act_dev, const float* prob1_dev, int32_t prob_stride,
                       int32_t* src_out_dev, int32_t* dst_out_dev, int32_t* eid_out_dev, float* prob_out_dev,
                       void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_clear_inactive(uint8_t* act_dev, const int32_t* eid_dev, const uint8_t* keep_dev, int64_t n, void* stream);
/* Host-side (CPU, sequential by nature): label integers exactly as compute_SCC_and_Clusters (utils.py:30-52)
 * assigns them — networkx SCC emission order, stable sort by size, isolated nodes last.  HOST pointers. */
/* ID_pred exactly as compute_SCC_and_Clusters numbers it (utils.py:30-52) for the activity flags `act_dev` of a (row, col)-sorted
 * graph: SCC partition and first-appearance keys on the device, the rank of (size, emission key) on the host over the
 * COMPONENTS (not the edges); only the components that one-directional edges tie together go through a sequential generator.
 * labels_out_host: HOST int64 [n_nodes].  Synchronises. */
int mpn_labels_reference(const mpn_graph* g, const uint8_t* act_dev, int64_t* labels_out_host, int32_t* n_components_host,
                         void* workspace_dev, size_t workspace_bytes, void* stream);
/* The same numbering (utils.py:30-52) for each graph of a batched (row, col)-sorted graph: labels_out_host HOST int64 [n_nodes]
 * numbered from 0 within every graph, exactly as mpn_labels_reference numbers that graph alone; n_components_host HOST int32
 * [n_graphs].  n_graphs <= 1: same as mpn_labels_reference.  Synchronises. */
int mpn_labels_reference_batched(const mpn_graph* g, const uint8_t* act_dev, int64_t* labels_out_host, int32_t* n_components_host,
                                 void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_labels_reference_host(const int32_t* src_host, const int32_t* dst_host, int64_t n_active, int32_t n_nodes,
                              int64_t* labels_out_host, int32_t* n_components_host);
/* Host-side SPLITTING in the reference's own order (utils.py:54-123): one oversized cluster at a time — the lowest label of the
 * reference numbering, the integer label re-read after every relabel as utils.py:112 does — dropping every active edge whose
 * probability equals (float ==, utils.py:96-98) the minimum among the active edges touching that cluster.  A step recomputes only
 * the weakly connected components it touched (csrc/split_exact.cu), not the whole graph as the reference does.  Input: active
 * edges in edge order with their probabilities — all of them, or the weakly connected components that SPLITTING can touch
 * (mpn_split gathers those: oversized clusters and probability ties).  Output keep_out[i] = 0 for the edges switched off;
 * stats_out[4] (optional): dropped values, steps taken on a label other than the lowest oversized one, clusters examined, 0.
 * HOST pointers. */
int mpn_split_exact_host(const int32_t* src_host, const int32_t* dst_host, const float* prob_host, int64_t n_active,
                         int32_t n_nodes, int32_t num_cameras, uint8_t* keep_out_host, int64_t* stats_out);

/* ------------------------------------------------------------------------------------------------
 * GEMM building block (exported for tests and for the roofline bench):
 *   C[M,N] = A[M,K] * B[N,K]^T (+ bias[N]), fp32 in / fp32 out, row-major, "NT".
 *   impl: 0 = fp32 SIMT, 1 = tcgen05 3xTF32 (TMA + TMEM).
 * ---------------------------------------------------------------------------------------------- */
size_t mpn_gemm_nt_workspace_bytes(int32_t M, int32_t N, int32_t K, int impl);
int mpn_gemm_nt(const float* A_dev, const float* B_dev, const float* bias_dev, float* C_dev,
                int32_t M, int32_t N, int32_t K, int impl, void* workspace_dev, size_t workspace_bytes, void* stream);
/* The Gram block the edge features use (inference.py:453-456 as one GEMM): C[M,N] = X[row0:row0+M] X^T, X [N,K] fp32.
 * amax_dev: device float = max |X| -> "3xFP16" operand planes (x * 2^k = hi + lo in fp16, three kind::f16 products, fp32
 * accumulate; K % 8 == 0); NULL -> 3xTF32.  Workspace: mpn_gemm_nt_workspace_bytes(M, N, K, 1). */
int mpn_gram_nt(const float* X_dev, int32_t row0, float* C_dev, int32_t M, int32_t N, int32_t K, const float* amax_dev,
                void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * After the hot path (SURVEY.md section 8f rows 2-3): evaluation counts and the tracking output.
 *   mpn_edge_confusion   compute_P_R_F (inference.py:20-66): counts_dev int64 [3][3] = label class x prediction class,
 *                        class = 0 / 1 / 2 for a value == 0 / == 1 / anything else (the reference only ever tests == 0 and == 1).
 *                        *_kind: 0 = uint8, 1 = int64, 2 = float32 element type.
 *   mpn_contingency      contingency table of two COMPACT labelings (labels in [0,Ka) x [0,Kb)), the input of every clustering
 *                        score the reference takes from sklearn.metrics on (ID_GT, ID_pred) (inference.py:507-519): COO entries in
 *                        arbitrary order (sort on the host), the number of non-zeros and both marginals.  Synchronises.
 *   mpn_expected_mutual_information_host   the EMI term of adjusted_mutual_info_score (scikit-learn 0.24.2
 *                        _expected_mutual_info_fast.pyx, env_gnn.yml:107) from the two marginals.  HOST pointers, CPU.
 *   mpn_relabel_detections   inference.py:540-548: out_id[r] = node_new[n] for the last tracklet n whose (id_cam, old id) equals the
 *                        detection's, else the detection keeps its id.  id_cam in [0,2^20), ids in [0,2^44).  Synchronises.
 *   mpn_write_mtmc_txt_host  np.savetxt(..., fmt='%d') of main.py:114 for an int64 table.  HOST pointers, CPU.
 * ---------------------------------------------------------------------------------------------- */
int mpn_edge_confusion(const void* pred_dev, int pred_kind, const void* labels_dev, int label_kind, int64_t n_edges,
                       int64_t* counts_dev /* [9] */, void* stream);
size_t mpn_contingency_workspace_bytes(int64_t n);
int mpn_contingency(const int64_t* a_dev, const int64_t* b_dev, int64_t n, int64_t Ka, int64_t Kb, int64_t* rows_out_dev,
                    int64_t* cols_out_dev, int64_t* counts_out_dev, int64_t* nnz_host, int64_t* row_sums_dev /* [Ka] */,
                    int64_t* col_sums_dev /* [Kb] */, void* workspace_dev, size_t workspace_bytes, void* stream);
double mpn_expected_mutual_information_host(const int64_t* row_sums_host, int64_t R, const int64_t* col_sums_host, int64_t C,
                                            int64_t n_samples);
size_t mpn_relabel_workspace_bytes(int64_t n_tracklets);
int mpn_relabel_detections(const int64_t* det_cam_dev, const int64_t* det_id_dev, int64_t n_detections, const int64_t* node_cam_dev,
                           const int64_t* node_old_id_dev, const int64_t* node_new_id_dev, int64_t n_tracklets,
                           int64_t* out_id_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_write_mtmc_txt_host(const char* path, const int64_t* table_host, int64_t rows, int32_t cols);

/* ------------------------------------------------------------------------------------------------
 * Before the hot path (SURVEY.md section 8f rows 1 and 4): what inference.py:383-451 still does per graph.
 *   mpn_edge_labels         edge_labels_g (inference.py:446-450): out[e] = 1.0f if node_labels[row[e]] == node_labels[col[e]]
 *                           else 0.0f, in the graph's edge order; node_labels_dev int64 [n_cols].
 *   mpn_normalize_columns   F.normalize(node_embeds, p=2, dim=0) (inference.py:403-404): out[i,j] = x[i,j] / max(||x[:,j]||_2, 1e-12);
 *                           out may alias x.
 *   mpn_normalize_columns_batched   the same for every graph of a batch alone (inference.py:403-404 inside the loop over graphs,
 *                           inference.py:375): rows [graph_nptr[g], graph_nptr[g+1]) are scaled by their own column norms.  fp64 sums
 *                           in a fixed order (deterministic), no workspace for n_graphs > 1; out may alias x.  n_graphs <= 1 is
 *                           mpn_normalize_columns with the workspace given (graph_nptr_dev unused); for n_graphs > 1 the workspace
 *                           arguments are unused and may be NULL / 0.
 * ---------------------------------------------------------------------------------------------- */
int mpn_edge_labels(const mpn_graph* g, const int64_t* node_labels_dev, float* out_dev, void* stream);
size_t mpn_normalize_columns_workspace_bytes(int32_t D);
int mpn_normalize_columns(const float* x_dev, int32_t n, int32_t D, float* out_dev, void* workspace_dev, size_t workspace_bytes,
                          void* stream);
int mpn_normalize_columns_batched(const float* x_dev, int32_t n, int32_t D, const int32_t* graph_nptr_dev, int32_t n_graphs,
                                  float* out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Half-width node features.  Every entry point that reads the node features x has an `_x` twin that takes
 * `const void* x_dev, int32_t x_kind` in place of `const float* x_dev` and is otherwise identical (the fp32 entry points are
 * these twins called with MPN_X_F32).  The kernels that read x convert each element to fp32 on load (exact for fp16 and bf16)
 * and keep every reduction's order, so each output is bit-identical to the same call on the fp32 copy of x; no such copy is
 * made.  The outputs stay fp32 (mpn_normalize_columns_x writes fp32 out_dev, which then cannot alias a 16-bit x).  An unknown
 * x_kind returns MPN_ERR_INVALID.  Half-precision features are the caller's choice: they are exact inputs, but not the
 * fp32 embeddings they were rounded from.
 * ---------------------------------------------------------------------------------------------- */
#define MPN_X_F32 0
#define MPN_X_F16 1
#define MPN_X_BF16 2
int mpn_edge_features_x(const mpn_graph* g, const void* x_dev, int32_t x_kind, int32_t D, float* edge_attr_dev,
                        int use_tensor_cores, void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_forward_x(const mpn_graph* g, const mpn_weights* w, const void* x_dev, int32_t x_kind, const float* edge_attr_dev,
                  int32_t num_enc_steps, int32_t num_class_steps, float* logits_out_dev, float* h_out_dev,
                  uint8_t* pred_out_dev, float* prob1_out_dev, int use_tensor_cores,
                  void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_forward_with_edge_features_x(const mpn_graph* g, const mpn_weights* w, const void* x_dev, int32_t x_kind,
                                     float* edge_attr_out_dev, int32_t num_enc_steps, int32_t num_class_steps, float* logits_out_dev,
                                     float* h_out_dev, uint8_t* pred_out_dev, float* prob1_out_dev, int use_tensor_cores,
                                     void* workspace_dev, size_t workspace_bytes, void* ef_workspace_dev, size_t ef_workspace_bytes,
                                     void* stream);
int mpn_forward_sharded_x(const mpn_graph* g, const mpn_weights* w, const void* x_dev, int32_t x_kind, const float* edge_attr_dev,
                          int32_t num_enc_steps, int32_t num_class_steps, int64_t total_edges, float* logits_out_dev,
                          float* h_out_dev, uint8_t* pred_out_dev, float* prob1_out_dev, int use_tensor_cores,
                          const mpn_peer_ctx* peers, void* workspace_dev, size_t workspace_bytes, void* stream);
int mpn_forward_sharded_with_edge_features_x(const mpn_graph* g, const mpn_weights* w, const void* x_dev, int32_t x_kind,
                                             float* edge_attr_out_dev, int32_t num_enc_steps, int32_t num_class_steps,
                                             int64_t total_edges, float* logits_out_dev, float* h_out_dev, uint8_t* pred_out_dev,
                                             float* prob1_out_dev, int use_tensor_cores, const mpn_peer_ctx* peers,
                                             void* workspace_dev, size_t workspace_bytes, void* ef_workspace_dev,
                                             size_t ef_workspace_bytes, void* stream);
int mpn_plan_node_encoder_x(mpn_fwd_plan* plan, const void* x_dev, int32_t x_kind, void* stream);
int mpn_normalize_columns_x(const void* x_dev, int32_t x_kind, int32_t n, int32_t D, float* out_dev, void* workspace_dev,
                            size_t workspace_bytes, void* stream);
int mpn_normalize_columns_batched_x(const void* x_dev, int32_t x_kind, int32_t n, int32_t D, const int32_t* graph_nptr_dev,
                                    int32_t n_graphs, float* out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPN_B200_H */
