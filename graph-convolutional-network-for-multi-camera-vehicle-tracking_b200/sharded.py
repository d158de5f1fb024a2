"""Row-block sharded MPN forward across the GPUs of one box (new; the reference is single-GPU, main.py:7).

Edges are sharded by the node at which messages are aggregated (``row = edge_index[0]``, models/mpn.py:97-99), so the
segment sums stay local.  Every BatchNorm over edges becomes an all-reduce of a 96-double moment vector; every
message-passing step after the first needs one all-gather of the updated node embeddings h [N,32].  ``x``, the weights
and the node encoder are replicated (cheaper than communicating).

The schedule (``sharded_forward``) is written against two small interfaces so it can be exercised on CPU with gloo:
``phases`` (the per-rank compute: CUDA plan API here, an oracle-backed fake in tests/) and ``comm`` (collectives).
"""
import ctypes as C

import torch

from . import _lib
from .graph import TrackletGraph, _on_device, current_stream_ptr, node_features, workspace


def partition_rows(rowptr: torch.Tensor, world: int):
    """Contiguous row blocks balanced by out-degree.  rowptr: int tensor [N+1] (CPU).  Returns list of (n0, n1)."""
    rp = rowptr.to(torch.int64).cpu()
    n = rp.numel() - 1
    total = int(rp[-1])
    bounds = [0]
    for r in range(1, world):
        target = total * r // world
        idx = int(torch.searchsorted(rp, torch.tensor(target), right=False))
        idx = min(max(idx, bounds[-1]), n)
        bounds.append(idx)
    bounds.append(n)
    return [(bounds[i], bounds[i + 1]) for i in range(world)]


def shard_edges(edge_index: torch.Tensor, n0: int, n1: int):
    """Slice [e0, e1) of a row-sorted edge_index whose rows fall in [n0, n1)."""
    row = edge_index[0].contiguous()
    lo = int(torch.searchsorted(row, torch.tensor(n0, device=row.device, dtype=row.dtype), right=False))
    hi = int(torch.searchsorted(row, torch.tensor(n1, device=row.device, dtype=row.dtype), right=False))
    return lo, hi


class TorchComm:
    """torch.distributed collectives (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0

    def all_reduce_sum(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)

    def all_gather_rows(self, full, blocks):
        """full: [N, W]; this rank's block is already written; fill the others."""
        if self.world == 1:
            return
        sizes = {b[1] - b[0] for b in blocks}
        n0, n1 = blocks[self.rank]
        if len(sizes) == 1 and blocks[-1][1] == full.shape[0]:
            self.dist.all_gather_into_tensor(full, full[n0:n1].clone(), group=self.group)
        else:                                       # ragged blocks: zero the rest and sum (x + 0 is exact)
            full[:n0].zero_()
            full[n1:].zero_()
            self.dist.all_reduce(full, op=self.dist.ReduceOp.SUM, group=self.group)


    def all_gather_ragged(self, t):
        """t: [R, n_local] (n_local differs per rank).  Returns the list of every rank's tensor, in rank order."""
        if self.world == 1:
            return [t]
        counts = torch.zeros(self.world, dtype=torch.int64, device=t.device)
        counts[self.rank] = t.shape[1]
        self.dist.all_reduce(counts, op=self.dist.ReduceOp.SUM, group=self.group)
        counts = [int(c) for c in counts.tolist()]
        width = max(max(counts), 1)
        mine = torch.zeros(t.shape[0], width, dtype=t.dtype, device=t.device)
        mine[:, :t.shape[1]] = t
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        self.dist.all_gather(parts, mine, group=self.group)
        return [p[:, :c] for p, c in zip(parts, counts)]


def _combine_sums(shards, comm):
    """Global BatchNorm moment sums: add the shards of this process, then all-reduce across processes."""
    if len(shards) == 1:
        comm.all_reduce_sum(shards[0].sums())
        return
    total = torch.stack([p.sums() for p in shards]).sum(dim=0)
    comm.all_reduce_sum(total)
    for p in shards:
        p.sums().copy_(total)


def _exchange_h(shards, comm, blocks):
    """Every shard needs h of ALL nodes for the next step's Pd table: the one all-gather per step."""
    if len(shards) == 1:
        comm.all_gather_rows(shards[0].h_full(), blocks)
        return
    assert comm.world == 1, "several local shards per process are only supported in a single process"
    for s, src in enumerate(shards):
        n0, n1 = blocks[s]
        for t, dst in enumerate(shards):
            if t != s:
                dst.h_full()[n0:n1].copy_(src.h_full()[n0:n1])


def sharded_forward(shards, comm, num_enc_steps: int, num_class_steps: int, blocks):
    """The phase/collective schedule of one forward over row-block shards.

    ``shards``: one phases object per row block held by this process (normally one; several emulate a multi-GPU run
    inside one process, which is how the 1-GPU and CPU tests cover the N>1 path).  Returns the number of classified steps.
    """
    if not isinstance(shards, (list, tuple)):
        shards = [shards]
    L, n_cls = int(num_enc_steps), int(num_class_steps)
    for p in shards:
        p.node_encoder()
    for stage in (_lib.STAGE_ENC0, _lib.STAGE_ENC1):
        for p in shards:
            p.sweep(0, stage)
            p.reduce(stage)
        _combine_sums(shards, comm)
        for p in shards:
            p.finalize(0, stage)
    k = 0
    if L == 0:
        for p in shards:
            p.sweep(0, _lib.STAGE_APPLY, out_index=0, last=True)
        return 1
    first_class_step = L - n_cls + 1
    for step in range(1, L + 1):
        if step > 1:
            _exchange_h(shards, comm, blocks)
        for p in shards:
            p.node_tables(step)
        for stage in (_lib.STAGE_EDGE, _lib.STAGE_NODE):
            for p in shards:
                p.sweep(step, stage)
                p.reduce(stage)
            _combine_sums(shards, comm)
            for p in shards:
                p.finalize(step, stage)
        cls = step >= first_class_step
        for p in shards:
            p.sweep(step, _lib.STAGE_APPLY, out_index=k if cls else None, last=(step == L))
            p.node_finalize(step)
        k += int(cls)
    return k


class CudaPhases:
    """Per-rank compute through the plan API of libmpn_b200 (include/mpn_b200.h)."""

    def __init__(self, graph: TrackletGraph, weights, x, edge_attr, L, n_cls, total_edges, logits, pred=None, prob1=None,
                 use_tensor_cores=True, ws_kind="forward_plan"):
        self.lib = _lib.lib()
        self.g, self.x, self.ea = graph, x, edge_attr
        self.dev = x.device
        self.logits, self.pred, self.prob1 = logits, pred, prob1
        need = self.lib.mpn_forward_workspace_bytes(graph.ref, C.byref(weights), L)
        self.ws = workspace(ws_kind, self.dev, need)
        self.plan = C.c_void_p()
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.mpn_plan_create(C.byref(self.plan), graph.ref, C.byref(weights), L, n_cls, int(total_edges),
                                                int(bool(use_tensor_cores)), self.ws.data_ptr(), self.ws.numel()))
        self._weights = weights
        sums_off = self.lib.mpn_plan_sums(self.plan) - self.ws.data_ptr()
        self._sums = self.ws[sums_off:sums_off + _lib.MPN_SUMS_DOUBLES * 8].view(torch.float64)
        h_off = self.lib.mpn_plan_h_full(self.plan) - self.ws.data_ptr()
        self._h = self.ws[h_off:h_off + graph.n_cols * _lib.MPN_DH * 4].view(torch.float32).view(graph.n_cols, _lib.MPN_DH)

    def close(self):
        if self.plan:
            self.lib.mpn_plan_destroy(self.plan)
            self.plan = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return current_stream_ptr(self.dev)

    def node_encoder(self):
        x, x_kind = node_features(self.x)
        _lib.check(self.lib.mpn_plan_node_encoder_x(self.plan, x.data_ptr(), x_kind, self.stream))

    def node_tables(self, step):
        _lib.check(self.lib.mpn_plan_node_tables(self.plan, step, self.stream))

    def sweep(self, step, stage, out_index=None, last=False):
        lg = pr = pb = None
        if stage == _lib.STAGE_APPLY and out_index is not None:
            lg = self.logits[out_index].data_ptr()
            if last:
                pr = self.pred.data_ptr() if self.pred is not None else None
                pb = self.prob1.data_ptr() if self.prob1 is not None else None
        _lib.check(self.lib.mpn_plan_sweep(self.plan, step, stage, self.ea.data_ptr(), lg, pr, pb, self.stream))

    def reduce(self, stage, with_consts=False):
        _lib.check(self.lib.mpn_plan_reduce(self.plan, stage, int(with_consts), self.stream))

    def finalize(self, step, stage):
        _lib.check(self.lib.mpn_plan_finalize(self.plan, step, stage, self.stream))

    def node_finalize(self, step):
        _lib.check(self.lib.mpn_plan_node_finalize(self.plan, step, self.stream))

    def sums(self):
        return self._sums

    def h_full(self):
        return self._h


SUMS_BYTES = 2 * _lib.MPN_MAX_PEERS * _lib.MPN_SUMS_DOUBLES * 8      # two slots x 16 source ranks x 96 fp64 moment sums (pushed by the sources)
FLAGS_OFFSET = SUMS_BYTES                            # 4 x 16 uint64 sequence flags: [moments][src], [h][src], [column stats][0], [node tables][src]
CSTATS_OFFSET = FLAGS_OFFSET + 512                   # two slots of [1024][2] fp64 column sums (sharded node encoder)
H_OFFSET = CSTATS_OFFSET + 2 * _lib.MPN_PEER_CSTAT_COLS * 2 * 8        # h buffer [n_cols, 32] fp32 starts here; the node table
                                                                       # [n_cols, 4] int32 of the shared Gram follows it


class PeerMemory:
    """NVLink peer-mapped exchange buffers (torch.distributed._symmetric_memory) for the fused collectives of
    ``mpn_forward_sharded``: per rank 2 x 96 fp64 moment-sum slots, two sequence flags and an h buffer [n_cols,32]."""

    def __init__(self, n_cols: int, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.tables_offset = H_OFFSET + n_cols * _lib.MPN_DH * 4
        nbytes = self.tables_offset + n_cols * 16
        self.n_cols = n_cols
        self.buf = symm_mem.empty(nbytes, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.hdl = symm_mem.rendezvous(self.buf, self.group)
        torch.cuda.synchronize(device)
        dist.barrier(group=self.group)                 # every rank's flags are zero before anyone publishes
        self.rank, self.world = int(self.hdl.rank), int(self.hdl.world_size)
        if self.world > _lib.MPN_MAX_PEERS:
            raise RuntimeError("at most %d peers" % _lib.MPN_MAX_PEERS)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self.seq_moments = self.seq_h = self.seq_c = self.seq_t = 0
        self.ea_buf = self.ea_hdl = self.ea_ptrs = None         # peer-visible edge_attr (shared symmetric Gram), made on first use
        self.ea_edges = 0

    def reserve_edge_attr(self, max_edges_per_rank: int, device):
        """COLLECTIVE: (re)allocates the peer-visible edge_attr buffers, ``max_edges_per_rank`` edges on every rank."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        cap = int(max_edges_per_rank)
        self.ea_buf = symm_mem.empty(cap * 8, dtype=torch.uint8, device=device)
        self.ea_hdl = symm_mem.rendezvous(self.ea_buf, self.group)
        self.ea_ptrs = [int(p) for p in self.ea_hdl.buffer_ptrs]
        self.ea_edges = cap
        torch.cuda.synchronize(device)
        dist.barrier(group=self.group)

    def edge_attr_buffer(self, n_edges: int, device):
        """This rank's peer-visible edge_attr [n_edges, 2] for the shared symmetric Gram (every pair of nodes is computed by one
        rank, which stores the mirrored entry into the owner's buffer over NVLink).  The first call allocates collectively
        (1.25 x the largest shard of the group); a shard that outgrows the buffers raises (see reserve_edge_attr)."""
        import torch.distributed as dist
        if self.ea_buf is None:                         # first use: collective (every rank is in its first fused forward)
            need = torch.tensor([n_edges], dtype=torch.int64, device=device)
            dist.all_reduce(need, op=dist.ReduceOp.MAX, group=self.group)
            self.reserve_edge_attr(int(int(need.item()) * 1.25) + 1024, device)
        if n_edges > self.ea_edges:
            raise RuntimeError("this rank's shard has %d edges, the peer-visible edge_attr buffers hold %d: call "
                               "ShardedMPN.reserve_edge_attr(max_edges_per_rank) on EVERY rank before a larger graph "
                               "(the allocation is a collective)" % (n_edges, self.ea_edges))
        return self.ea_buf[:n_edges * 8].view(torch.float32).view(n_edges, 2)

    def ctx(self, shard_encoder: bool, blocks=None) -> "_lib.MpnPeerCtx":
        """The peer table of one call.  The pointer part is built once per (encoder mode, row blocks) — ~100 ctypes stores cost
        tens of microseconds on the host's critical path of every step — only the sequence numbers change per call."""
        shared = blocks is not None and self.ea_ptrs is not None
        key = (bool(shard_encoder), tuple(map(tuple, blocks)) if shared else None, self.ea_ptrs[0] if shared else 0)
        cache = self.__dict__.setdefault("_ctx_cache", {})
        c = cache.get(key)
        if c is None:
            if len(cache) > 8:
                cache.clear()
            c = cache[key] = _lib.MpnPeerCtx()
            c.rank, c.world = self.rank, self.world
            for r, base in enumerate(self.ptrs):
                c.sums[r] = base
                c.flags[r] = base + FLAGS_OFFSET
                c.cstats[r] = base + CSTATS_OFFSET
                c.h[r] = base + H_OFFSET
            c.shard_node_encoder = int(shard_encoder)
            if shared:                                         # shared symmetric Gram
                for r, base in enumerate(self.ptrs):
                    c.edge_attr[r] = self.ea_ptrs[r]
                    c.node_tables[r] = base + self.tables_offset
                for r, (b0, b1) in enumerate(blocks):
                    c.block_start[r] = int(b0)
                c.block_start[len(blocks)] = int(blocks[-1][1])
        c.seq_moments, c.seq_h, c.seq_c, c.seq_t = self.seq_moments, self.seq_h, self.seq_c, self.seq_t
        return c

    def advance(self, L: int, shard_encoder: bool, n_layers: int, shared_gram: bool = False):
        self.seq_t += 1 if shared_gram else 0
        self.seq_moments += 2 + 2 * L
        self.seq_h += max(L - 1, 0) + (1 if shard_encoder else 0)
        self.seq_c += n_layers if shard_encoder else 0


class ShardedMPN:
    """Row-block sharded forward.  Each rank passes its own shard (``edge_index`` rows inside its block, global ids)
    plus the replicated ``x``; outputs stay sharded (logits of the local edges, h of the local rows).

    ``fused=True`` (default): one launch sequence per rank with the collectives inside the kernels over NVLink peer
    memory (``mpn_forward_sharded``).  If symmetric memory cannot be set up the call RAISES (there is no silent change of
    schedule); ``fused=False`` selects the phase schedule with NCCL collectives between the phases (``sharded_forward``) — the
    reference schedule the fused kernels are tested against.  ``path`` names the one in use.
    """

    def __init__(self, model, group=None, fused: bool = True, shard_node_encoder: bool = True, shared_gram: bool = True):
        """``shared_gram`` (fused path, edge features computed inside the call): the ranks share ONE symmetric Gram — every pair of
        nodes is computed by one rank only, the mirrored entry goes into its owner's edge_attr over NVLink (half the tensor-core
        work per rank).  Needs contiguous row blocks that cover all nodes in rank order; ``last_edge_attr`` is then a view of a
        peer-visible buffer that the next call overwrites."""
        self.model = model
        self.shared_gram = bool(shared_gram)
        self.shard_node_encoder = shard_node_encoder
        self.comm = TorchComm(group)
        self.fused = fused and self.comm.world > 1
        self.peers = None
        self._totals = {}

    def _total_edges(self, g, dev):
        key = id(g)
        if key not in self._totals:
            tot = torch.tensor([g.n_edges], dtype=torch.float64, device=dev)
            self.comm.all_reduce_sum(tot)
            if len(self._totals) > 16:
                self._totals.clear()
            self._totals[key] = (g, int(tot.item()))
        return self._totals[key][1]

    def reserve_edge_attr(self, max_edges_per_rank: int, n_cols: int, device):
        """COLLECTIVE: size the peer-visible edge_attr buffers of the shared symmetric Gram for shards of up to
        ``max_edges_per_rank`` edges (graphs of ``n_cols`` nodes).  Only needed before a graph larger than 1.25 x the first one."""
        self._peer_memory(n_cols, device).reserve_edge_attr(max_edges_per_rank, device)

    def _blocks_cover(self, blocks, world, n_nodes) -> bool:
        """Contiguous non-empty row blocks in rank order that cover all nodes (what the shared Gram needs); cached per block list
        (the check is on the host's critical path of every step)."""
        key = (tuple(map(tuple, blocks)), int(world), int(n_nodes))
        hit = self.__dict__.get("_cover_cache")
        if hit is not None and hit[0] == key:
            return hit[1]
        ok = (len(blocks) == world and blocks[0][0] == 0 and blocks[-1][1] == n_nodes and
              all(blocks[i][1] == blocks[i + 1][0] for i in range(len(blocks) - 1)) and all(b1 > b0 for b0, b1 in blocks))
        self._cover_cache = (key, ok)
        return ok

    def shared_gram_used(self) -> bool:
        """True when the last fused forward with ``local_edge_attr=None`` took the shared symmetric Gram (every rank's rows dense
        cross-camera); synchronises the stream.  Tests / bench."""
        last = getattr(self, "_last_ef", None)
        if last is None:
            return False
        g, D, ef_ws = last
        return _lib.lib().mpn_shared_gram_mode(g.ref, D, ef_ws.data_ptr(), ef_ws.numel(), current_stream_ptr(g.device)) == 2

    @property
    def path(self) -> str:
        return "fused_peer_memory" if self.fused else "nccl_phase_schedule"

    def _peer_memory(self, n_cols, dev):
        if self.peers is not None and self.peers.n_cols == n_cols:
            return self.peers
        try:
            self.peers = PeerMemory(n_cols, dev, self.comm.group)
        except Exception as e:                          # noqa: BLE001
            self.peers = None
            raise RuntimeError("ShardedMPN(fused=True): the NVLink peer-memory exchange buffers could not be set up (%s: %s); "
                               "pass fused=False for the NCCL phase schedule" % (type(e).__name__, e)) from e
        return self.peers

    def post_processing(self, num_cameras, graph, pred, prob1, CONFIG, numbering='reference'):
        """CUT / PRUNE / CUT / SPLIT + labels for this rank's shard (see ``sharded_post_processing``)."""
        return sharded_post_processing(num_cameras, (graph, pred, prob1), CONFIG, graph.n_cols, comm=self.comm,
                                       numbering=numbering)

    @torch.no_grad()
    def forward(self, x, local_edge_index, local_edge_attr, blocks, fuse_decisions=False, graph=None, total_edges=None):
        """``total_edges``: number of edges of the WHOLE graph if the caller knows it (saves one all-reduce + host sync).
        ``local_edge_attr=None``: the edge features of this rank's rows (inference.py:453-456) are computed inside the call — they
        overlap the node encoder and hand the first BatchNorm's moment sums over — and kept in ``self.last_edge_attr``."""
        from .mpn import USE_TENSOR_CORES
        m, comm = self.model, self.comm
        dev = x.device
        n0, n1 = blocks[comm.rank]
        g = graph if graph is not None else TrackletGraph(local_edge_index, x.shape[0], row_offset=n0, n_rows=n1 - n0)
        if g.perm is not None:
            raise ValueError("sharded forward needs (row, col)-sorted local edges")
        W = m._weights(dev)
        L, n_cls = int(m.num_enc_steps), int(m.num_class_steps)
        if L > 0:
            n_cls = min(n_cls, L)         # as MOTMPNet.forward (models/mpn.py:281,290)
        n_out = 1 if L == 0 else n_cls
        x, x_kind = node_features(x)
        make_features = local_edge_attr is None          # edge features of this rank's rows computed inside the call
        logits = torch.empty(max(n_out, 1), g.n_edges, 2, dtype=torch.float32, device=dev)
        pred = torch.empty(g.n_edges, dtype=torch.uint8, device=dev) if fuse_decisions else None
        prob1 = torch.empty(g.n_edges, dtype=torch.float32, device=dev) if fuse_decisions else None
        peers = self._peer_memory(x.shape[0], dev) if (self.fused and L >= 1) else None
        if peers is not None and g.n_edges == 0:
            # every rank takes part in every exchange of the fused schedule; a block without edges cannot (its peers would wait
            # for it until the 10 s trap of the flag wait)
            raise ValueError("fused sharded forward: this rank's row block [%d, %d) has no edges; balance the blocks by degree "
                             "(partition_rows) or use ShardedMPN(fused=False)" % (n0, n1))
        if make_features and peers is None:
            from .edge_features import edge_features
            ea = edge_features(x, None, graph=g)
        elif make_features:
            shared = self.shared_gram and g.n_edges > 0 and self._blocks_cover(blocks, peers.world, x.shape[0])
            ea = peers.edge_attr_buffer(g.n_edges, dev) if shared else torch.empty(g.n_edges, 2, dtype=torch.float32, device=dev)
        else:
            ea = local_edge_attr.contiguous().float()
        self.last_edge_attr = ea
        if peers is not None:
            total = int(total_edges) if total_edges is not None else -1      # -1: summed on the device, no host collective
            lib = _lib.lib()
            need = lib.mpn_forward_workspace_bytes(g.ref, C.byref(W), L)
            ws = workspace("forward_sharded", dev, need)
            h_local = torch.empty(g.n_nodes, _lib.MPN_DH, dtype=torch.float32, device=dev)
            enc = self.__dict__.get("_enc_mode")                   # (weights struct, layers, sharded encoder?): per weight version
            if enc is None or enc[0] is not W:
                nl = int(W.n_node_layers)
                enc = self._enc_mode = (W, nl, self.shard_node_encoder and max(W.node_dims[1:nl + 1]) <= _lib.MPN_PEER_CSTAT_COLS)
            n_layers, shard_enc = enc[1], enc[2]
            shared = make_features and self.shared_gram and ea.data_ptr() == (peers.ea_ptrs[peers.rank] if peers.ea_ptrs else -1)
            ctx = peers.ctx(shard_enc, blocks if shared else None)
            with _on_device(dev):
                if make_features:
                    ef_ws = workspace("edge_features", dev, lib.mpn_edge_features_workspace_bytes(g.ref, x.shape[1]))
                    _lib.check(lib.mpn_forward_sharded_with_edge_features_x(
                        g.ref, C.byref(W), x.data_ptr(), x_kind, ea.data_ptr(), L, n_cls, total, logits.data_ptr(), h_local.data_ptr(),
                        pred.data_ptr() if pred is not None else None, prob1.data_ptr() if prob1 is not None else None,
                        int(bool(USE_TENSOR_CORES)), C.byref(ctx), ws.data_ptr(), ws.numel(), ef_ws.data_ptr(), ef_ws.numel(),
                        current_stream_ptr(dev)))
                else:
                    _lib.check(lib.mpn_forward_sharded_x(g.ref, C.byref(W), x.data_ptr(), x_kind, ea.data_ptr(), L, n_cls, total,
                                                         logits.data_ptr(), h_local.data_ptr(),
                                                         pred.data_ptr() if pred is not None else None,
                                                         prob1.data_ptr() if prob1 is not None else None,
                                                         int(bool(USE_TENSOR_CORES)), C.byref(ctx), ws.data_ptr(), ws.numel(),
                                                         current_stream_ptr(dev)))
            peers.advance(L, shard_enc, n_layers, shared_gram=shared)
            self._last_ef = (g, int(x.shape[1]), ef_ws) if make_features else None
            return {'classified_edges': [logits[i] for i in range(n_out)]}, h_local, pred, prob1
        total = int(total_edges) if total_edges is not None else self._total_edges(g, dev)
        with torch.cuda.device(dev):
            ph = CudaPhases(g, W, x, ea, L, n_cls, total, logits, pred, prob1, USE_TENSOR_CORES)
            try:
                sharded_forward(ph, comm, L, n_cls, blocks)
                h_local = ph.h_full()[n0:n1].clone()
            finally:
                ph.close()
        return {'classified_edges': [logits[i] for i in range(n_out)]}, h_local, pred, prob1


# ------------------------------------------------------------------------------------------------------------------
# Post-processing of a row-block sharded graph (new; inference.post_processing, inference.py:70-169, is single-GPU)
# ------------------------------------------------------------------------------------------------------------------
class CudaPostOps:
    """Per-rank pieces of the sharded post-processing through libmpn_b200 (include/mpn_b200.h): shard compaction,
    the fixed-point rounds on the merged active list, and the write-back into the shard's decisions."""

    def compact(self, graph, pred, prob1):
        """Active edges of one shard in edge order: (src, dst) global int32, shard-local edge id int32, prob1 f32."""
        if not (pred.is_cuda and prob1.is_cuda):
            raise RuntimeError("sharded post-processing needs CUDA tensors: the B200 path has no CPU fallback")
        if pred.dtype != torch.uint8 or not pred.is_contiguous() or pred.numel() != graph.n_edges:
            raise ValueError("pred must be the shard's contiguous uint8 decisions, one per local edge")
        if graph.perm is not None:
            raise ValueError("sharded post-processing needs (row, col)-sorted local edges")
        stride = 1
        if prob1.dim() == 2:                                  # [E,2] softmax: column 1 in place
            prob1, stride = prob1[:, 1], int(prob1.stride(0))
        elif prob1.numel() > 1:
            stride = int(prob1.stride(0))
        if prob1.dtype != torch.float32 or stride < 1 or prob1.numel() != graph.n_edges:
            raise ValueError("prob1 must be float32 with one entry per local edge")
        dev, lib = pred.device, _lib.lib()
        ws = workspace("compact", dev, lib.mpn_compact_workspace_bytes(graph.ref))
        n = C.c_int64(0)
        stream = current_stream_ptr(dev)
        with torch.cuda.device(dev):
            _lib.check(lib.mpn_count_active(graph.ref, pred.data_ptr(), C.byref(n), ws.data_ptr(), ws.numel(), stream))
            n = int(n.value)
            src, dst, eid = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3))
            prob = torch.empty(n, dtype=torch.float32, device=dev)
            if n:
                _lib.check(lib.mpn_compact_active(graph.ref, pred.data_ptr(), prob1.data_ptr(), stride, src.data_ptr(),
                                                  dst.data_ptr(), eid.data_ptr(), prob.data_ptr(), ws.data_ptr(), ws.numel(),
                                                  stream))
        return src, dst, eid, prob

    def run(self, num_cameras, src, dst, prob, CONFIG, n_nodes, numbering):
        """CUT / PRUNE / CUT / SPLIT + labels on the merged active list (every entry active).  Returns
        (ID_pred int64 CPU [n_nodes], keep uint8 [A] on the device)."""
        from types import SimpleNamespace
        from .postprocess import compute_SCC_and_Clusters, post_processing
        a = int(src.numel())
        keep = torch.ones(a, dtype=torch.uint8, device=src.device)
        if a == 0:
            return torch.arange(n_nodes, dtype=torch.int64), keep
        ei = torch.stack([src.long(), dst.long()])
        if not any(CONFIG[k] for k in ('CUTTING', 'PRUNING', 'SPLITTING')):
            return compute_SCC_and_Clusters(ei.t().cpu().numpy(), n_nodes)[0], keep
        data = SimpleNamespace(edge_index=ei, num_nodes=int(n_nodes))
        ID, new_pred = post_processing(num_cameras, None, None, keep.long(), None, CONFIG, data, prob.contiguous(),
                                       numbering=numbering)
        return ID, (new_pred != 0).to(torch.uint8)

    def clear(self, pred, eid, keep):
        if eid.numel():
            keep = keep.contiguous()
            with torch.cuda.device(pred.device):
                _lib.check(_lib.lib().mpn_clear_inactive(pred.data_ptr(), eid.data_ptr(), keep.data_ptr(), eid.numel(),
                                                         current_stream_ptr(pred.device)))


def sharded_post_processing(num_cameras, shards, CONFIG, n_nodes, comm=None, numbering='reference', ops=None):
    """inference.post_processing (inference.py:70-169) for a graph whose edges are sharded by row block.

    ``shards``: ``(graph, pred, prob1)`` of this rank - the shard's TrackletGraph, its uint8 decisions and softmax[:,1]
    as ``ShardedMPN.forward(..., fuse_decisions=True)`` returns them - or a list of such triples held by this process
    (consecutive row blocks; how the 1-GPU and CPU tests emulate N > 1).  Every stage of the reference only ever looks
    at ACTIVE edges, so each shard contributes the order-preserving compaction of its active edges (the E-sized sweep
    stays sharded), the ranks exchange those lists ONCE (A << E entries of 12 bytes) and run the fixed-point rounds on
    the merged list, whose order is the global edge order (so arg-min ties and the label numbering match the reference
    bit for bit); finally every shard clears the decisions the rounds removed.

    Returns ``(ID_pred, preds)``: int64 CPU labels [n_nodes], identical on every rank, and the shard decisions (updated in
    place), one tensor per triple passed in."""
    from .postprocess import _as_bool
    single = isinstance(shards, tuple)
    if single:
        shards = [shards]
    comm = comm if comm is not None else TorchComm()
    ops = ops if ops is not None else CudaPostOps()
    cfg = {k: _as_bool(CONFIG[k]) for k in ('CUTTING', 'PRUNING', 'SPLITTING')}
    lists = [ops.compact(g, pred, prob1) for (g, pred, prob1) in shards]
    mine = torch.cat([torch.stack([s, d, p.view(torch.int32)]) for (s, d, _e, p) in lists], dim=1)
    parts = comm.all_gather_ragged(mine)
    merged = torch.cat(parts, dim=1) if len(parts) > 1 else parts[0]
    ID, keep = ops.run(int(num_cameras), merged[0].contiguous(), merged[1].contiguous(),
                       merged[2].contiguous().view(torch.float32), cfg, int(n_nodes), numbering)
    off = sum(int(p.shape[1]) for p in parts[:comm.rank])
    for (g, pred, _prob1), (_s, _d, eid, _p) in zip(shards, lists):
        ops.clear(pred, eid, keep[off:off + eid.numel()])
        off += int(eid.numel())
    preds = [pred for (_g, pred, _p) in shards]
    return ID, (preds[0] if single else preds)
