"""Throughput path for a stream of tracklet graphs held in HOST memory.

The reference driver handles one graph per loop iteration (``for data in val_loader`` with batch size 1,
inference.py:375): load the tracklets' ReID features, ``.cuda()`` them (inference.py:399), build the graph, run the MPN
(inference.py:469), read the decisions back (inference.py:482-485).  Done one graph at a time, the PCIe copies either side of
the kernels are serial time (configs[1]: 0.6 ms in, 0.27 ms out, around 0.9 ms of kernels).  ``GraphStream`` keeps ``depth``
graphs in flight on three CUDA streams so that the host->device copy of graph i+1 and the device->host copy of graph i-1
overlap the kernels of graph i; every graph still pays its own copies, they just stop being serial.

Nothing here computes: it is stream / event / buffer plumbing around ``TrackletGraph.from_cameras`` and
``MOTMPNet.forward`` (edge features inside the call), which run unchanged on the caller's current stream.
"""
import torch

from . import _lib
from .graph import TrackletGraph, current_stream_ptr, release_scope, workspace_scope


class _Slot:
    __slots__ = ("x_dev", "in_done", "compute_done", "out_done", "keep", "busy", "seen_key", "cap_key", "cap")

    def __init__(self):
        self.x_dev = None
        self.in_done = torch.cuda.Event()
        self.compute_done = torch.cuda.Event()
        self.out_done = torch.cuda.Event()
        self.keep = None             # device tensors of the graph in flight (outputs of the forward, graph tables)
        self.busy = False
        self.seen_key = self.cap_key = self.cap = None       # graph_replay: signature run eagerly once / captured signature


class GraphStream:
    """``submit`` enqueues one graph (pinned host features + camera ids in, pinned host decisions out) and returns without
    waiting; ``drain`` waits for everything submitted.  A slot's buffers are reused ``depth`` submits later; the stream /
    event order guarantees the previous occupant's copies have finished by then, so the caller must have consumed a
    ``pred_host`` buffer before passing the same buffer to a submit ``depth`` calls later (or simply use ``depth + 1`` buffers).
    """

    def __init__(self, model, device, depth: int = 2, graph_replay: bool = False, packed_decisions: bool = False):
        """``graph_replay``: when a slot sees the same signature (feature shape, camera layout, weights) a second time, the graph
        tables + edge features + forward + decisions of that slot are captured as one CUDA graph over slot-static buffers and
        replayed from then on: one launch instead of ~40 per graph (configs[1]: 0.84 -> 0.79 ms per step, same bits; the win is
        larger for small graphs, whose time is mostly launches).  Off by default: a stream of graphs of ever-changing shapes
        would only pay the captures.
        ``packed_decisions``: the decisions travel to the host as a bit mask (``mpn_pack_decisions``: 1 bit per edge, 1/8 of the
        D2H bytes — on a multi-GPU box the host's memory system, shared by all GPUs, bounds the stream); ``pred_host`` is then
        pinned uint8 [4 * ceil(E / 32)], ``unpack_decisions(pred_host, E)`` gives the 0/1 array back."""
        self.packed = bool(packed_decisions)
        if depth < 1:
            raise ValueError("depth must be >= 1")
        self.model, self.device, self.depth = model, torch.device(device), int(depth)
        self.graph_replay = bool(graph_replay)
        if self.device.type != "cuda":
            raise RuntimeError("GraphStream needs a CUDA device: the B200 path has no CPU fallback")
        self.copy_in = torch.cuda.Stream(self.device)
        self.copy_out = torch.cuda.Stream(self.device)
        self.slots = [_Slot() for _ in range(self.depth)]
        self.n_submitted = 0
        GraphStream._instances = getattr(GraphStream, "_instances", 0) + 1
        self._id = GraphStream._instances

    def submit(self, x_host, cam_ids, pred_host, prob_host=None):
        """``x_host``: pinned fp32, fp16 or bf16 [N, D] (column-normalised ReID features, inference.py:403-404; 16-bit features
        cross PCIe in half the bytes and give the decisions of their fp32 widening); ``cam_ids``: host sequence of
        per-node camera ids, nodes grouped by ascending camera (dataset.py:279-281); ``pred_host``: pinned uint8 [E] that
        receives argmax(logits) (inference.py:479) in the graph's edge order; ``prob_host``: optional pinned fp32 [E] for
        softmax(logits)[:, 1] (inference.py:475-477).  Returns the ticket to pass to ``wait``."""
        if x_host.is_cuda or pred_host.is_cuda or not (x_host.is_pinned() and pred_host.is_pinned()):
            raise ValueError("GraphStream.submit takes pinned HOST tensors (x_host, pred_host)")
        if x_host.dtype not in (torch.float32, torch.float16, torch.bfloat16) or x_host.dim() != 2 or not x_host.is_contiguous():
            raise ValueError("x_host must be a contiguous float32, float16 or bfloat16 [N, D] tensor")
        dev = self.device
        compute = torch.cuda.current_stream(dev)
        slot = self.slots[self.n_submitted % self.depth]
        ticket = self.n_submitted
        with torch.cuda.device(dev):
            full_shape = self._device_feature_shape(x_host, cam_ids)
            if slot.x_dev is None or tuple(slot.x_dev.shape) != tuple(full_shape) or slot.x_dev.dtype != x_host.dtype:
                if slot.busy:
                    slot.compute_done.synchronize()
                slot.x_dev = torch.empty(full_shape, dtype=x_host.dtype, device=dev)
                self.copy_in.wait_stream(compute)          # the allocator may hand out memory this stream still uses
            if slot.busy:
                compute.wait_event(slot.out_done)            # the previous occupant's outputs have left the device: free them
            slot.keep = None
            cap = None
            if self.graph_replay:
                key = self._signature(slot, cam_ids)
                if slot.cap_key == key:
                    cap = slot.cap
                elif slot.seen_key == key:                   # second time: capture (the first, eager run did the lazy set-up)
                    slot.cap, slot.cap_key = self._capture(slot, cam_ids, self.n_submitted % self.depth), key
                    cap = slot.cap
                else:
                    slot.seen_key, slot.cap, slot.cap_key = key, None, None
            # K0 on the device (does not need x): only the camera layout crosses PCIe
            g = cap.g if cap is not None else self._tables(cam_ids)
            n_out = 4 * ((g.n_edges + 31) // 32) if self.packed else g.n_edges
            if pred_host.numel() != n_out or pred_host.dtype != torch.uint8:
                raise ValueError("pred_host must be uint8 with %d entries (%s)" % (n_out, "bit mask, 4 * ceil(E / 32) bytes" if self.packed
                                                                                  else "one per edge"))
            if prob_host is not None and (prob_host.numel() != g.n_edges or prob_host.dtype != torch.float32
                                          or not prob_host.is_pinned()):
                raise ValueError("prob_host must be pinned float32 with one entry per edge")
            if g.n_cols != slot.x_dev.shape[0]:
                raise ValueError("cam_ids has %d entries, the features %d rows" % (g.n_cols, slot.x_dev.shape[0]))
            if slot.busy:
                self.copy_in.wait_event(slot.compute_done)   # the previous occupant's kernels have read x_dev
            with torch.cuda.stream(self.copy_in):
                self._copy_in(slot, x_host)
                slot.in_done.record(self.copy_in)
            compute.wait_event(slot.in_done)
            if cap is not None:
                cap.graph.replay()                           # tables + edge features + forward + decisions: one launch
                data, pred, prob1 = cap.data, cap.pred, cap.prob1
                out = cap.bits if self.packed else pred
            else:
                data, pred, prob1 = self._compute(slot, g)
                out = self._pack(pred) if self.packed else pred
            slot.compute_done.record(compute)
            self.copy_out.wait_event(slot.compute_done)
            with torch.cuda.stream(self.copy_out):
                pred_host.copy_(out, non_blocking=True)
                if prob_host is not None:
                    prob_host.copy_(prob1, non_blocking=True)
                slot.out_done.record(self.copy_out)
            slot.keep = (g, pred, prob1, data, out)
            slot.busy = True
        self.n_submitted += 1
        return ticket

    def _pack(self, pred):
        """uint8 [E] decisions -> uint8 [4 * ceil(E / 32)] bit mask, on the current stream."""
        bits = torch.empty(4 * ((pred.numel() + 31) // 32), dtype=torch.uint8, device=pred.device)
        _lib.check(_lib.lib().mpn_pack_decisions(pred.data_ptr(), pred.numel(), bits.data_ptr(), current_stream_ptr(pred.device)))
        return bits

    # ---- hooks (ShardedGraphStream overrides them)
    def _device_feature_shape(self, x_host, cam_ids):
        return tuple(x_host.shape)

    def _tables(self, cam_ids):
        return TrackletGraph.from_cameras(cam_ids, self.device)          # K0 on the device: only the camera layout crosses PCIe

    def _copy_in(self, slot, x_host):
        slot.x_dev.copy_(x_host, non_blocking=True)

    def _compute(self, slot, g):
        data = _Batch()
        data.x, data.mpn_graph, data.edge_attr, data.num_nodes = slot.x_dev, g, None, g.n_cols
        fuse = self.model.fuse_decisions
        self.model.fuse_decisions = True
        try:
            self.model(data)
        finally:
            self.model.fuse_decisions = fuse
        return data, self.model.last_pred, self.model.last_prob1

    def _signature(self, slot, cam_ids):
        import numpy as np
        cam = np.ascontiguousarray(np.asarray(cam_ids.cpu() if isinstance(cam_ids, torch.Tensor) else cam_ids).reshape(-1))
        self.model._weights(self.device)                   # refreshes the packed-weights key if a parameter changed
        return (slot.x_dev.data_ptr(), tuple(slot.x_dev.shape), slot.x_dev.dtype, str(cam.dtype), cam.tobytes(), self.model._packed[0])

    def _capture(self, slot, cam_ids, index):
        """One CUDA graph of K0 + K1 + forward + decisions for this slot.  Tensors allocated while capturing (graph tables,
        edge features, logits, decisions) live in the graph's private pool: their addresses are the same at every replay.  The
        library's scratch buffers are taken from a scope of this slot's own (and pre-sized by an eager run inside the scope), so
        no other call can grow — and thereby free — memory whose address the graph has baked in."""
        model, dev = self.model, self.device
        tag = "graphstream%d.slot%d" % (self._id, index)
        slot.cap = None
        release_scope(tag)
        with workspace_scope(tag):
            warm = _Batch()
            warm.x, warm.edge_attr = slot.x_dev, None
            warm.mpn_graph = TrackletGraph.from_cameras(cam_ids, dev)
            warm.num_nodes = warm.mpn_graph.n_cols
            fuse0, small0 = model.fuse_decisions, model.use_cuda_graph
            model.fuse_decisions, model.use_cuda_graph = True, False
            try:
                model(warm)                                     # sizes the scoped workspaces outside the capture
            finally:
                model.fuse_decisions, model.use_cuda_graph = fuse0, small0
            return self._capture_scoped(slot, cam_ids)

    def _capture_scoped(self, slot, cam_ids):
        model, dev = self.model, self.device
        cap = _Batch()
        cap.graph = torch.cuda.CUDAGraph()
        fuse, small = model.fuse_decisions, model.use_cuda_graph
        model.fuse_decisions, model.use_cuda_graph = True, False      # no replay of the small-graph CUDA graph inside a capture
        try:
            with torch.cuda.graph(cap.graph):
                cap.g = TrackletGraph.from_cameras(cam_ids, dev)
                cap.data = _Batch()
                cap.data.x, cap.data.mpn_graph, cap.data.edge_attr, cap.data.num_nodes = slot.x_dev, cap.g, None, cap.g.n_cols
                model(cap.data)
                cap.pred, cap.prob1 = model.last_pred, model.last_prob1
                cap.bits = self._pack(cap.pred) if self.packed else None
        finally:
            model.fuse_decisions, model.use_cuda_graph = fuse, small
        return cap

    def wait(self, ticket: int):
        """Blocks the host until the decisions of ``ticket`` are in its ``pred_host``."""
        if not 0 <= ticket < self.n_submitted:
            raise ValueError("unknown ticket")
        # a reused slot's event belongs to a later graph: the copy-out stream is in order, so that one implies this one
        self.slots[ticket % self.depth].out_done.synchronize()

    def drain(self, host_sync: bool = True):
        """Orders the caller's current stream after every outstanding copy (so an event recorded next on that stream closes a
        timed region around the whole pipeline) and, with ``host_sync``, blocks the host until they are done."""
        compute = torch.cuda.current_stream(self.device)
        for slot in self.slots:
            if slot.busy:
                compute.wait_event(slot.out_done)
        if host_sync:
            for slot in self.slots:
                if slot.busy:
                    slot.out_done.synchronize()
                    slot.keep = None


def unpack_decisions(bits_host, n_edges: int):
    """The 0/1 decisions (numpy uint8 [n_edges]) of a ``GraphStream(packed_decisions=True)`` output buffer."""
    import numpy as np
    arr = bits_host.numpy() if isinstance(bits_host, torch.Tensor) else np.asarray(bits_host)
    return np.unpackbits(arr.reshape(-1).view(np.uint8), bitorder="little")[:int(n_edges)]


class _Batch:
    """Attribute bag standing in for torch_geometric.data.Data (inference.py:458)."""


class ShardedGraphStream(GraphStream):
    """The same pipeline for a row-block sharded graph (one process per GPU, ``ShardedMPN``): every rank copies only ITS rows of
    the features from its pinned host buffer, the ranks all-gather them over NVLink on the copy-in stream (NCCL), each rank runs
    its shard (tables of its row block, edge features of its rows, sharded forward) and copies its shard's decisions back (fp16 /
    bf16 rows are gathered in half and read in place, as in ``GraphStream``).  One
    graph computes at a time (the peer-memory exchange buffers of ``ShardedMPN`` are single-buffered); the copies and the
    all-gather of graph i+1 overlap the kernels of graph i.  ``submit(x_rows_host, cam_ids, pred_host)``: ``x_rows_host`` =
    rows ``blocks[rank]`` of the feature matrix."""

    def __init__(self, sharded, blocks, device, depth: int = 2, packed_decisions: bool = False):
        super().__init__(sharded.model, device, depth=depth, graph_replay=False, packed_decisions=packed_decisions)
        self.sharded, self.blocks = sharded, [tuple(b) for b in blocks]
        self.rank = sharded.comm.rank
        n0, n1 = self.blocks[self.rank]
        if any(b[1] - b[0] != n1 - n0 for b in self.blocks):
            raise ValueError("ShardedGraphStream needs equal row blocks (NCCL all-gather of the feature rows)")

    def _device_feature_shape(self, x_host, cam_ids):
        n0, n1 = self.blocks[self.rank]
        if x_host.shape[0] != n1 - n0:
            raise ValueError("x_host must hold this rank's %d rows" % (n1 - n0))
        return (self.blocks[-1][1], x_host.shape[1])

    def _tables(self, cam_ids):
        import numpy as np
        cam = np.asarray(cam_ids.cpu() if isinstance(cam_ids, torch.Tensor) else cam_ids).reshape(-1)
        sizes = np.bincount(cam - cam.min()).astype(np.int64)
        self._total_edges = int((sizes * (cam.size - sizes)).sum())       # of the WHOLE graph: no all-reduce / host sync per submit
        return TrackletGraph.from_cameras(cam_ids, self.device, row_block=self.blocks[self.rank])

    def _copy_in(self, slot, x_host):
        import torch.distributed as dist
        n0, n1 = self.blocks[self.rank]
        mine = slot.x_dev[n0:n1]
        mine.copy_(x_host, non_blocking=True)
        dist.all_gather_into_tensor(slot.x_dev, mine, group=self.sharded.comm.group)      # in place: rank r's rows sit at offset r

    def _compute(self, slot, g):
        out, h, pred, prob1 = self.sharded.forward(slot.x_dev, None, None, self.blocks, fuse_decisions=True, graph=g,
                                                   total_edges=self._total_edges)
        return (out, h, self.sharded.last_edge_attr), pred, prob1
