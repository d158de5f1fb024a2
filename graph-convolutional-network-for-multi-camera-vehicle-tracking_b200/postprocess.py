"""Drop-in CUTTING / PRUNING / SPLITTING post-processing (inference.py:70-169, utils.py:30-339) on the GPU.

Function names, argument order and return conventions mirror the reference so that ``inference.py`` can bind
them unchanged (see INTEGRATION.md).  Arguments the reference only uses to rebuild Python tuple lists
(``predicted_active_edges``, ``edge_list``) are accepted and ignored: the kernels read ``data.edge_index``.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .graph import current_stream_ptr, graph_for, workspace


def _as_bool(v):
    """CLI overrides arrive as strings (inference.py:75-91)."""
    if isinstance(v, str):
        return v == 'True'
    return bool(v)


def _stage_flags(CONFIG):
    """The CUT | PRUNE | SPLIT flag word of CONFIG, after the same in-place fix-up of its values as inference.py:75-91."""
    for k in ('CUTTING', 'PRUNING', 'SPLITTING'):
        CONFIG[k] = _as_bool(CONFIG[k])
    return (_lib.POST_CUT if CONFIG['CUTTING'] else 0) | (_lib.POST_PRUNE if CONFIG['PRUNING'] else 0) | \
        (_lib.POST_SPLIT if CONFIG['SPLITTING'] else 0)


class _Post:
    """Shared plumbing: graph tables, uint8 activity flags and fp32 probabilities in the graph's edge order."""

    def __init__(self, data, predictions, probs=None):
        if not predictions.is_cuda:
            raise RuntimeError("post-processing needs CUDA tensors: the B200 path has no CPU fallback")
        self.dev = predictions.device
        pre = getattr(data, "mpn_graph", None)
        self.g = pre if pre is not None else graph_for(data, data.edge_index, int(data.num_nodes))
        self.g.validate()                          # a graph built with validate='deferred' is checked here at the latest
        self.lib = _lib.lib()
        act = (predictions.reshape(-1) != 0).to(torch.uint8)
        self.act = act[self.g.perm].contiguous() if self.g.perm is not None else act.contiguous()
        self.prob_ptr, self.prob_stride, self._prob_keep = None, 1, None
        if probs is not None:
            p = probs
            if p.dim() == 2:                       # [E,2] softmax: use column 1 in place (stride 2)
                p = p[:, 1]
            if p.dtype != torch.float32 or not p.is_cuda:
                p = p.float().to(self.dev)
            if self.g.perm is not None:
                p = p[self.g.perm].contiguous()
            if p.dim() != 1 or p.numel() != self.g.n_edges:
                raise ValueError("probabilities must have one entry per edge")
            st = p.stride(0) if p.numel() > 1 else 1
            if st < 1:
                p, st = p.contiguous(), 1
            self._prob_keep, self.prob_ptr, self.prob_stride = p, p.data_ptr(), int(st)
        need = self.lib.mpn_post_workspace_bytes(self.g.ref)
        self.ws = workspace("post", self.dev, need)
        self.stream = current_stream_ptr(self.dev)

    def predictions(self, like):
        act = self.act
        if self.g.perm is not None:
            out = torch.empty_like(act)
            out[self.g.perm] = act
            act = out
        return act.to(like.dtype)

    def caller_order_active(self):
        """(src, dst) int64 device tensors of the active edges in the CALLER's edge order (graphs with a ``perm``)."""
        g = self.g
        orig = torch.empty_like(self.act)
        orig[g.perm] = self.act
        idx = torch.nonzero(orig, as_tuple=False).reshape(-1)
        ei = g._keepalive                                      # sorted copy
        inv = torch.empty_like(g.perm)
        inv[g.perm] = torch.arange(g.perm.numel(), device=self.dev)
        sel = inv[idx]
        return ei[0, sel], ei[1, sel]

    def labels_reference(self):
        """ID_pred exactly as compute_SCC_and_Clusters numbers it (utils.py:30-52): int64 CPU tensor."""
        g = self.g
        act = self.act
        if g.perm is not None:
            # the reference scans active edges in the CALLER's edge order: compact in that order
            s, d = self.caller_order_active()
            s_h, d_h = s.to(torch.int32).cpu(), d.to(torch.int32).cpu()
            n = int(s.numel())
        else:
            # sorted graphs: partition + first-appearance keys on the device, the rank over the components on the host
            labels = torch.empty(g.n_nodes, dtype=torch.int64)
            ncomp = C.c_int32(0)
            with torch.cuda.device(self.dev):
                _lib.check(self.lib.mpn_labels_reference(g.ref, act.data_ptr(), labels.data_ptr(), C.byref(ncomp),
                                                         self.ws.data_ptr(), self.ws.numel(), self.stream))
            return labels, int(ncomp.value)
        labels = torch.empty(g.n_nodes, dtype=torch.int64)
        ncomp = C.c_int32(0)
        _lib.check(self.lib.mpn_labels_reference_host(s_h.data_ptr(), d_h.data_ptr(), n, g.n_nodes, labels.data_ptr(),
                                                      C.byref(ncomp)))
        return labels, int(ncomp.value)

    def labels_reference_batched(self):
        """The reference numbering of each graph of a batch, each numbered from 0: (int64 CPU [N], int64 CPU [G] counts)."""
        g = self.g
        if g.n_graphs <= 1:
            labels, n = self.labels_reference()
            return labels, torch.tensor([n], dtype=torch.int64)
        labels = torch.empty(g.n_nodes, dtype=torch.int64)
        counts = torch.empty(g.n_graphs, dtype=torch.int32)
        if g.perm is None:
            with torch.cuda.device(self.dev):
                _lib.check(self.lib.mpn_labels_reference_batched(g.ref, self.act.data_ptr(), labels.data_ptr(), counts.data_ptr(),
                                                                 self.ws.data_ptr(), self.ws.numel(), self.stream))
            return labels, counts.long()
        # unsorted batch: each graph's active edges in the caller's order, numbered on the host graph by graph
        s, d = self.caller_order_active()
        gid = g.node_gid[s].long()
        order = torch.sort(gid, stable=True).indices
        n0 = g.graph_nptr.long()[gid[order]]
        s_h = (s[order] - n0).to(torch.int32).cpu()
        d_h = (d[order] - n0).to(torch.int32).cpu()
        e_ptr = [0] + torch.bincount(gid, minlength=g.n_graphs).cumsum(0).tolist()
        nptr = g.graph_nptr.tolist()
        nc = C.c_int32(0)
        for k in range(g.n_graphs):
            e0, e1 = e_ptr[k], e_ptr[k + 1]
            _lib.check(self.lib.mpn_labels_reference_host(s_h[e0:].data_ptr(), d_h[e0:].data_ptr(), e1 - e0, nptr[k + 1] - nptr[k],
                                                          labels[nptr[k]:].data_ptr(), C.byref(nc)))
            counts[k] = nc.value
        return labels, counts.long()

    def labels_canonical(self):
        lab = torch.empty(self.g.n_nodes, dtype=torch.int32, device=self.dev)
        ncomp = C.c_int32(0)
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.mpn_scc_labels(self.g.ref, self.act.data_ptr(), lab.data_ptr(), C.byref(ncomp),
                                               self.ws.data_ptr(), self.ws.numel(), self.stream))
        return lab, int(ncomp.value)


def compute_SCC_and_Clusters(G, n_nodes):
    """utils.py:30-52.  ``G`` is anything with ``.edges`` (an nx.DiGraph) or an iterable / array of (u, v) pairs in
    insertion order.  Returns (ID_pred int64 CPU tensor [n_nodes], n_components)."""
    edges = list(G.edges) if hasattr(G, "edges") else G
    arr = np.asarray(edges, dtype=np.int32).reshape(-1, 2)
    s, d = np.ascontiguousarray(arr[:, 0]), np.ascontiguousarray(arr[:, 1])
    labels = torch.empty(int(n_nodes), dtype=torch.int64)
    ncomp = C.c_int32(0)
    _lib.check(_lib.lib().mpn_labels_reference_host(s.ctypes.data, d.ctypes.data, int(arr.shape[0]), int(n_nodes),
                                                    labels.data_ptr(), C.byref(ncomp)))
    return labels, int(ncomp.value)


def _active_tuple_list(data, predictions):
    idx = torch.nonzero(predictions.reshape(-1) != 0, as_tuple=False).reshape(-1)
    ei = data.edge_index[:, idx].cpu().numpy()
    return list(zip(ei[0].tolist(), ei[1].tolist()))


def remove_edges_single_direction(active_edges, predictions, edge_list, data=None):
    """CUTTING (utils.py:125-142): returns (new_predictions (a clone), new_active_edge_list)."""
    if data is None:
        raise TypeError("the B200 remove_edges_single_direction needs data=<graph> (edge_index on the device)")
    p = _Post(data, predictions)
    with torch.cuda.device(p.dev):
        _lib.check(p.lib.mpn_cut(p.g.ref, p.act.data_ptr(), p.ws.data_ptr(), p.ws.numel(), p.stream))
    new_pred = p.predictions(predictions)
    return new_pred, _active_tuple_list(data, new_pred)


def pruning(graph_obj, edges_out, probs, predicted_active_edges, num_cameras):
    """PRUNING (utils.py:144-339).  Returns [] when no node violates the flow constraint initially
    (utils.py:184-188), else the new prediction vector (a new tensor)."""
    p = _Post(graph_obj, edges_out, probs)
    changed, rounds = C.c_int32(0), C.c_int32(0)
    with torch.cuda.device(p.dev):
        _lib.check(p.lib.mpn_prune(p.g.ref, p.act.data_ptr(), p.prob_ptr, p.prob_stride, int(num_cameras), C.byref(changed),
                                   C.byref(rounds), p.ws.data_ptr(), p.ws.numel(), p.stream))
    if not changed.value:
        return []
    return p.predictions(edges_out)


def splitting(ID_pred, predictions, preds_prob, edge_list, data_batch, predicted_act_edges, num_cameras):
    """SPLITTING (utils.py:54-123).  Mutates ``predictions`` in place like the reference and returns it."""
    p = _Post(data_batch, predictions, preds_prob)
    rounds = C.c_int32(0)
    with torch.cuda.device(p.dev):
        _lib.check(p.lib.mpn_split(p.g.ref, p.act.data_ptr(), p.prob_ptr, p.prob_stride, int(num_cameras), C.byref(rounds),
                                   p.ws.data_ptr(), p.ws.numel(), p.stream))
    predictions.copy_(p.predictions(predictions).reshape(predictions.shape))
    return predictions


def split_stats():
    """SPLITTING of this thread's last ``splitting`` / ``post_processing`` / ``post_processing_batched`` call (mpn_split_last_stats):
    dict with the number of active edges that carried a tied probability value, rounds / dropped values, off-lowest steps, the mode
    that ran and ``host_order_graphs``, the number of graphs that took the reference order on the host (0 or 1 for one graph).
    After a batched call the counts are summed over the graphs."""
    out = (C.c_int64 * 4)()
    _lib.lib().mpn_split_last_stats(C.cast(out, C.c_void_p))
    return {"tied_edges": int(out[0]), "rounds": int(out[1]), "off_lowest_steps": int(out[2]),
            "mode": "reference_order_host" if out[3] else "device_rounds", "host_order_graphs": int(out[3])}


def post_processing(num_cameras, ID_pred, predicted_active_edges, predictions, edge_list, CONFIG, data, preds_prob,
                    numbering='reference', verbose=False):
    """inference.post_processing (inference.py:70-169): CUT -> PRUNE -> CUT -> SPLIT, then SCC labels.

    Returns (ID_pred: int64 CPU tensor [N], predictions: int64 [E] on the device).  ``numbering='reference'``
    reproduces the reference's label integers (host Tarjan over the few active edges); ``'canonical'`` labels each
    cluster with its smallest node id and stays on the device until the final copy.

    SPLITTING is exact under probability ties (utils.py:96-98 removes every edge with the dropped value, which couples the
    clusters that share it): ties are detected on the device; without one every oversized cluster drops its minimum in the same
    round on the device, with one the components SPLITTING can touch follow the reference's own order (csrc/split_exact.cu).
    ``split_stats()`` tells which ran.
    """
    flags = _stage_flags(CONFIG)
    if flags == 0:
        return ID_pred, predictions
    p = _Post(data, predictions, preds_prob)
    lab = torch.empty(p.g.n_nodes, dtype=torch.int32, device=p.dev)
    ncomp, changed = C.c_int32(0), C.c_int32(0)
    with torch.cuda.device(p.dev):
        _lib.check(p.lib.mpn_post_processing(p.g.ref, p.act.data_ptr(), p.prob_ptr, p.prob_stride, int(num_cameras), flags,
                                             lab.data_ptr(), C.byref(ncomp), C.byref(changed), p.ws.data_ptr(),
                                             p.ws.numel(), p.stream))
    new_pred = p.predictions(predictions).reshape(predictions.shape)
    if flags == _lib.POST_SPLIT:
        predictions.copy_(new_pred)                           # splitting mutates its argument in place (utils.py:98)
        new_pred = predictions
    if numbering == 'reference':
        ID, n = p.labels_reference()
    elif numbering == 'canonical':
        ID, n = lab.cpu().long(), int(ncomp.value)
    else:
        raise ValueError("numbering must be 'reference' or 'canonical'")
    if verbose:
        print('# CC = ' + str(n))
    return ID, new_pred


def _graph_count(data):
    """Number of graphs the batch carries, read without touching the device: a cached ``data.mpn_graph`` or ``data.ptr``."""
    pre = getattr(data, "mpn_graph", None)
    if pre is not None:
        return int(pre.n_graphs)
    ptr = getattr(data, "ptr", None)
    return 1 if ptr is None else int(ptr.numel()) - 1


def _cameras_per_graph(num_cameras, n_graphs):
    """``num_cameras`` as a list of n_graphs ints >= 1: one int for every graph, or one per graph (sequence / 1-D array / tensor)."""
    if isinstance(num_cameras, torch.Tensor):
        if num_cameras.dim() > 1:
            raise ValueError("num_cameras must be an int or a 1-D sequence with one entry per graph")
        vals = num_cameras.detach().cpu().reshape(-1).tolist() if num_cameras.dim() == 1 else [num_cameras.item()] * n_graphs
    elif isinstance(num_cameras, (int, np.integer)) and not isinstance(num_cameras, bool):
        vals = [int(num_cameras)] * n_graphs
    else:
        try:
            vals = np.asarray(num_cameras).reshape(-1).tolist() if np.ndim(num_cameras) == 1 else None
        except (TypeError, ValueError):
            vals = None
        if vals is None:
            raise ValueError("num_cameras must be an int or a 1-D sequence with one entry per graph")
    if len(vals) != n_graphs:
        raise ValueError("num_cameras has %d entries for a batch of %d graphs" % (len(vals), n_graphs))
    out = []
    for v in vals:
        try:
            ok = not isinstance(v, bool) and float(v).is_integer() and 1 <= v < 2 ** 31
        except (TypeError, ValueError):
            ok = False
        if not ok:
            raise ValueError("every num_cameras entry must be an integer >= 1, got %r" % (v,))
        out.append(int(v))
    return out


def post_processing_batched(num_cameras, predictions, CONFIG, data, preds_prob, numbering='reference', verbose=False):
    """``post_processing`` for every graph of a batch in one call (new; the reference loops over graphs, inference.py:475-497).

    ``data`` carries the batch as the batched forward takes it: ``data.ptr`` (G+1 node offsets) or a cached ``data.mpn_graph``;
    ``predictions`` [E] (uint8 / int64) and ``preds_prob`` ([E,2] softmax or [E] prob1) as ``post_processing`` takes them, e.g.
    ``MOTMPNet.last_pred`` / ``last_prob1`` of a batched forward with ``fuse_decisions=True``.  ``num_cameras``: an int for every
    graph or one int >= 1 per graph.  ``CONFIG`` is fixed up in place as in ``post_processing``.

    Returns (ID_pred int64 CPU [N], predictions (a new device tensor, the caller's dtype and shape), n_components int64 CPU [G]).
    For every graph g the slices ``ID_pred[ptr[g]:ptr[g+1]]`` (numbered from 0) and ``predictions`` of its edges equal what
    ``post_processing(num_cameras[g], ...)`` returns for that graph alone; with all three flags off, ID_pred holds each graph's SCC
    labels of the active edges.  ``split_stats()`` sums over the graphs and reports ``host_order_graphs``.
    """
    if numbering not in ('reference', 'canonical'):
        raise ValueError("numbering must be 'reference' or 'canonical'")
    n_graphs = _graph_count(data)
    cams = _cameras_per_graph(num_cameras, n_graphs)
    flags = _stage_flags(CONFIG)
    p = _Post(data, predictions, preds_prob)
    if p.g.n_graphs != n_graphs:
        raise ValueError("data.ptr describes %d graphs, its cached graph tables %d" % (n_graphs, p.g.n_graphs))
    ncam = torch.tensor(cams, dtype=torch.int32).to(p.dev)
    lab = torch.empty(p.g.n_nodes, dtype=torch.int32, device=p.dev)
    ncomp = torch.empty(max(1, n_graphs), dtype=torch.int32)
    with torch.cuda.device(p.dev):
        _lib.check(p.lib.mpn_post_processing_batched(p.g.ref, p.act.data_ptr(), p.prob_ptr, p.prob_stride, ncam.data_ptr(), flags,
                                                     lab.data_ptr(), ncomp.data_ptr(), p.ws.data_ptr(), p.ws.numel(), p.stream))
    new_pred = p.predictions(predictions).reshape(predictions.shape)
    if numbering == 'reference':
        ID, n = p.labels_reference_batched()
    else:
        ID, n = lab.cpu().long(), ncomp.long()
    if verbose:
        print('# CC = ' + ' '.join(str(v) for v in n.tolist()))
    return ID, new_pred, n
