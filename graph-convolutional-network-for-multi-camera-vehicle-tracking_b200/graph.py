"""Device-side graph tables (int32 CSR + task table) for a tracklet graph.

The reference indexes node features with ``row, col = edge_index`` (models/mpn.py:44,82) on the int64
[2,E] tensor built by ``torch.cartesian_prod`` per camera (inference.py:407-413).  The kernels use an int32
CSR over ``row`` (the node at which messages are aggregated, models/mpn.py:97-99) plus a table of *tasks*
(runs of at most ``chunk`` edges of one row) that warps iterate over.
"""
import ctypes as C

import torch

from . import _lib

_WORKSPACES = {}
_SCOPE = []              # workspace_scope() tags (innermost last)


class workspace_scope:
    """``with workspace_scope(tag):`` gives the calls inside their own scratch buffers (keyed by tag).  A captured CUDA graph bakes
    the addresses of its scratch memory in, so every capture runs under a tag of its own: buffers that another caller could grow
    (= free) must never end up inside a graph (GraphStream._capture, _GraphedForward)."""

    def __init__(self, tag: str):
        self.tag = str(tag)

    def __enter__(self):
        _SCOPE.append(self.tag)
        return self

    def __exit__(self, *exc):
        _SCOPE.pop()
        return False


def workspace(kind: str, device: torch.device, nbytes: int) -> torch.Tensor:
    """Grow-only uint8 scratch buffer per (kind[, scope], device); torch owns the memory, the C ABI only borrows it.

    Contract (also in INTEGRATION.md / include/mpn_b200.h): ONE host thread and ONE CUDA stream per device use the library at a
    time.  The buffers are shared by consecutive calls; growing one frees the old allocation, which is safe only because the
    caching allocator defers the reuse of a block to the stream that last used it — the caller's single compute stream."""
    key = (kind if not _SCOPE else kind + "#" + _SCOPE[-1], device.index)
    buf = _WORKSPACES.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = None
        _WORKSPACES.pop(key, None)
        buf = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        _WORKSPACES[key] = buf
    return buf


def release_scope(tag: str):
    """Drops the scratch buffers of a scope (a captured graph that used them has been destroyed)."""
    for key in [k for k in _WORKSPACES if k[0].endswith("#" + str(tag))]:
        _WORKSPACES.pop(key, None)


def current_stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class _NoContext:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_CONTEXT = _NoContext()


def _on_device(dev):
    """``torch.cuda.device(dev)`` only when ``dev`` is not already current (the guard costs several microseconds per call)."""
    return _NO_CONTEXT if dev.index is None or dev.index == torch.cuda.current_device() else torch.cuda.device(dev)


_FLAG_SLOTS = {}


def _flag_slot(dev):
    """(device int, pinned host int) pair for one deferred graph build; recycled by validate()."""
    free = _FLAG_SLOTS.setdefault(str(dev), [])
    if free:
        return free.pop()
    return (torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32).pin_memory())


def _release_flag_slot(dev, slot):
    _FLAG_SLOTS.setdefault(str(dev), []).append(slot)


def choose_chunk(n_edges: int) -> int:
    """Edges per task: aim for >= 4 tasks per resident warp slot of a 148-SM part, within [32, 1024]."""
    target = max(1, n_edges // (148 * 32 * 4))
    chunk = 32
    while chunk * 2 <= target and chunk < 1024:
        chunk *= 2
    return chunk


def host_node_ptr(ptr, n_nodes: int):
    """The G+1 node offsets of a batch (PyG ``Batch.ptr``: host sequence, numpy array or tensor; a CUDA tensor is copied to the
    host once) as an int64 numpy array, checked to run strictly increasing from 0 to ``n_nodes``."""
    import numpy as np
    p = np.asarray(ptr.detach().cpu() if isinstance(ptr, torch.Tensor) else ptr)
    if p.ndim != 1 or p.size < 2 or not np.issubdtype(p.dtype, np.integer):
        raise ValueError("ptr must be strictly increasing from 0 to num_nodes")
    p = p.astype(np.int64)
    if p[0] != 0 or p[-1] != n_nodes or np.any(p[1:] <= p[:-1]):
        raise ValueError("ptr must be strictly increasing from 0 to num_nodes")
    return p


class TrackletGraph:
    """CSR + task tables on the device.  ``perm`` is None when the caller's edge order is already (row, col)-sorted,
    otherwise ``sorted_edge = original_edge[perm]``."""

    def __init__(self, edge_index: torch.Tensor, num_nodes: int, chunk: int = None, row_offset: int = 0,
                 n_rows: int = None, ptr: torch.Tensor = None, validate: str = "sync"):
        """``validate='sync'`` (default) checks the edge list before returning (one host round trip; unsorted training-style
        graphs are sorted transparently).  ``validate='deferred'`` returns without synchronising: the check result travels to
        pinned host memory behind the build and ``.validate()`` (called by the user after the pipeline has been enqueued, and by
        post_processing) raises then; an invalid list leaves an empty graph on the device, never inconsistent tables."""
        if not edge_index.is_cuda:
            raise RuntimeError("TrackletGraph needs a CUDA edge_index: the B200 path has no CPU fallback")
        if edge_index.dim() != 2 or edge_index.shape[0] != 2:
            raise ValueError("edge_index must have shape [2, E]")
        dev = edge_index.device
        _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
        self.device = dev
        self.n_cols = int(num_nodes)
        self.n_nodes = int(n_rows if n_rows is not None else num_nodes)
        self.row_offset = int(row_offset)
        self.n_edges = int(edge_index.shape[1])
        self.chunk = int(chunk or choose_chunk(self.n_edges))
        self.max_tasks = self.n_edges // self.chunk + self.n_nodes
        ptrs = self._alloc_tables(dev)
        self.perm = None
        # batched small graphs: ptr = node offsets [G+1] (PyG ``Batch.ptr``); BatchNorm statistics are then per graph
        self.n_graphs, self.node_gid, self.graph_nptr, self.max_graph_nodes = 1, None, None, 0
        if ptr is not None and ptr.numel() > 2:
            if row_offset != 0 or self.n_nodes != self.n_cols:
                raise ValueError("batched graphs cannot be row-sharded")
            nptr = ptr.to(device=dev, dtype=torch.int64).contiguous()
            if int(nptr[0]) != 0 or int(nptr[-1]) != self.n_nodes or bool((nptr[1:] <= nptr[:-1]).any()):
                raise ValueError("ptr must be strictly increasing from 0 to num_nodes")
            self.n_graphs = nptr.numel() - 1
            self.node_gid = torch.repeat_interleave(torch.arange(self.n_graphs, device=dev, dtype=torch.int32),
                                                    (nptr[1:] - nptr[:-1])).contiguous()
            self.graph_nptr = nptr.to(torch.int32).contiguous()
            row_g, col_g = self.node_gid[edge_index[0].long()], self.node_gid[edge_index[1].long()]
            if bool((row_g != col_g).any()):
                raise ValueError("batched graphs must be block-diagonal: an edge connects two different graphs")
            e_per_graph = torch.bincount(row_g.long(), minlength=self.n_graphs)
            self.max_graph_nodes = int((nptr[1:] - nptr[:-1]).max())
            if int(e_per_graph.min()) < 2 or int((nptr[1:] - nptr[:-1]).min()) < 2:
                raise ValueError("every graph of a batch needs at least 2 nodes and 2 edges (BatchNorm over one value "
                                 "raises in the reference)")
        self.struct = _lib.MpnGraph(self.n_nodes, self.n_cols, self.row_offset, self.chunk, self.n_edges, self.max_tasks, 0,
                                    ptrs[0], ptrs[4], ptrs[1], ptrs[3], ptrs[2], self.n_graphs, self.max_graph_nodes,
                                    self.node_gid.data_ptr() if self.node_gid is not None else None,
                                    self.graph_nptr.data_ptr() if self.graph_nptr is not None else None)
        ei = edge_index
        if ei.dtype != torch.int64:
            ei = ei.long()
        ei = ei.contiguous()
        stream = current_stream_ptr(dev)
        self._pending = None
        if validate not in ("sync", "deferred"):
            raise ValueError("validate must be 'sync' or 'deferred'")
        if validate == "deferred":
            slot = _flag_slot(dev)
            with _on_device(dev):
                _lib.check(_lib.lib().mpn_graph_build_deferred(C.byref(self.struct), ei.data_ptr(), slot[0].data_ptr(),
                                                               slot[1].data_ptr(), stream))
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            self._pending = (slot, ev)
            self._keepalive = ei
            return
        with torch.cuda.device(dev):
            try:
                _lib.check(_lib.lib().mpn_graph_build(C.byref(self.struct), ei.data_ptr(), stream))
            except _lib.UnsortedEdgeIndex:
                # training-style graphs (train.py:295-302) are not row-sorted: sort once, remember the permutation
                key = ei[0] * self.n_cols + ei[1]
                skey, perm = torch.sort(key, stable=True)
                if self.n_edges > 1 and bool((skey[1:] == skey[:-1]).any()):
                    raise ValueError("edge_index contains duplicate edges")
                self.perm = perm
                ei = ei[:, perm].contiguous()
                _lib.check(_lib.lib().mpn_graph_build(C.byref(self.struct), ei.data_ptr(), stream))
        self._keepalive = ei

    # The five int32 tables live in ONE allocation (building a graph is on the host's critical path of every step: one
    # torch.empty instead of five, no fill kernel); .rowptr / .taskptr / .n_tasks / .task_row / .col are views made on first use.
    _SECTIONS = {"rowptr": 0, "taskptr": 1, "n_tasks": 2, "task_row": 3, "col": 4}

    def _alloc_tables(self, dev):
        n1 = self.n_nodes + 1
        sizes = (n1, n1, 1, max(self.max_tasks, 1), max(self.n_edges, 1))
        offs, o = [], 0
        for n in sizes:
            offs.append(o)
            o += (n + 3) & ~3                                   # 16-byte aligned sections
        self._tables = torch.empty(o, dtype=torch.int32, device=dev)
        self._sections = tuple(zip(offs, sizes))
        base = self._tables.data_ptr()
        return tuple(base + 4 * off for off in offs)

    def __getattr__(self, name):                                # only reached when the attribute is not set
        idx = TrackletGraph._SECTIONS.get(name)
        sections = self.__dict__.get("_sections")
        if idx is None or sections is None:
            raise AttributeError(name)
        off, n = sections[idx]
        view = self._tables[off:off + n]
        self.__dict__[name] = view
        return view

    def validate(self):
        """Deferred validation: wait for the build, then raise what ``validate='sync'`` would have raised.  No-op otherwise."""
        if getattr(self, "_pending", None) is None:
            return self
        slot, ev = self._pending
        ev.synchronize()
        flags = int(slot[1].item())
        self._pending = None
        _release_flag_slot(self.device, slot)
        if flags & 2:
            raise _lib.MpnError(_lib.MPN_ERR_INVALID, "edge_index has node ids outside [row_offset, row_offset+n_nodes) x [0, n_cols)")
        if flags & 1:
            raise _lib.UnsortedEdgeIndex(_lib.MPN_ERR_UNSORTED, "edge_index is not strictly (row, col)-sorted (unsorted or duplicate "
                                         "edges): build the graph with validate='sync' to have it sorted")
        return self

    @classmethod
    def from_cameras(cls, cam_ids, device, chunk: int = None, materialize_edge_index: bool = False, row_block=None, ptr=None):
        """Dense cross-camera graph built on the device from the per-node camera ids (inference.py:407-414), without
        the int64 edge_index ever crossing PCIe or being read: 4 B/edge written instead of 16 B read + 4 B written.
        ``cam_ids``: host sequence / array / CPU tensor, nodes grouped by camera in ascending camera order
        (dataset.py:279-281).  ``materialize_edge_index`` also writes the reference's int64 [2,E] tensor (``.edge_index``).
        ``row_block=(n0, n1)`` builds only the rows of one shard (column ids stay global).
        ``ptr``: G+1 node offsets of a batch of graphs (PyG ``Batch.ptr``); with G > 1 every graph gets its own dense
        cross-camera rows (the per-graph edge_index offset by ptr[g], concatenated) and per-graph BatchNorm statistics, as
        ``TrackletGraph(edge_index, N, ptr=ptr)``; cameras are grouped in ascending order within each graph.  Does not
        synchronise (a CUDA ``ptr`` is read on the host once).
        """
        import numpy as np
        cam = np.asarray(cam_ids.cpu() if isinstance(cam_ids, torch.Tensor) else cam_ids).reshape(-1)
        if ptr is not None:
            nptr = host_node_ptr(ptr, cam.size)
            if nptr.size > 2:
                if row_block is not None:
                    raise ValueError("batched graphs cannot be row-sharded")
                return cls._from_cameras_batched(cam, nptr, device, chunk, materialize_edge_index)
        if cam.size < 2 or np.any(cam[1:] < cam[:-1]):
            raise ValueError("from_cameras needs nodes grouped by ascending camera id (as the reference dataset orders them)")
        starts = np.flatnonzero(np.r_[True, cam[1:] != cam[:-1]])
        cam_ptr = np.ascontiguousarray(np.r_[starts, cam.size].astype(np.int32))
        n_cams = int(cam_ptr.size - 1)
        dev = torch.device(device)
        _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
        L = _lib.lib()
        self = object.__new__(cls)
        n0, n1 = (0, int(cam.size)) if row_block is None else (int(row_block[0]), int(row_block[1]))
        self.device, self.n_cols, self.n_nodes, self.row_offset = dev, int(cam.size), n1 - n0, n0
        self.n_edges = int(L.mpn_cross_camera_block_edges(cam_ptr.ctypes.data, n_cams, n0, n1 - n0))
        if self.n_edges < 0:
            raise ValueError("bad row block")
        self.chunk = int(chunk or choose_chunk(self.n_edges))
        self.max_tasks = self.n_edges // self.chunk + self.n_nodes
        ptrs = self._alloc_tables(dev)
        self.perm = None
        self.n_graphs, self.node_gid, self.graph_nptr, self.max_graph_nodes = 1, None, None, 0
        self.edge_index = torch.empty(2, self.n_edges, dtype=torch.int64, device=dev) if materialize_edge_index else None
        self.struct = _lib.MpnGraph(self.n_nodes, self.n_cols, self.row_offset, self.chunk, self.n_edges, self.max_tasks, 0,
                                    ptrs[0], ptrs[4], ptrs[1], ptrs[3], ptrs[2], 1, 0, None, None)
        with _on_device(dev):
            _lib.check(L.mpn_graph_build_cross_camera(C.byref(self.struct), cam_ptr.ctypes.data, n_cams,
                                                      self.edge_index.data_ptr() if materialize_edge_index else None,
                                                      current_stream_ptr(dev)))
        self._keepalive = self.edge_index
        return self

    @classmethod
    def _from_cameras_batched(cls, cam, nptr, device, chunk, materialize_edge_index):
        import numpy as np
        n, n_graphs = int(cam.size), int(nptr.size - 1)
        first = np.zeros(n, dtype=bool)
        first[nptr[:-1]] = True                                   # first node of every graph
        if np.any((cam[1:] < cam[:-1]) & ~first[1:]):
            raise ValueError("from_cameras needs nodes grouped by ascending camera id within every graph (as the reference "
                             "dataset orders them)")
        # one segment per (graph, camera); layout = [seg_ebase int64 [S+1] | seg_ptr [S+1] | graph_seg [G+1]] (int32 words)
        starts = np.flatnonzero(first | np.r_[True, cam[1:] != cam[:-1]])
        n_segs = int(starts.size)
        n_ints = 2 * (n_segs + 1) + (n_segs + 1) + (n_graphs + 1)
        host = np.empty(n_ints, dtype=np.int32)
        seg_ebase = host[:2 * (n_segs + 1)].view(np.int64)
        seg_ptr = host[2 * (n_segs + 1):3 * (n_segs + 1)]
        graph_seg = host[3 * (n_segs + 1):]
        seg_ptr[:-1], seg_ptr[-1] = starts, n
        graph_seg[:] = np.searchsorted(starts, nptr)
        L = _lib.lib()
        E = int(L.mpn_cross_camera_batched_layout(seg_ptr.ctypes.data, n_segs, graph_seg.ctypes.data, n_graphs,
                                                  seg_ebase.ctypes.data))
        if E < 0:
            raise ValueError("malformed camera layout")
        e_per_graph = seg_ebase[graph_seg[1:]] - seg_ebase[graph_seg[:-1]]
        n_per_graph = nptr[1:] - nptr[:-1]
        if int(e_per_graph.min()) < 2 or int(n_per_graph.min()) < 2:
            raise ValueError("every graph of a batch needs at least 2 nodes and 2 edges (BatchNorm over one value "
                             "raises in the reference)")
        if E >= (1 << 31):
            raise ValueError("a batch of cross-camera graphs needs fewer than 2^31 edges (%d)" % E)
        dev = torch.device(device)
        _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
        self = object.__new__(cls)
        self.device, self.n_cols, self.n_nodes, self.row_offset, self.n_edges = dev, n, n, 0, E
        self.chunk = int(chunk or choose_chunk(E))
        self.max_tasks = E // self.chunk + n
        ptrs = self._alloc_tables(dev)
        self.perm = None
        self.n_graphs, self.max_graph_nodes = n_graphs, int(n_per_graph.max())
        # node_gid [N] | graph_nptr [G+1] | layout, in one allocation; the layout arrives in ONE copy from pinned memory
        o_nptr = (n + 3) & ~3
        o_lay = o_nptr + ((n_graphs + 1 + 3) & ~3)
        aux = torch.empty(o_lay + n_ints, dtype=torch.int32, device=dev)
        pinned = torch.empty(n_ints, dtype=torch.int32, pin_memory=True)
        pinned.numpy()[:] = host
        aux[o_lay:].copy_(pinned, non_blocking=True)
        self.node_gid, self.graph_nptr = aux[:n], aux[o_nptr:o_nptr + n_graphs + 1]
        base = aux.data_ptr() + 4 * o_lay
        self.edge_index = torch.empty(2, E, dtype=torch.int64, device=dev) if materialize_edge_index else None
        self.struct = _lib.MpnGraph(n, n, 0, self.chunk, E, self.max_tasks, 0, ptrs[0], ptrs[4], ptrs[1], ptrs[3], ptrs[2],
                                    n_graphs, self.max_graph_nodes, self.node_gid.data_ptr(), self.graph_nptr.data_ptr())
        with _on_device(dev):
            _lib.check(L.mpn_graph_build_cross_camera_batched(C.byref(self.struct), base + 8 * (n_segs + 1), n_segs,
                                                              base + 12 * (n_segs + 1), base,
                                                              self.edge_index.data_ptr() if materialize_edge_index else None,
                                                              current_stream_ptr(dev)))
        self._keepalive = (self.edge_index, aux, pinned)         # pinned: the staging buffer outlives its copy
        return self

    @property
    def ref(self):
        return C.byref(self.struct)


def graph_for(data, edge_index: torch.Tensor, num_nodes: int) -> TrackletGraph:
    """Graph tables cached on the data object (one graph per batch in the reference driver, inference.py:375)."""
    ptr = getattr(data, "ptr", None) if data is not None else None
    key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, int(num_nodes),
           None if ptr is None else (ptr.data_ptr(), ptr._version))
    cached = getattr(data, "_mpn_b200_graph", None) if data is not None else None
    if cached is not None and cached[0] == key:
        return cached[1]
    g = TrackletGraph(edge_index, num_nodes, ptr=ptr)
    if data is not None:
        try:
            object.__setattr__(data, "_mpn_b200_graph", (key, g))
        except Exception:
            pass
    return g
