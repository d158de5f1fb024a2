"""What inference.py:383-451 does per graph besides the edge list (SURVEY.md section 8f rows 1 and 4), on the device:

  normalize_columns    F.normalize(node_embeds_g, p=2, dim=0), one graph or every graph of a batch  inference.py:403-404
  edge_labels          the ground-truth edge labels (an O(E*N) Python comprehension)  inference.py:446-450
  pack_reid_features / load_packed_features
                       the reference keeps ONE pickle per tracklet (libs/reid_feature_extraction.py:176-184) and loads them one
                       by one, each followed by its own ``.cuda()`` (libs/dataset.py:298-307, inference.py:399): here the
                       tracklets of a sequence live in one packed file that reaches the device with a single pinned H->D copy.
"""
import ctypes as C
import json
import os
import pickle

import numpy as np
import torch

from . import _lib
from .graph import TrackletGraph, current_stream_ptr, graph_for, host_node_ptr, node_features, workspace


def normalize_columns(x: torch.Tensor, out: torch.Tensor = None, ptr=None) -> torch.Tensor:
    """``F.normalize(x, p=2, dim=0)``: every feature column scaled to unit L2 norm over the nodes (eps 1e-12).
    ``ptr``: G+1 node offsets of a batch (PyG ``Batch.ptr``): every graph's rows ``x[ptr[g]:ptr[g+1]]`` are normalised on
    their own, as inference.py:403-404 does inside the loop over graphs, in one kernel.
    ``x`` may be fp32, fp16 or bf16 (16-bit features are read in place); the result is always fp32, equal to the one on
    ``x.float()``.  ``out``: a contiguous fp32 tensor of x's shape on x's device (``out=x`` normalises an fp32 x in place)."""
    if not x.is_cuda:
        raise RuntimeError("normalize_columns needs a CUDA tensor: the B200 path has no CPU fallback")
    if x.dim() != 2:
        raise ValueError("x must be [N, D]")
    if out is not None and (out.dtype != torch.float32 or out.shape != x.shape or out.device != x.device
                            or not out.is_contiguous()):
        raise ValueError("out must be a contiguous float32 tensor of x's shape %s on %s (got %s %s on %s)"
                         % (tuple(x.shape), x.device, out.dtype, tuple(out.shape), out.device))
    nptr = host_node_ptr(ptr, x.shape[0]) if ptr is not None else None
    x, x_kind = node_features(x)
    out = torch.empty(x.shape, dtype=torch.float32, device=x.device) if out is None else out
    L = _lib.lib()
    stream = current_stream_ptr(x.device)
    with torch.cuda.device(x.device):
        if nptr is not None and nptr.size > 2:
            pinned = torch.from_numpy(nptr.astype(np.int32)).pin_memory()
            gptr = pinned.to(x.device, non_blocking=True)
            _lib.check(L.mpn_normalize_columns_batched_x(x.data_ptr(), x_kind, x.shape[0], x.shape[1], gptr.data_ptr(),
                                                         nptr.size - 1, out.data_ptr(), None, 0, stream))
        else:
            ws = workspace("normalize_columns", x.device, L.mpn_normalize_columns_workspace_bytes(x.shape[1]))
            _lib.check(L.mpn_normalize_columns_x(x.data_ptr(), x_kind, x.shape[0], x.shape[1], out.data_ptr(), ws.data_ptr(),
                                                 ws.numel(), stream))
    return out


def edge_labels(node_labels, edge_index: torch.Tensor = None, graph: TrackletGraph = None, data=None) -> torch.Tensor:
    """float32 [E]: 1 where both endpoints carry the same identity label, else 0 — in the caller's edge order."""
    g = graph
    if g is None:
        if edge_index is None or not edge_index.is_cuda:
            raise RuntimeError("edge_labels needs a CUDA edge_index or a TrackletGraph: the B200 path has no CPU fallback")
        g = graph_for(data, edge_index, int(len(node_labels)))
    lab = torch.as_tensor(np.array(node_labels) if not torch.is_tensor(node_labels) else node_labels)
    lab = lab.to(device=g.device, dtype=torch.int64).reshape(-1).contiguous()
    if lab.numel() != g.n_cols:
        raise ValueError("node_labels must have one entry per node")
    out = torch.empty(g.n_edges, dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        _lib.check(_lib.lib().mpn_edge_labels(g.ref, lab.data_ptr(), out.data_ptr(), current_stream_ptr(g.device)))
    if g.perm is not None:
        unsorted = torch.empty_like(out)
        unsorted[g.perm] = out
        out = unsorted
    return out


# ------------------------------------------------------------------------------------------------ packed ReID features
MAGIC = b"MPNFEAT1"
# header dtype -> element type of the feature matrix (bfloat16 is stored as its raw 16-bit words)
_PACKED_DTYPES = {"float32": torch.float32, "float16": torch.float16, "bfloat16": torch.bfloat16}


def reid_feature_path(root, scenario, id_cam, track_id, file, cnn_model_name):
    """The per-tracklet pickle of the reference (libs/dataset.py:298-299)."""
    return os.path.join(root, scenario, 'c' + str(int(id_cam)).zfill(3), str(int(track_id)).zfill(4),
                        file + '_' + cnn_model_name + '.pkl')


def pack_reid_features(path, features, cam_ids, track_ids, dtype="float32"):
    """Write one packed file: header (JSON) + id_cam int64[N] + id int64[N] + features [N,D] (row-major, 4096-byte aligned so
    the matrix can be mapped).  ``features``: [N,D] array / tensor, or a list of per-tracklet vectors.  ``dtype``: element type
    stored, ``"float32"``, ``"float16"`` or ``"bfloat16"`` (or the torch dtype); fp32 values are rounded to nearest even.
    Half-width files halve the bytes read and copied to the device; the features are then exact 16-bit values."""
    name = str(dtype).replace("torch.", "")
    if name not in _PACKED_DTYPES:
        raise ValueError("dtype must be float32, float16 or bfloat16 (got %r)" % (dtype,))
    if isinstance(features, (list, tuple)):                       # (.float(): numpy has no bfloat16; the widening is exact)
        features = np.stack([np.asarray(f.detach().cpu().float() if torch.is_tensor(f) else f, dtype=np.float32).reshape(-1)
                             for f in features])
    x = np.ascontiguousarray(features.detach().cpu().float().numpy() if torch.is_tensor(features) else features, dtype=np.float32)
    if name != "float32":                                        # 16-bit: raw words of the rounded values
        x = torch.from_numpy(x).to(_PACKED_DTYPES[name]).view(torch.int16).numpy()
    cam = np.ascontiguousarray(np.asarray(cam_ids), dtype=np.int64).reshape(-1)
    tid = np.ascontiguousarray(np.asarray(track_ids), dtype=np.int64).reshape(-1)
    if x.ndim != 2 or not (x.shape[0] == cam.size == tid.size):
        raise ValueError("features must be [N,D] with one camera id and one track id per row")
    header = json.dumps({"n": int(x.shape[0]), "d": int(x.shape[1]), "dtype": name}).encode()
    pre = len(MAGIC) + 8 + len(header) + cam.nbytes + tid.nbytes
    pad = (-pre) % 4096
    with open(path, "wb") as f:
        f.write(MAGIC)
        f.write(np.int64(len(header)).tobytes())
        f.write(header)
        f.write(cam.tobytes())
        f.write(tid.tobytes())
        f.write(b"\0" * pad)
        f.write(x.tobytes())


def pack_reid_features_from_pickles(path, root, scenario, file, cnn_model_name, cam_ids, track_ids):
    """Convert the reference's layout (one pickled CPU tensor per tracklet) into one packed file."""
    feats = []
    for c, t in zip(cam_ids, track_ids):
        with open(reid_feature_path(root, scenario, c, t, file, cnn_model_name), "rb") as fin:
            v = pickle.load(fin)                                   # libs/dataset.py:302-303
        feats.append(v.numpy() if torch.is_tensor(v) else np.asarray(v))
    pack_reid_features(path, feats, cam_ids, track_ids)


def read_packed_features(path):
    """Host view of a packed file: (features [N,D] memory-mapped, id_cam int64 [N], id int64 [N]).  The features keep the
    file's element type: a numpy float32 / float16 array, or for bfloat16 (which numpy lacks) a torch.bfloat16 tensor over a
    copy-on-write mapping of the file."""
    with open(path, "rb") as f:
        if f.read(len(MAGIC)) != MAGIC:
            raise ValueError("%s is not a packed ReID feature file" % path)
        hlen = int(np.frombuffer(f.read(8), dtype=np.int64)[0])
        h = json.loads(f.read(hlen).decode())
        n, d = int(h["n"]), int(h["d"])
        name = h.get("dtype", "float32")
        if name not in _PACKED_DTYPES:
            raise ValueError("%s: unknown feature dtype %r in the header" % (path, name))
        cam = np.frombuffer(f.read(8 * n), dtype=np.int64).copy()
        tid = np.frombuffer(f.read(8 * n), dtype=np.int64).copy()
        pre = len(MAGIC) + 8 + hlen + 16 * n
        off = pre + ((-pre) % 4096)
    if name == "bfloat16":
        words = np.memmap(path, dtype=np.int16, mode="c", offset=off, shape=(n, d)) if n else np.zeros((0, d), dtype=np.int16)
        return torch.from_numpy(words).view(torch.bfloat16), cam, tid
    npt = np.float32 if name == "float32" else np.float16
    x = np.memmap(path, dtype=npt, mode="r", offset=off, shape=(n, d)) if n else np.zeros((0, d), dtype=npt)
    return x, cam, tid


def load_packed_features(path, device, l2norm: bool = False):
    """One pinned staging buffer, one H->D copy (the reference does N pickle loads + N ``.cuda()`` calls, inference.py:383-401).
    Returns (x [N,D] on the device in the file's dtype, id_cam int64 [N] host array, id int64 [N] host array); ``l2norm``
    applies inference.py:403-404 on the device (in place for an fp32 file; a 16-bit file gives a new fp32 tensor)."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("load_packed_features copies to a CUDA device: the B200 path has no CPU fallback")
    x, cam, tid = read_packed_features(path)
    dt = x.dtype if torch.is_tensor(x) else torch.from_numpy(np.empty(0, dtype=x.dtype)).dtype
    pinned = torch.empty(x.shape, dtype=dt).pin_memory()
    if torch.is_tensor(x):
        pinned.copy_(x)
    else:
        np.copyto(pinned.numpy(), x)
    xd = torch.empty(x.shape, dtype=dt, device=dev)
    xd.copy_(pinned, non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()                    # the staging buffer is released on return
    if l2norm and xd.shape[0]:
        xd = normalize_columns(xd, out=xd if dt == torch.float32 else None)
    return xd, cam, tid
