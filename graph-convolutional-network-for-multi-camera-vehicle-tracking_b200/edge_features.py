"""Initial edge features on the device (replaces inference.py:453-456)."""
import ctypes as C

import torch

from . import _lib
from .graph import TrackletGraph, current_stream_ptr, graph_for, node_features, workspace

USE_TENSOR_CORES = True


def edge_features(x: torch.Tensor, edge_index: torch.Tensor, graph: TrackletGraph = None, data=None,
                  use_tensor_cores: bool = None, out: torch.Tensor = None) -> torch.Tensor:
    """edge_attr[e] = [ ||x_r - x_c + 1e-6||_2 , 1 - cos(x_r, x_c) ], fp32 [E,2], in the caller's edge order.

    One Gram GEMM (3xTF32 tcgen05, or fp32 SIMT) plus a per-edge epilogue; the reference's two [E,2048] gathers
    (240 GB at N=4096) are never materialised.  ``out``: optional preallocated [E,2] result buffer.
    ``x`` may be fp32, fp16 or bf16: 16-bit features are read in place and give exactly the result of ``x.float()``.
    """
    if not x.is_cuda:
        raise RuntimeError("edge_features needs CUDA tensors: the B200 path has no CPU fallback")
    x, x_kind = node_features(x)
    g = graph if graph is not None else graph_for(data, edge_index, x.shape[0])
    if out is None:
        out = torch.empty(g.n_edges, 2, dtype=torch.float32, device=x.device)
    elif (out.shape != (g.n_edges, 2) or out.dtype != torch.float32 or out.device != x.device or not out.is_contiguous()
          or g.perm is not None):
        raise ValueError("out must be a contiguous fp32 [E,2] tensor on x's device (and the graph must be in the caller's order)")
    L = _lib.lib()
    need = L.mpn_edge_features_workspace_bytes(g.ref, x.shape[1])
    ws = workspace("edge_features", x.device, need)
    tc = USE_TENSOR_CORES if use_tensor_cores is None else use_tensor_cores
    with torch.cuda.device(x.device):
        _lib.check(L.mpn_edge_features_x(g.ref, x.data_ptr(), x_kind, x.shape[1], out.data_ptr(), int(bool(tc)), ws.data_ptr(),
                                         ws.numel(), current_stream_ptr(x.device)))
    if g.perm is not None:
        unsorted = torch.empty_like(out)
        unsorted[g.perm] = out
        out = unsorted
    return out
