"""Batched cross-camera graphs built from camera ids (TrackletGraph.from_cameras(cam, ptr=)) against the route through the offset
reference edge_index (TrackletGraph(edge_index, N, ptr=)): identical tables, a bit-identical batched forward, identical
post-processing and edge labels; and normalize_columns(x, ptr=) against the per-graph call.  B200 only."""
import numpy as np
import pytest
import torch

from oracle import mpn_oracle as mo
from tests._util import Data

pytestmark = pytest.mark.gpu

FULL = {"CUTTING": True, "PRUNING": True, "SPLITTING": True}


@pytest.fixture(scope="module")
def m():
    import gcn_mtmc_b200 as mod
    mod._lib.require_device(0)
    return mod


def dev():
    return torch.device("cuda", 0)


def ragged_batch(seed):
    """Graphs of 3 / 4 / 5 / 8 cameras with unequal camera sizes and non-contiguous ids -> (cam_ids, ptr, cameras per graph)."""
    rng = np.random.default_rng(seed)
    specs = [[2, 5, 7], [0, 1, 2, 3], [1, 3, 4, 8, 9], list(range(8)), [2, 5, 7], [10, 11, 12, 13], [0, 6, 9]]
    cams = [np.repeat(ids, rng.integers(1, 40, size=len(ids))) for ids in specs]
    return np.concatenate(cams), np.cumsum([0] + [c.size for c in cams]), [len(s) for s in specs]


def uniform_batch(G, n, C):
    cam = np.tile(np.arange(n) * C // n, G)
    return cam, np.arange(G + 1) * n


def offset_edge_index(cam, ptr):
    """The reference's edge_index of every graph (inference.py:407-413), offset by the graph's first node and concatenated."""
    parts = [mo.cross_camera_edge_index(torch.from_numpy(cam[ptr[g]:ptr[g + 1]])) + int(ptr[g]) for g in range(ptr.size - 1)]
    return torch.cat(parts, dim=1).contiguous()


def edge_index_route(m, cam, ptr, chunk=None):
    ei = offset_edge_index(cam, ptr).to(dev())
    return ei, m.TrackletGraph(ei, cam.size, chunk=chunk, ptr=torch.from_numpy(ptr).to(dev()))


def assert_same_tables(a, b):
    torch.cuda.synchronize()
    for name in ("n_nodes", "n_cols", "n_edges", "chunk", "max_tasks", "n_graphs", "max_graph_nodes"):
        assert getattr(a, name) == getattr(b, name), name
    assert a.struct.layout_hint == b.struct.layout_hint
    for name in ("rowptr", "taskptr", "n_tasks"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    for name in ("node_gid", "graph_nptr"):                   # None for a single graph
        u, v = getattr(a, name), getattr(b, name)
        assert (u is None and v is None) if a.n_graphs == 1 else torch.equal(u, v), name
    assert torch.equal(a.col[:a.n_edges], b.col[:b.n_edges])
    nt = int(a.n_tasks.item())
    assert torch.equal(a.task_row[:nt], b.task_row[:nt])


@pytest.mark.parametrize("case", ["uniform", "ragged", "ragged_chunk64"])
def test_tables_equal_the_edge_index_route(m, case):
    cam, ptr = uniform_batch(16, 300, 4) if case == "uniform" else ragged_batch(1)[:2]
    chunk = 64 if case == "ragged_chunk64" else None
    ei, ref = edge_index_route(m, cam, ptr, chunk)
    g = m.TrackletGraph.from_cameras(cam, dev(), chunk=chunk, materialize_edge_index=True, ptr=ptr)
    assert_same_tables(g, ref)
    assert g.struct.layout_hint == 0 and g.n_graphs == ptr.size - 1
    assert torch.equal(g.edge_index, ei)


def test_ptr_forms_and_single_graph(m):
    cam, ptr, _ = ragged_batch(2)
    ref = m.TrackletGraph.from_cameras(cam, dev(), ptr=ptr)
    for p in (list(ptr), torch.from_numpy(ptr), torch.from_numpy(ptr).to(dev()).int()):
        assert_same_tables(m.TrackletGraph.from_cameras(torch.from_numpy(cam), dev(), ptr=p), ref)
    c1 = cam[ptr[3]:ptr[4]]                                    # one graph: exactly from_cameras(cam)
    one = m.TrackletGraph.from_cameras(c1, dev(), ptr=[0, c1.size], materialize_edge_index=True)
    alone = m.TrackletGraph.from_cameras(c1, dev(), materialize_edge_index=True)
    assert_same_tables(one, alone)
    assert one.struct.layout_hint == 1 and one.n_graphs == 1 and one.node_gid is None
    assert torch.equal(one.edge_index, alone.edge_index)


def test_build_does_not_synchronise(m):
    cam, ptr, _ = ragged_batch(3)
    m.TrackletGraph.from_cameras(cam, dev(), ptr=ptr)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        g = m.TrackletGraph.from_cameras(cam, dev(), ptr=ptr, materialize_edge_index=True)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert_same_tables(g, edge_index_route(m, cam, ptr)[1])


def forward_both_ways(m, net, x, cam, ptr):
    ei, _ = edge_index_route(m, cam, ptr)
    a = Data(x=x, edge_index=ei, ptr=torch.from_numpy(ptr).to(dev()), edge_attr=None)
    out_a, h_a = net(a)
    res_a = (out_a["classified_edges"][-1], h_a, net.last_pred, net.last_prob1, a.edge_attr)
    b = Data(x=x, mpn_graph=m.TrackletGraph.from_cameras(cam, dev(), ptr=ptr), edge_attr=None)
    out_b, h_b = net(b)
    res_b = (out_b["classified_edges"][-1], h_b, net.last_pred, net.last_prob1, b.edge_attr)
    return a, b, res_a, res_b


def test_forward_and_downstream_calls_are_identical(m):
    import bench
    cam, ptr, n_cams = ragged_batch(4)
    net = bench.make_model(dev())
    net.fuse_decisions = True
    x = torch.randn(cam.size, bench.FEAT_DIM, generator=torch.Generator(device=dev()).manual_seed(5), device=dev())
    x = m.normalize_columns(x, ptr=ptr)
    a, b, res_a, res_b = forward_both_ways(m, net, x, cam, ptr)
    for name, u, v in zip(("logits", "h", "last_pred", "last_prob1", "edge_attr"), res_a, res_b):
        assert u.shape == v.shape and torch.equal(u, v), name
    pred, prob = res_a[2], res_a[3]
    for numbering in ("reference", "canonical"):
        ID_a, P_a, nc_a = m.post_processing_batched(n_cams, pred.clone(), dict(FULL), a, prob, numbering=numbering)
        ID_b, P_b, nc_b = m.post_processing_batched(n_cams, pred.clone(), dict(FULL), b, prob, numbering=numbering)
        assert torch.equal(ID_a, ID_b) and torch.equal(P_a, P_b) and torch.equal(nc_a, nc_b), numbering
    labels = torch.from_numpy(np.random.default_rng(6).integers(0, 12, size=cam.size))
    ga = m.graph_for(a, a.edge_index, cam.size)
    assert torch.equal(m.edge_labels(labels, graph=ga), m.edge_labels(labels, graph=b.mpn_graph))


def test_configs2_size(m):
    """configs[2]: 2000 graphs x (300 nodes, 4 cameras, 67,500 edges)."""
    import bench
    G, n, C = 2000, 300, 4
    cam, ptr = uniform_batch(G, n, C)
    _, tmpl = bench.device_graph(n, C, 0, dev())
    E1 = tmpl.shape[1]
    ei = (tmpl[None] + (torch.arange(G, device=dev()) * n)[:, None, None]).permute(1, 0, 2).reshape(2, G * E1).contiguous()
    ptr_d = torch.from_numpy(ptr).to(dev())
    g = m.TrackletGraph.from_cameras(cam, dev(), ptr=ptr)
    assert_same_tables(g, m.TrackletGraph(ei, G * n, ptr=ptr_d))
    net = bench.make_model(dev())
    net.fuse_decisions = True
    x = torch.randn(G * n, bench.FEAT_DIM, generator=torch.Generator(device=dev()).manual_seed(3), device=dev())
    x = m.normalize_columns(x, ptr=ptr)
    net(Data(x=x, edge_index=ei, ptr=ptr_d, edge_attr=None))
    pred_a, prob_a = net.last_pred, net.last_prob1
    del ei
    net(Data(x=x, mpn_graph=g, edge_attr=None))
    assert torch.equal(net.last_pred, pred_a) and torch.equal(net.last_prob1, prob_a)


def ulp_distance(a, b):
    a, b = a.cpu().numpy().view(np.int32).astype(np.int64), b.cpu().numpy().view(np.int32).astype(np.int64)
    return np.abs(a - b).max()


@pytest.mark.parametrize("sizes, D", [
    ([1, 3, 5000, 2, 1, 40], 70),          # graphs of one node and a large graph next to small ones; D not a multiple of a slab
    ([300] * 64, 2048),                    # S02-shaped graphs at the reference's feature width
    ([4000, 3000], 256),                   # few large graphs: narrower slabs
])
def test_normalize_columns_per_graph(m, sizes, D):
    ptr = np.cumsum([0] + sizes)
    x = torch.randn(ptr[-1], D, generator=torch.Generator(device=dev()).manual_seed(D), device=dev())
    x[:, 5] = 0                                               # a zero column in every graph
    g0, g1 = ptr[-2], ptr[-1]
    x[g0:g1, 7] = 0                                           # and one in the last graph only
    out = m.normalize_columns(x, ptr=ptr)
    for g in range(len(sizes)):
        sl = x[ptr[g]:ptr[g + 1]].contiguous()
        o = out[ptr[g]:ptr[g + 1]]
        assert ulp_distance(o, m.normalize_columns(sl)) <= 1, g
        assert (o - torch.nn.functional.normalize(sl, p=2, dim=0)).abs().max().item() <= 2e-7, g
    assert not out[:, 5].any() and not out[g0:g1, 7].any() and out[:g0, 7].any()
    assert torch.equal(m.normalize_columns(x, ptr=torch.from_numpy(ptr).to(dev())), out)
    y = x.clone()
    assert m.normalize_columns(y, out=y, ptr=list(ptr)).data_ptr() == y.data_ptr()
    assert torch.equal(y, out)
