"""post_processing_batched: every graph of a batch gets, bit for bit, what post_processing gives it alone (which is itself pinned
against the unmodified reference), for every flag set, both numberings, under probability ties, at configs[2] scale and end to
end after the batched forward.  B200 only."""
import os

import numpy as np
import pytest
import torch

from oracle import postproc_c as pc
from oracle import postproc_oracle as po
from tests._util import GOLDEN, Data, same_partition
from tests.test_batched_post_cpu import TRAP_CAMERAS, coupling_trap_case, union_of
from tests.test_c_oracle import _ties_cases

pytestmark = pytest.mark.gpu

GOLDEN_CASES = ("post_n36_c3", "post_n40_c4", "post_n50_c4_clean", "post_n64_c4", "post_n90_c5", "post_n120_c4_noisy",
                "s02post_n300_c4")
FLAG_SETS = (("none", (False, False, False)), ("cut_only", (True, False, False)), ("prune_only", (False, True, False)),
             ("split_only", (False, False, True)), ("full", (True, True, True)))


@pytest.fixture(scope="module")
def m():
    import gcn_mtmc_b200 as mod
    mod._lib.require_device(0)
    return mod


def dev():
    return torch.device("cuda", 0)


def cfg_of(flags):
    return {"CUTTING": flags[0], "PRUNING": flags[1], "SPLITTING": flags[2]}


def make_batch(graphs):
    """graphs: [(src, dst, prob1, pred, n_nodes)] with graph-local ids -> (Data with ptr, pred, prob1, node ptr, edge ptr)."""
    src, dst, prob, pred, n, ptr = union_of(graphs)
    eptr = np.cumsum([0] + [g[0].size for g in graphs])
    data = Data(x=torch.zeros(n, 1, device=dev()), edge_index=torch.from_numpy(np.stack([src, dst])).to(dev()),
                ptr=torch.from_numpy(ptr).to(dev()))
    return data, torch.from_numpy(pred).to(dev()), torch.from_numpy(prob).to(dev()), ptr, eptr


def single(m, graph, cams, flags, numbering="reference"):
    """post_processing on one graph alone -> (ID numpy, predictions numpy, host-order mode)."""
    s, d, p, a, n = graph
    data = Data(x=torch.zeros(n, 1, device=dev()), edge_index=torch.from_numpy(np.stack([s, d])).to(dev()))
    ID, P = m.post_processing(cams, None, None, torch.from_numpy(a).to(dev()), None, cfg_of(flags), data,
                              torch.from_numpy(p).to(dev()), numbering=numbering)
    if ID is None:                                  # all flags off: post_processing hands ID_pred back untouched
        ID, _ = m.compute_SCC_and_Clusters(list(zip(s[a != 0].tolist(), d[a != 0].tolist())), n)
    host = m.split_stats()["mode"] == "reference_order_host" if flags[2] else False
    return ID.numpy(), P.cpu().numpy(), host


def check_per_graph(m, graphs, cams, flags, ID, P, nc, ptr, eptr, numbering="reference"):
    n_host = 0
    P = P.cpu().numpy()
    for k, g in enumerate(graphs):
        ID1, P1, host = single(m, g, cams[k], flags, numbering)
        n_host += host
        assert np.array_equal(P[eptr[k]:eptr[k + 1]], P1), (k, flags)
        lab = ID.numpy()[ptr[k]:ptr[k + 1]]
        assert np.array_equal(lab, ID1), (k, flags, numbering)       # canonical: smallest graph-local node id on both sides
        assert int(nc[k]) == np.unique(lab).size, (k, flags)
    return n_host


def load_golden(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    N, C = [int(v) for v in g["spec"][:2]]
    return g, (g["src"].astype(np.int64), g["dst"].astype(np.int64), g["prob1"], g["pred"].astype(np.int64), N), C


def test_reference_golden_mixed_camera_counts(m):
    cases = [load_golden(name) for name in GOLDEN_CASES]
    graphs, cams = [c[1] for c in cases], [c[2] for c in cases]
    assert sorted(set(cams)) == [3, 4, 5]
    data, pred, prob, ptr, eptr = make_batch(graphs)
    preds_prob = torch.stack([1 - prob, prob], dim=1)
    for tag, flags in FLAG_SETS:
        ID, P, nc = m.post_processing_batched(cams, pred.clone(), cfg_of(flags), data, preds_prob)
        assert ID.dtype == torch.int64 and not ID.is_cuda and P.is_cuda and P.dtype == torch.int64 and P.shape == pred.shape
        assert nc.dtype == torch.int64 and not nc.is_cuda and nc.shape == (len(graphs),)
        Pn = P.cpu().numpy()
        for k, (g, _, _) in enumerate(cases):
            want_p = g["pred"] if tag == "none" else g["pred_" + tag]
            want_l = g["labels_initial"] if tag == "none" else g["labels_" + tag]
            lab = ID.numpy()[ptr[k]:ptr[k + 1]]
            assert np.array_equal(Pn[eptr[k]:eptr[k + 1]], want_p), (GOLDEN_CASES[k], tag)
            assert np.array_equal(lab, want_l), (GOLDEN_CASES[k], tag)
            assert int(nc[k]) == int(want_l.max()) + 1
        IDc, Pc, ncc = m.post_processing_batched(torch.tensor(cams), pred.clone(), cfg_of(flags), data, preds_prob,
                                                 numbering="canonical")
        assert torch.equal(Pc, P) and torch.equal(ncc, nc)
        for k, (g, _, _) in enumerate(cases):
            want_l = g["labels_initial"] if tag == "none" else g["labels_" + tag]
            assert same_partition(IDc.numpy()[ptr[k]:ptr[k + 1]], want_l), (GOLDEN_CASES[k], tag)
    # one camera count for every graph: the C=3 and C=5 graphs no longer match their fixtures
    ID, P, _ = m.post_processing_batched(4, pred.clone(), cfg_of((True, True, True)), data, preds_prob)
    Pn = P.cpu().numpy()
    for k, (g, _, C) in enumerate(cases):
        same = np.array_equal(Pn[eptr[k]:eptr[k + 1]], g["pred_full"]) and np.array_equal(ID.numpy()[ptr[k]:ptr[k + 1]], g["labels_full"])
        assert same == (C == 4), GOLDEN_CASES[k]


def test_batch_of_one_graph_equals_post_processing(m):
    g, graph, C = load_golden("post_n64_c4")
    data, pred, prob, ptr, eptr = make_batch([graph])
    for numbering in ("reference", "canonical"):
        ID, P, nc = m.post_processing_batched([C], pred.clone(), cfg_of((True, True, True)), data, prob, numbering=numbering)
        ID1, P1, _ = single(m, graph, C, (True, True, True), numbering)
        assert np.array_equal(ID.numpy(), ID1) and np.array_equal(P.cpu().numpy(), P1) and nc.tolist() == [np.unique(ID1).size]


def test_ties_golden(m):
    cases = list(_ties_cases())
    graphs = [(s, d, p, a, n) for (_i, s, d, p, a, C, n, _ref) in cases]
    cams = [C for (_i, _s, _d, _p, _a, C, _n, _ref) in cases]
    data, pred, prob, ptr, eptr = make_batch(graphs)
    host = 0
    for tag, flags in (("full", (True, True, True)), ("split_only", (False, False, True)), ("prune_split", (False, True, True))):
        ID, P, nc = m.post_processing_batched(cams, pred.clone(), cfg_of(flags), data, prob)
        host += m.split_stats()["host_order_graphs"]
        Pn = P.cpu().numpy()
        for k, (i, _s, _d, _p, _a, _C, _n, ref) in enumerate(cases):
            assert np.array_equal(Pn[eptr[k]:eptr[k + 1]], ref["pred_" + tag]), (i, tag)
            assert np.array_equal(ID.numpy()[ptr[k]:ptr[k + 1]], ref["labels_" + tag]), (i, tag)
    assert host > 0


def test_cross_graph_coupling_trap(m):
    graphs = coupling_trap_case()
    src, dst, prob, pred, n, _ = union_of(graphs)
    union_act = pc.split_sequential(src, dst, pred, prob, TRAP_CAMERAS, n)
    per_act = [pc.split_sequential(s, d, a, p, TRAP_CAMERAS, ng) for (s, d, p, a, ng) in graphs]
    assert not np.array_equal(union_act, np.concatenate(per_act))      # the case tells the two answers apart
    data, pred_d, prob_d, ptr, eptr = make_batch(graphs)
    for flags in ((False, False, True), (True, False, True)):
        ID, P, nc = m.post_processing_batched(TRAP_CAMERAS, pred_d.clone(), cfg_of(flags), data, prob_d)
        assert m.split_stats()["host_order_graphs"] == 0
        assert np.array_equal(P.cpu().numpy(), np.concatenate(per_act))
        for k, (s, d, p, a, ng) in enumerate(graphs):
            assert np.array_equal(ID.numpy()[ptr[k]:ptr[k + 1]], pc.scc_labels(s, d, per_act[k], ng)[0])
        check_per_graph(m, graphs, [TRAP_CAMERAS] * 2, flags, ID, P, nc, ptr, eptr)


def test_mixed_modes_in_one_batch(m):
    ties = [(s, d, p, a, n, C) for (_i, s, d, p, a, C, n, _ref) in _ties_cases()]
    clean = [load_golden(name) for name in ("post_n50_c4_clean", "post_n64_c4", "s02post_n300_c4")]
    graphs = [t[:5] for t in ties[:5]] + [c[1] for c in clean] + [t[:5] for t in ties[5:]]
    cams = [t[5] for t in ties[:5]] + [c[2] for c in clean] + [t[5] for t in ties[5:]]
    data, pred, prob, ptr, eptr = make_batch(graphs)
    for flags in ((False, False, True), (True, True, True)):
        for numbering in ("reference", "canonical"):
            ID, P, nc = m.post_processing_batched(cams, pred.clone(), cfg_of(flags), data, prob, numbering=numbering)
            host = m.split_stats()["host_order_graphs"]
            n_host_single = check_per_graph(m, graphs, cams, flags, ID, P, nc, ptr, eptr, numbering)
            assert 0 < host < len(graphs) and host == n_host_single, (flags, host, n_host_single)


def test_configs2_scale_2000_planted_graphs(m):
    """2000 S02-shaped planted predicted graphs (300 nodes, 4 cameras, 67,500 edges each, distinct seeds) in one batch: every graph
    equals the single-graph post_processing, in both numberings; two batched runs are bit-identical."""
    G, n, C = 2000, 300, 4
    gen = [po.planted_prediction_graph(n, C, 20000 + k, dense=True) for k in range(G)]
    src, dst = gen[0][0], gen[0][1]
    assert src.size == 67500 and all(np.array_equal(g[0], src) and np.array_equal(g[1], dst) for g in gen[:3])
    E1 = src.size
    tmpl = torch.from_numpy(np.stack([src, dst])).to(dev())
    ei = (tmpl[None] + (torch.arange(G, device=dev()) * n)[:, None, None]).permute(1, 0, 2).reshape(2, G * E1).contiguous()
    ptr = torch.arange(G + 1, device=dev()) * n
    data = Data(x=torch.zeros(G * n, 1, device=dev()), edge_index=ei, ptr=ptr)
    pred = torch.from_numpy(np.concatenate([g[3] for g in gen])).to(dev())
    prob = torch.from_numpy(np.concatenate([g[2] for g in gen])).to(dev())
    del gen
    one = Data(x=torch.zeros(n, 1, device=dev()), edge_index=tmpl)
    cfg = cfg_of((True, True, True))
    for numbering in ("reference", "canonical"):
        ID, P, nc = m.post_processing_batched(C, pred.clone(), dict(cfg), data, prob, numbering=numbering)
        ID2, P2, nc2 = m.post_processing_batched(C, pred.clone(), dict(cfg), data, prob, numbering=numbering)
        assert torch.equal(ID, ID2) and torch.equal(P, P2) and torch.equal(nc, nc2)
        for k in range(G):
            e0, e1 = k * E1, (k + 1) * E1
            ID1, P1 = m.post_processing(C, None, None, pred[e0:e1].clone(), None, dict(cfg), one, prob[e0:e1], numbering=numbering)
            assert torch.equal(P[e0:e1], P1), (k, numbering)
            assert torch.equal(ID[k * n:(k + 1) * n], ID1), (k, numbering)
            assert int(nc[k]) == torch.unique(ID1).numel()


def test_end_to_end_after_batched_forward(m):
    import bench
    G, n, C = 64, 300, 4
    net = bench.make_model(dev())
    net.fuse_decisions = True
    gen = torch.Generator(device=dev()).manual_seed(11)
    x = torch.randn(G, n, bench.FEAT_DIM, generator=gen, device=dev())
    x = torch.nn.functional.normalize(x, p=2, dim=1).reshape(G * n, bench.FEAT_DIM)
    _, tmpl = bench.device_graph(n, C, 0, dev())
    E1 = tmpl.shape[1]
    ei = (tmpl[None] + (torch.arange(G, device=dev()) * n)[:, None, None]).permute(1, 0, 2).reshape(2, G * E1).contiguous()
    b = bench.Batch()
    b.x, b.edge_index, b.num_nodes, b.ptr, b.edge_attr = x, ei, G * n, torch.arange(G + 1, device=dev()) * n, None
    net(b)
    pred, prob1 = net.last_pred, net.last_prob1
    assert pred.dtype == torch.uint8 and pred.numel() == G * E1
    one = Data(x=torch.zeros(n, 1, device=dev()), edge_index=tmpl)
    cfg = cfg_of((True, True, True))
    ID, P, nc = m.post_processing_batched(C, pred, dict(cfg), b, prob1)
    assert P.dtype == torch.uint8
    for k in range(G):
        e0, e1 = k * E1, (k + 1) * E1
        ID1, P1 = m.post_processing(C, None, None, pred[e0:e1].clone(), None, dict(cfg), one, prob1[e0:e1])
        assert torch.equal(P[e0:e1], P1) and torch.equal(ID[k * n:(k + 1) * n], ID1), k


def test_unsorted_batch(m):
    rng = np.random.default_rng(5)
    shuffled, cams = [], []
    for k, (N, C) in enumerate(((60, 4), (45, 3), (80, 5), (50, 4))):
        s, d, p, a, _ = po.planted_prediction_graph(N, C, 300 + k, n_extra_per_node=4.0, flip_on=0.06, flip_off=0.04, single_dir=0.03)
        o = rng.permutation(s.size)                       # each graph's edges stay together, in a shuffled order
        shuffled.append((s[o], d[o], p[o], a[o], N))
        cams.append(C)
    data, pred, prob, ptr, eptr = make_batch(shuffled)
    for flags in ((True, True, True), (False, False, True), (False, True, False)):
        for numbering in ("reference", "canonical"):
            ID, P, nc = m.post_processing_batched(cams, pred.clone(), cfg_of(flags), data, prob, numbering=numbering)
            assert m.graph_for(data, data.edge_index, data.num_nodes).perm is not None
            check_per_graph(m, shuffled, cams, flags, ID, P, nc, ptr, eptr, numbering)
