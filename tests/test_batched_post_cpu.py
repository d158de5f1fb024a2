"""post_processing_batched: argument checks that need no GPU, and the coupling-trap case of tests/test_batched_post_gpu.py checked
on the CPU (the C oracle tells the union-as-one-graph answer from the per-graph answers, so the GPU test cannot pass by accident)."""
import numpy as np
import pytest
import torch

from oracle import postproc_c as pc
from tests._util import Data

TRAP_CAMERAS = 2


def coupling_trap_case():
    """Two graphs of one batch that share a probability value, with no tie inside either graph.

    Graph A: 3 nodes, all 6 directed edges active (one SCC of 3 > 2 cameras); SPLITTING drops its smallest value 0.61 first.
    Graph B: 2 nodes, both directions active (an SCC of 2, not oversized); its edge 1 -> 0 carries 0.61 as well.
    Per graph (the reference's loop over graphs) B is never touched.  As ONE graph, dropping 0.61 in A also removes B's 1 -> 0
    (utils.py:96-98 compares against every edge of the graph) and splits B in two.
    Returns [(src, dst, prob1, pred, n_nodes)] per graph, graph-local ids, edges (row, col)-sorted."""
    a_src = np.array([0, 0, 1, 1, 2, 2], dtype=np.int64)
    a_dst = np.array([1, 2, 0, 2, 0, 1], dtype=np.int64)
    a_prob = np.array([0.61, 0.64, 0.66, 0.62, 0.65, 0.63], dtype=np.float32)
    b_src = np.array([0, 1], dtype=np.int64)
    b_dst = np.array([1, 0], dtype=np.int64)
    b_prob = np.array([0.9, 0.61], dtype=np.float32)
    return [(a_src, a_dst, a_prob, np.ones(6, dtype=np.int64), 3), (b_src, b_dst, b_prob, np.ones(2, dtype=np.int64), 2)]


def union_of(graphs):
    """The graphs of a batch as one disjoint-union graph: (src, dst, prob1, pred, n_nodes, node offsets)."""
    ptr = np.cumsum([0] + [g[4] for g in graphs])
    src = np.concatenate([g[0] + ptr[k] for k, g in enumerate(graphs)])
    dst = np.concatenate([g[1] + ptr[k] for k, g in enumerate(graphs)])
    return (src, dst, np.concatenate([g[2] for g in graphs]), np.concatenate([g[3] for g in graphs]), int(ptr[-1]), ptr)


def test_coupling_trap_separates_union_from_per_graph_answers():
    graphs = coupling_trap_case()
    src, dst, prob, pred, n, ptr = union_of(graphs)
    union_act = pc.split_sequential(src, dst, pred, prob, TRAP_CAMERAS, n)
    union_lab, _ = pc.scc_labels(src, dst, union_act, n)
    per_act, per_lab = [], []
    for s, d, p, a, ng in graphs:
        act = pc.split_sequential(s, d, a, p, TRAP_CAMERAS, ng)
        per_act.append(act)
        per_lab.append(pc.scc_labels(s, d, act, ng)[0])
    assert not np.array_equal(union_act, np.concatenate(per_act))
    assert per_act[1].tolist() == [1, 1] and union_act[6:].tolist() == [1, 0]          # only the union touches graph B
    assert len(set(union_lab[3:].tolist())) == 2 and len(set(per_lab[1].tolist())) == 1
    # no value is shared by two edges inside one graph: a per-graph engine has no tie to resolve
    for s, d, p, a, ng in graphs:
        assert np.unique(p).size == p.size


def _cpu_batch():
    graphs = coupling_trap_case()
    src, dst, prob, pred, n, ptr = union_of(graphs)
    data = Data(x=torch.zeros(n, 1), edge_index=torch.from_numpy(np.stack([src, dst])), ptr=torch.from_numpy(ptr))
    return data, torch.from_numpy(pred), torch.from_numpy(prob)


@pytest.mark.parametrize("cams", [[2], [2, 2, 2], 0, [2, 0], [2, -1], [2, 2.5], [[2, 2]], "two"])
def test_bad_num_cameras_raise_value_error_before_device_work(cams):
    import gcn_mtmc_b200 as m
    data, pred, prob = _cpu_batch()
    with pytest.raises(ValueError):
        m.post_processing_batched(cams, pred, {"CUTTING": True, "PRUNING": True, "SPLITTING": True}, data, prob)


@pytest.mark.parametrize("cams", [2, [2, 3], np.array([2, 3]), torch.tensor([2, 3])])
def test_cpu_tensors_have_no_fallback(cams):
    import gcn_mtmc_b200 as m
    data, pred, prob = _cpu_batch()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.post_processing_batched(cams, pred, {"CUTTING": True, "PRUNING": True, "SPLITTING": True}, data, prob)
