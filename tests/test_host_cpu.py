"""CPU-side checks: the C-ABI library loads and exports every declared symbol; host logic that needs no GPU."""
import copy
import os
import re

import pytest
import torch

import gcn_mtmc_b200 as m
from oracle import mpn_oracle as mo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = m._lib.lib()
    header = open(os.path.join(ROOT, "include", "mpn_b200.h")).read()
    declared = set(re.findall(r"\b(mpn_[a-z0-9_]+)\s*\(", header))
    declared -= {"mpn_graph", "mpn_weights", "mpn_fwd_plan"}
    assert len(declared) >= 25
    for name in sorted(declared):
        assert hasattr(lib, name), "symbol %s declared in include/mpn_b200.h is not exported" % name
    assert set(m._lib.EXPORTED_SYMBOLS) == declared
    assert lib.mpn_abi_version() == m._lib.ABI_VERSION == 6


def test_pdl_switch_defaults_on():
    """Programmatic dependent launch is compiled in and on by default; mpn_set_pdl(0/1) is the A/B switch of the tools."""
    lib = m._lib.lib()
    assert lib.mpn_set_pdl(-1) == 2                   # 1 = off, 2 = on
    assert lib.mpn_set_pdl(0) == 1 and lib.mpn_set_pdl(-1) == 1 and lib.mpn_set_pdl(1) == 2


def test_no_device_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(m._lib.MpnError):
        m._lib.require_device(0)
    net = m.MOTMPNet(copy.deepcopy(mo.shipped_model_params(1, 1, 64, (48,))), None, "resnet101").eval()
    x, ei, _, _ = mo.synth_graph(20, 2, 1, D=64)

    class D:
        pass
    d = D(); d.x, d.edge_index, d.edge_attr = x, ei, torch.zeros(ei.shape[1], 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(d)


def test_state_dict_layout_matches_reference_names():
    p = mo.shipped_model_params()
    net = m.MOTMPNet(copy.deepcopy(p), None, "resnet101")
    sd = mo.init_weights(p, "resnet101", 0)
    assert list(net.state_dict().keys()) == list(sd.keys())
    net.load_state_dict(sd, strict=True)
    assert sum(v.numel() for v in net.state_dict().values()) == 2697750          # SURVEY.md section 8b
    # the constructor mutates the params dict exactly like the reference (models/mpn.py:169)
    q = mo.shipped_model_params()
    m.MOTMPNet(q, None, "resnet101")
    assert "node_in_dim" in q["encoder_feats_dict"]["edges"]


def test_unsupported_configs_raise():
    p = mo.shipped_model_params()
    p["node_agg_fn"] = "median"                       # the reference's own check (models/mpn.py:193)
    with pytest.raises(AssertionError):
        m.MOTMPNet(p, None, "resnet101")
    for agg in ("mean", "max", "sum"):                # all three aggregators of models/mpn.py:196-202 are supported
        p = mo.shipped_model_params()
        p["node_agg_fn"] = agg
        assert m.MOTMPNet(p, None, "resnet101")._node_agg == {"sum": 0, "mean": 1, "max": 2}[agg]
    for re_n, re_e, edge_in, node_in in [(True, False, 132, 68), (False, True, 72, 36), (True, True, 136, 68)]:
        p = mo.shipped_model_params()                 # reattach_initial_* (models/mpn.py:207-215): the MLP input widths follow
        p["reattach_initial_nodes"], p["reattach_initial_edges"] = re_n, re_e
        net = m.MOTMPNet(p, None, "resnet101")
        sd = net.state_dict()
        assert sd["MPNet.edge_model.edge_mlp.fc_layers.0.weight"].shape == (4, edge_in)
        assert sd["MPNet.node_model.node_mlp.fc_layers.0.weight"].shape == (32, node_in)
    p = mo.shipped_model_params()
    p["edge_model_feats_dict"]["fc_dims"] = [8]
    with pytest.raises(NotImplementedError):
        m.MOTMPNet(p, None, "resnet101")


def test_host_reference_numbering_matches_oracle():
    import numpy as np
    from oracle import postproc_oracle as po
    rng = np.random.default_rng(3)
    for _ in range(30):
        n = int(rng.integers(4, 60))
        k = int(rng.integers(0, 5 * n))
        s, d = rng.integers(0, n, k), rng.integers(0, n, k)
        keep = s != d
        key = np.unique(s[keep] * n + d[keep])
        key = key[rng.permutation(key.size)]
        s, d = key // n, key % n
        ref, nref = po.scc_labels_reference(s, d, np.ones(s.size), n)
        lab, nc = m.compute_SCC_and_Clusters(list(zip(s.tolist(), d.tolist())), n)
        assert nc == nref and np.array_equal(lab.numpy(), ref)


def test_stream_and_sharded_post_refuse_cpu():
    """The throughput pipeline and the sharded post-processing are CUDA-only like the rest of the product path."""
    from types import SimpleNamespace
    net = m.MOTMPNet(copy.deepcopy(mo.shipped_model_params(1, 1, 64, (48,))), None, "resnet101").eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.GraphStream(net, "cpu")
    with pytest.raises(ValueError):
        m.GraphStream(net, "cuda:0", depth=0)
    g = SimpleNamespace(n_edges=4, perm=None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.CudaPostOps().compact(g, torch.ones(4, dtype=torch.uint8), torch.rand(4))


def test_split_exact_host_matches_the_oracle_under_ties():
    """mpn_split_exact_host (product, C++: the reference's order with per-component recomputation) against the independent plain-C oracle of the reference's SPLITTING order
    (oracle/postproc_oracle.c::po_split_sequential, itself pinned against the Python statement mirror), on graphs with heavily
    tied probabilities and on a 3 k-node planted graph.  Host pointers only: runs without a GPU."""
    import ctypes as C
    import numpy as np
    from oracle import postproc_c as pc
    from oracle import postproc_oracle as po
    lib = m._lib.lib()

    def host_split(src, dst, act, prob, cams, n_nodes):
        a = np.flatnonzero(act)
        s32, d32 = np.ascontiguousarray(src[a], dtype=np.int32), np.ascontiguousarray(dst[a], dtype=np.int32)
        p32 = np.ascontiguousarray(prob[a], dtype=np.float32)
        keep = np.empty(a.size, dtype=np.uint8)
        stats = (C.c_int64 * 4)()
        m._lib.check(lib.mpn_split_exact_host(s32.ctypes.data, d32.ctypes.data, p32.ctypes.data, a.size, n_nodes, cams,
                                              keep.ctypes.data, C.cast(stats, C.c_void_p)))
        out = np.array(act, dtype=np.int64, copy=True)
        out[a[keep == 0]] = 0
        return out, int(stats[0])

    rng = np.random.default_rng(17)
    checked = 0
    for trial in range(600):
        n, cams = int(rng.integers(8, 40)), int(rng.integers(2, 5))
        cam = np.sort(rng.integers(0, cams, n))
        s, d = np.nonzero(cam[:, None] != cam[None, :])
        keep = rng.random(s.size) < rng.uniform(0.4, 1.0)
        s, d = s[keep], d[keep]
        if s.size == 0:
            continue
        q = 10 ** (1 + trial % 3)
        prob = (np.round(rng.random(s.size) * q) / q).astype(np.float32)
        pred = (prob > 0.5).astype(np.int64)
        start = po.cut_sequential(s, d, pred) if trial % 2 else pred
        got, _ = host_split(s, d, start, prob, cams, n)
        assert np.array_equal(got, pc.split_sequential(s, d, start, prob, cams, n)), trial
        checked += 1
    assert checked > 450
    src, dst, prob, pred, _ = po.planted_prediction_graph(3000, 6, 1, n_extra_per_node=6.0, flip_on=0.05, flip_off=0.03, single_dir=0.05)
    act = pc.cut(src, dst, pred, 3000)
    act, _ = pc.prune(src, dst, act, prob, 6, 3000)
    act = pc.cut(src, dst, act, 3000)
    got, steps = host_split(src, dst, act, prob, 6, 3000)
    assert steps > 0 and np.array_equal(got, pc.split_sequential(src, dst, act, prob, 6, 3000))
    with pytest.raises(m._lib.MpnError):
        m._lib.check(lib.mpn_split_exact_host(None, None, None, 3, 10, 4, None, None))


def test_split_exact_host_200k_nodes_zero_differing_decisions():
    """mpn_split_exact_host on the 200 k-node graph of tests/test_zz_c_oracle_gpu.py (0.9 M active edges, 1568 tied values, 44
    steps off the lowest label) against the stored result of the C statement-order oracle (tests/golden/make_split200k.py,
    11 minutes of po_split_sequential): zero differing decisions, the reference's label integers."""
    import ctypes as C
    import hashlib
    import numpy as np
    from oracle import postproc_c as pc
    from oracle import postproc_oracle as po
    from tests._util import GOLDEN
    g = np.load(os.path.join(GOLDEN, "split200k_sequential.npz"))
    n_nodes, cams, seed = [int(v) for v in g["spec"]]
    src, dst, prob, pred, _ = po.planted_prediction_graph(n_nodes, cams, seed, n_extra_per_node=6.0, flip_on=0.05, flip_off=0.03,
                                                          single_dir=0.05)
    act = pc.cut(src, dst, pred, n_nodes)
    act, _ = pc.prune(src, dst, act, prob, cams, n_nodes)
    act = pc.cut(src, dst, act, n_nodes)
    a = np.flatnonzero(act)
    assert a.size == int(g["n_start_active"][0])
    ref = np.zeros(src.size, dtype=np.int64)
    ref[a] = np.unpackbits(g["final_bits"])[:a.size]
    s32, d32 = np.ascontiguousarray(src[a], dtype=np.int32), np.ascontiguousarray(dst[a], dtype=np.int32)
    p32 = np.ascontiguousarray(prob[a], dtype=np.float32)
    keep = np.empty(a.size, dtype=np.uint8)
    stats = (C.c_int64 * 4)()
    m._lib.check(m._lib.lib().mpn_split_exact_host(s32.ctypes.data, d32.ctypes.data, p32.ctypes.data, a.size, n_nodes, cams,
                                                   keep.ctypes.data, C.cast(stats, C.c_void_p)))
    got = act.copy()
    got[a[keep == 0]] = 0
    assert int((got != ref).sum()) == 0
    assert stats[0] > 8000 and stats[1] > 0                      # dropped values; steps on a label other than the lowest
    lab, _ = pc.scc_labels(src, dst, got, n_nodes)
    assert hashlib.sha256(np.ascontiguousarray(lab, dtype=np.int64).tobytes()).digest() == g["labels_sha256"].tobytes()
    assert int((pc.split(src, dst, act, prob, cams, n_nodes) != ref).sum()) > 0       # all-clusters-per-round differs here


def test_host_numbering_equals_networkx_on_random_digraphs():
    """mpn_labels_reference_host against the library the reference calls (utils.py:31: sorted(nx.strongly_connected_components(G),
    key=len), then the nodes without an active edge in index order, utils.py:34-42), on random digraphs of up to 2000 nodes."""
    import ctypes as C
    import numpy as np
    nx = pytest.importorskip("networkx")
    lib = m._lib.lib()
    rng = np.random.default_rng(4)
    for trial in range(25):
        n = int(rng.integers(50, 2000))
        e = int(rng.integers(1, 4 * n))
        s, d = rng.integers(0, n, e), rng.integers(0, n, e)
        keep = s != d
        s, d = s[keep], d[keep]
        if s.size == 0:
            continue
        sccs = sorted(nx.strongly_connected_components(nx.DiGraph(list(zip(s.tolist(), d.tolist())))), key=len)
        expect = np.full(n, -1, dtype=np.int64)
        for i, c in enumerate(sccs):
            expect[list(c)] = i
        k = len(sccs)
        for i in range(n):
            if expect[i] < 0:
                expect[i] = k
                k += 1
        s32, d32 = np.ascontiguousarray(s, dtype=np.int32), np.ascontiguousarray(d, dtype=np.int32)
        lab = np.empty(n, dtype=np.int64)
        nc = C.c_int32(0)
        m._lib.check(lib.mpn_labels_reference_host(s32.ctypes.data, d32.ctypes.data, s.size, n, lab.ctypes.data, C.byref(nc)))
        assert nc.value == k and np.array_equal(lab, expect), trial


def test_shared_gram_every_pair_computed_exactly_once():
    """The pair-ownership rule of the shared symmetric Gram (csrc/kernels.h GeShare; the kernels' own functions compiled for the
    host): for every world size and ragged row blocks, each unordered pair of nodes is computed by exactly one rank, a rank only
    claims pairs whose row it owns, and the ranks' shares of the cross-block pairs are balanced."""
    import ctypes as C
    import numpy as np
    lib = m._lib.lib()
    rng = np.random.default_rng(11)
    for world in range(2, 9):
        for trial in range(4):
            n = int(rng.integers(world * 3, 90))
            cuts = np.sort(rng.choice(np.arange(1, n), size=world - 1, replace=False)) if trial else np.arange(1, world) * (n // world)
            blk = np.r_[0, cuts, n].astype(np.int32)
            owner = np.searchsorted(blk, np.arange(n), side="right") - 1
            claimed = np.zeros((n, n), dtype=np.int32)            # claimed[r, c]: ranks that compute pair {r, c} as (row r, column c)
            out = (C.c_int32 * 2)()
            for rank in range(world):
                for c in range(n):
                    got = lib.mpn_shared_gram_row_range(rank, world, blk.ctypes.data, c, out)
                    assert got == owner[c]
                    lo, hi = max(out[0], blk[rank]), min(out[1], blk[rank + 1])
                    if hi > lo:
                        claimed[lo:hi, c] += 1
            both = claimed + claimed.T                            # pair {r, c} computed as (r, c) or as (c, r)
            off = ~np.eye(n, dtype=bool)
            assert np.all(both[off] == 1), (world, blk)
            assert np.all(np.diag(claimed) == 0)
            work = np.array([claimed[blk[r]:blk[r + 1]].sum() for r in range(world)])
            if trial == 0 and n % world == 0:                     # equal blocks: equal shares (antipodal blocks are split in half)
                assert work.max() - work.min() <= n, (world, work)
    assert lib.mpn_shared_gram_row_range(0, 0, None, 0, None) == -1


def test_unpack_decisions_and_block_cover_host_logic():
    """Host-only pieces of the multi-GPU / stream paths: the bit-mask decisions unpack in np.packbits(bitorder='little') order
    (what mpn_pack_decisions writes: bit e & 31 of word e >> 5), and the row-block check that gates the shared symmetric Gram."""
    import numpy as np
    rng = np.random.default_rng(3)
    for n in (1, 31, 32, 33, 1000):
        pred = (rng.random(n) < 0.4).astype(np.uint8)
        words = np.zeros(4 * ((n + 31) // 32), dtype=np.uint8)
        packed = np.packbits(pred, bitorder="little")
        words[:packed.size] = packed
        assert np.array_equal(m.unpack_decisions(words, n), pred)
        assert np.array_equal(m.unpack_decisions(torch.from_numpy(words), n), pred)
    sh = m.ShardedMPN(None, fused=False)
    assert sh._blocks_cover([(0, 5), (5, 9)], 2, 9)
    assert sh._blocks_cover([(0, 5), (5, 9)], 2, 9)               # cached answer
    assert not sh._blocks_cover([(0, 5), (6, 9)], 2, 9)           # hole
    assert not sh._blocks_cover([(0, 5), (5, 9)], 2, 10)          # does not reach the last node
    assert not sh._blocks_cover([(0, 5), (5, 5), (5, 9)], 3, 9)   # empty block
    assert not sh._blocks_cover([(0, 9)], 2, 9)                   # one block per rank


def test_bench_dump_outputs_sample_and_format(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 .npy files; per-edge arrays at the same seeded, sorted edge sample every run."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_EDGES", 64)
    gen = torch.Generator().manual_seed(2)
    E = 1000
    res = {"classified_edges": [torch.randn(E, 2, generator=gen) for _ in range(2)], "h": torch.randn(30, 32, generator=gen),
           "pred": (torch.rand(E, generator=gen) < 0.5).to(torch.uint8), "prob1": torch.rand(E, generator=gen),
           "edge_attr": torch.randn(E, 2, generator=gen)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["classified_edges.npy", "edge_attr.npy", "edge_ids.npy", "h.npy", "pred.npy", "prob1.npy"]
    got = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    ids = got["edge_ids"].astype(np.int64)
    assert ids.size == 64 and np.all(np.diff(ids) > 0) and ids[-1] < E
    assert np.array_equal(got["classified_edges"], torch.stack(res["classified_edges"]).numpy()[:, ids])
    assert np.array_equal(got["pred"], res["pred"].numpy()[ids].astype(np.float32))
    assert np.array_equal(got["prob1"], res["prob1"].numpy()[ids]) and np.array_equal(got["h"], res["h"].numpy())
    assert np.array_equal(got["edge_attr"], res["edge_attr"].numpy()[ids])
    for n in names:
        assert (tmp_path / "a" / n).read_bytes() == (tmp_path / "b" / n).read_bytes()
