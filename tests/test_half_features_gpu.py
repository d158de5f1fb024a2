"""fp16 / bf16 node features read in place: every output must equal, bit for bit, the same call on ``x.float()`` (the kernels
convert each element on load, which is exact, and keep every reduction's order).  B200 only."""
import copy

import numpy as np
import pytest
import torch

from oracle import mpn_oracle as mo
from tests._util import Data

pytestmark = pytest.mark.gpu

HALF = [torch.float16, torch.bfloat16]


@pytest.fixture(scope="module")
def m():
    import gcn_mtmc_b200 as mod
    mod._lib.require_device(0)
    return mod


def dev():
    return torch.device("cuda", 0)


def model(m, params, sd, fuse=True):
    net = m.MOTMPNet(copy.deepcopy(params), None, "resnet101")
    net.load_state_dict(sd, strict=True)
    net = net.to(dev()).eval()
    net.fuse_decisions = fuse
    return net


def half_pair(x, dt):
    """(16-bit x on the device, its exact fp32 widening on the device)."""
    xh = x.to(dev()).to(dt)
    return xh, xh.float()


def run(net, x, **kw):
    """Every output of one forward: logits, h, edge_attr, last_pred, last_prob1."""
    d = Data(x=x, **kw)
    out, h = net(d)
    torch.cuda.synchronize()
    return ([o.clone() for o in out["classified_edges"]], h.clone(), d.edge_attr.clone(),
            None if net.last_pred is None else net.last_pred.clone(), None if net.last_prob1 is None else net.last_prob1.clone())


def assert_same(a, b):
    la, ha, ea, pa, qa = a
    lb, hb, eb, pb, qb = b
    assert len(la) == len(lb) and all(torch.equal(u, v) for u, v in zip(la, lb)), "logits differ"
    assert torch.equal(ha, hb), "h differs"
    assert torch.equal(ea, eb), "edge_attr differs"
    assert (pa is None and pb is None) or torch.equal(pa, pb), "last_pred differs"
    assert (qa is None and qb is None) or torch.equal(qa, qb), "last_prob1 differs"


# ------------------------------------------------------------------------------------------------ edge features
@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
@pytest.mark.parametrize("case", ["dense_fused", "dense_staged_d4096", "thinned", "duplicates_and_zero_rows", "simt", "odd_d",
                                  "batched"])
def test_edge_features_equal_fp32_route(m, dt, case):
    D = {"dense_staged_d4096": 4096, "odd_d": 50}.get(case, 128)
    N, C = (300, 4) if case != "dense_staged_d4096" else (200, 3)
    x, ei, cam, _ = mo.synth_graph(N, C, 3, D=D, planted=True, noise=0.05)
    if case == "duplicates_and_zero_rows":                 # cancelling pairs reach the refine list; zero rows have no direction
        x[N // C] = x[0]                                   # first node of the next camera: the pair is an edge
        x[2 * N // C] = x[0] * (1 + 1e-3)
        x[7] = 0
        x[8] = 0
    if case == "thinned":                                  # not every row is "all columns but one gap": Gram + gather path
        ei = ei[:, torch.arange(ei.shape[1]) % 5 != 2].contiguous()
    xh, xf = half_pair(x, dt)
    tc = case != "simt"
    if case == "batched":
        cams, ptr = np.concatenate([np.arange(n) * c // n for n, c in ((40, 3), (75, 4), (9, 2))]), np.array([0, 40, 115, 124])
        xh, xf = xh[:124].contiguous(), xf[:124].contiguous()
        g = m.TrackletGraph.from_cameras(cams, dev(), ptr=ptr)
        a = m.edge_features(xh, None, graph=g, use_tensor_cores=tc)
        b = m.edge_features(xf, None, graph=g, use_tensor_cores=tc)
    else:
        eid = ei.to(dev())
        a = m.edge_features(xh, eid, use_tensor_cores=tc)
        b = m.edge_features(xf, eid, use_tensor_cores=tc)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    if case == "duplicates_and_zero_rows":
        assert float(a[:, 0].min()) < 1e-3                  # the duplicate pair was recomputed from its rows


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
@pytest.mark.parametrize("L,n_cls,agg,reattach", [(0, 1, "sum", False), (1, 1, "mean", False), (2, 1, "max", True),
                                                  (3, 2, "sum", True)])
@pytest.mark.parametrize("given_edge_attr", [False, True], ids=["ea_none", "ea_given"])
def test_forward_equals_fp32_route(m, dt, L, n_cls, agg, reattach, given_edge_attr):
    params = mo.shipped_model_params(L, n_cls, 128, (96, 64))
    params["node_agg_fn"] = agg
    params["reattach_initial_nodes"] = params["reattach_initial_edges"] = reattach
    sd = mo.init_weights(params, "resnet101", 5)
    x, ei, _, _ = mo.synth_graph(400, 4, 9, D=128, planted=True)
    xh, xf = half_pair(x, dt)
    eid = ei.to(dev())
    for replay in (True, False):                          # small-graph CUDA-graph replay / direct call (fused edge features)
        net = model(m, params, sd)
        net.use_cuda_graph = replay
        ea = m.edge_features(xf, eid) if given_edge_attr else None
        for _ in range(2):                                # the second call replays the captured graph
            a = run(net, xh, edge_index=eid, edge_attr=ea)
            b = run(net, xf, edge_index=eid, edge_attr=ea)
            assert_same(a, b)
        if replay:                                        # one captured graph per x dtype
            assert {k[8] for k in net._graphs} == {dt, torch.float32}


@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
def test_forward_ragged_batch_from_cameras(m, dt):
    params = mo.shipped_model_params(2, 1, 64, (48, 40))
    sd = mo.init_weights(params, "resnet101", 8)
    sizes = (60, 33, 120, 7, 90)
    cams = np.concatenate([np.arange(n) * c // n for n, c in zip(sizes, (3, 4, 5, 2, 8))])
    ptr = np.cumsum((0,) + sizes)
    x = torch.cat([mo.synth_graph(n, 3, i, D=64, planted=True)[0] for i, n in enumerate(sizes)])
    xh, xf = half_pair(x, dt)
    net = model(m, params, sd)
    g = m.TrackletGraph.from_cameras(cams, dev(), ptr=ptr)
    assert_same(run(net, xh, mpn_graph=g, edge_attr=None), run(net, xf, mpn_graph=g, edge_attr=None))


@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
def test_forward_configs1_size(m, dt):
    """4096 nodes, 8 cameras, 2048-d features, the shipped encoder: the fused edge-feature kernel and layer 0 on 3xFP16 planes."""
    params = mo.shipped_model_params(1, 1)
    sd = mo.init_weights(params, "resnet101", 0)
    x, _, cam, _ = mo.synth_graph(4096, 8, 1, planted=True)
    xh, xf = half_pair(x, dt)
    net = model(m, params, sd)
    g = m.TrackletGraph.from_cameras(cam, dev())
    assert_same(run(net, xh, mpn_graph=g, edge_attr=None), run(net, xf, mpn_graph=g, edge_attr=None))


def test_forward_makes_no_fp32_copy(m):
    """A warmed forward on fp16 x allocates less than N*D*2 bytes more at peak than the forward on a pre-made fp32 copy (an fp32
    copy of x would cost N*D*4)."""
    params = mo.shipped_model_params(1, 1)
    sd = mo.init_weights(params, "resnet101", 0)
    x, _, cam, _ = mo.synth_graph(2048, 4, 2, planted=True)
    xh, xf = half_pair(x, torch.float16)
    net = model(m, params, sd)
    g = m.TrackletGraph.from_cameras(cam, dev())

    def peak(xx):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        net(Data(x=xx, mpn_graph=g, edge_attr=None))
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    peak(xh), peak(xf)                                      # warm: workspaces sized, captured graphs made
    p16, p32 = peak(xh), peak(xf)
    assert p16 - p32 < x.numel() * 2, (p16, p32)


# ------------------------------------------------------------------------------------------------ column normalisation
@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
def test_normalize_columns_equal_fp32_route(m, dt):
    x = torch.randn(700, 130) * 3
    xh, xf = half_pair(x, dt)
    a, b = m.normalize_columns(xh), m.normalize_columns(xf)
    assert a.dtype == torch.float32 and torch.equal(a, b)
    ptr = [0, 1, 90, 400, 700]
    a, b = m.normalize_columns(xh, ptr=ptr), m.normalize_columns(xf, ptr=ptr)
    assert torch.equal(a, b)
    out = torch.empty(700, 130, device=dev())
    assert m.normalize_columns(xh, out=out, ptr=ptr) is out and torch.equal(out, b)


def test_normalize_columns_rejects_bad_out(m):
    x16 = torch.randn(64, 32, device=dev()).half()
    bad = [x16,                                             # 16-bit out: the fp32 result would overrun it
           torch.empty(64, 31, device=dev()),              # wrong shape
           torch.empty(64, 32),                            # wrong device
           torch.empty(32, 64, device=dev()).t()]          # not contiguous
    for out in bad:
        with pytest.raises(ValueError):
            m.normalize_columns(x16, out=out)
        with pytest.raises(ValueError):
            m.normalize_columns(x16, out=out, ptr=[0, 20, 64])
    x32 = torch.randn(64, 32, device=dev())
    ref = m.normalize_columns(x32)
    assert torch.equal(m.normalize_columns(x32, out=x32), ref)            # in place stays allowed for fp32


# ------------------------------------------------------------------------------------------------ packed files
@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
def test_load_packed_features_half(m, dt, tmp_path):
    x = torch.randn(50, 64)
    p = str(tmp_path / "f.bin")
    m.pack_reid_features(p, x, np.zeros(50), np.arange(50), dtype=dt)
    xd, _, _ = m.load_packed_features(p, dev())
    assert xd.dtype == dt and torch.equal(xd.cpu(), x.to(dt))
    xn, _, _ = m.load_packed_features(p, dev(), l2norm=True)
    assert xn.dtype == torch.float32 and torch.equal(xn, m.normalize_columns(x.to(dt).float().to(dev())))


# ------------------------------------------------------------------------------------------------ streams
@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
@pytest.mark.parametrize("depth,replay,packed", [(1, False, False), (2, False, True), (2, True, False), (2, True, True)])
def test_graph_stream_half(m, dt, depth, replay, packed):
    params = mo.shipped_model_params(1, 1, 64, (48, 40))
    sd = mo.init_weights(params, "resnet101", 21)
    net = model(m, params, sd)
    xs, refs, cam = [], [], None
    for seed in range(5):
        x, ei, cam, _ = mo.synth_graph(2048 if seed % 2 else 200, 4, seed, D=64, planted=True)
        xh, xf = half_pair(x, dt)
        net(Data(x=xf, edge_index=ei.to(dev())))
        xs.append((xh.cpu().pin_memory(), cam.numpy(), ei.shape[1]))
        pred = net.last_pred.cpu()
        refs.append(torch.from_numpy(np.packbits(pred.numpy(), bitorder="little")) if packed else pred)
    gs = m.GraphStream(net, dev(), depth=depth, graph_replay=replay, packed_decisions=packed)
    outs = []
    for (xh, c, E), r in zip(xs + xs, refs + refs):             # twice over: the replay path sees repeated signatures
        o = torch.zeros(4 * ((E + 31) // 32) if packed else E, dtype=torch.uint8).pin_memory()
        gs.submit(xh, c, o)
        outs.append(o)
    gs.drain()
    for o, r in zip(outs, refs + refs):
        assert torch.equal(o[:r.numel()], r)
    assert all(s.x_dev.dtype == dt for s in gs.slots if s.x_dev is not None)


# ------------------------------------------------------------------------------------------------ sharded (one process)
class _NoComm:
    world, rank = 1, 0

    def all_reduce_sum(self, t):
        pass

    def all_gather_rows(self, full, blocks):
        pass

    def all_gather_ragged(self, t):
        return [t]


@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
def test_sharded_cuda_shards_in_one_process_half(m, dt):
    params = mo.shipped_model_params(2, 1, 64, (48, 40))
    x, ei, _, _ = mo.synth_graph(90, 3, 41, D=64, planted=True)
    sd = mo.init_weights(params, "resnet101", 13)
    ea = mo.edge_features(x, ei).to(dev())
    xh, xf = half_pair(x, dt)
    net = model(m, params, sd, fuse=False)
    W = net._weights(dev())
    N, E = x.shape[0], ei.shape[1]
    rowptr = torch.searchsorted(ei[0].contiguous(), torch.arange(N + 1))
    blocks = m.partition_rows(rowptr, 3)
    res = {}
    for xx in (xh, xf):
        shards, keep = [], []
        for i, (n0, n1) in enumerate(blocks):
            lo, hi = m.shard_edges(ei, n0, n1)
            g = m.TrackletGraph(ei[:, lo:hi].to(dev()), N, row_offset=n0, n_rows=n1 - n0)
            logits = torch.empty(1, hi - lo, 2, device=dev())
            ph = m.CudaPhases(g, W, xx, ea[lo:hi].contiguous(), 2, 1, E, logits, None, None, True, ws_kind="halfshard%d" % i)
            shards.append(ph); keep.append((g, logits, lo, hi))
        m.sharded_forward(shards, _NoComm(), 2, 1, blocks)
        torch.cuda.synchronize()
        logits = torch.cat([k[1][0] for k in keep])
        hs = torch.cat([p.h_full()[b[0]:b[1]] for p, b in zip(shards, blocks)])
        efs = torch.cat([m.edge_features(xx, None, graph=k[0]) for k in keep])
        res[xx.dtype] = (logits.clone(), hs.clone(), efs.clone())
        for p in shards:
            p.close()
    for u, v in zip(res[dt], res[torch.float32]):
        assert torch.equal(u, v)


def test_multi_gpu_half_features_torchrun(m):
    """ShardedMPN (shared Gram) and ShardedGraphStream with 16-bit x on >= 2 GPUs (skipped otherwise)."""
    import os
    import subprocess
    import sys
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(n, 4)),
           "--master-addr", "127.0.0.1", "--master-port", "29583", os.path.join(root, "tests", "half_features_dist.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=400)
    assert r.returncode == 0 and "half_features_dist ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("dt", HALF, ids=["f16", "bf16"])
def test_layer0_rows_off_a_16_byte_boundary(m, dt):
    """16-bit rows that start 8 bytes off a 16-byte boundary (K = 132, a row-slice view): layer 0 of the encoder reads them in
    place through the plan API with the result of the fp32 widening (the TF32 split needs four-element alignment only, 8 bytes),
    and the Python entry points, which realign such a view, return the bits of the x.float() route."""
    params = mo.shipped_model_params(1, 1, 132, (96, 64))
    sd = mo.init_weights(params, "resnet101", 4)
    x, ei, _, _ = mo.synth_graph(300, 4, 2, D=132, planted=True)
    xv = torch.cat([torch.zeros(1, 132), x]).to(dev()).to(dt)[1:]
    assert xv.is_contiguous() and xv.data_ptr() % 16 == 8
    xf = xv.float()
    net = model(m, params, sd, fuse=False)
    W = net._weights(dev())
    eid = ei.to(dev())
    g = m.TrackletGraph(eid, 300)
    ea = m.edge_features(xf, None, graph=g)
    kind = m._lib.MPN_X_F16 if dt == torch.float16 else m._lib.MPN_X_BF16
    hs = []
    for ptr, k in ((xv.data_ptr(), kind), (xf.data_ptr(), m._lib.MPN_X_F32)):
        logits = torch.empty(1, g.n_edges, 2, device=dev())
        ph = m.CudaPhases(g, W, xf, ea, 1, 1, g.n_edges, logits, None, None, True, ws_kind="unaligned_rows")
        m._lib.check(ph.lib.mpn_plan_node_encoder_x(ph.plan, ptr, k, ph.stream))
        torch.cuda.synchronize()
        hs.append(ph.h_full().clone())
        ph.close()
    assert torch.equal(hs[0], hs[1])
    assert_same(run(net, xv, edge_index=eid, edge_attr=None), run(net, xf, edge_index=eid, edge_attr=None))
