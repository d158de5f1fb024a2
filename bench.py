#!/usr/bin/env python
"""Benchmark of the MPN hot path (BASELINE.json metric: MPN inference directed edges/sec; p50 latency per S02-shape graph).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-extras] [--dump-outputs DIR]

A step = one pass of the hot path over one synthetic graph that is already resident in HBM, through the public call
(`MOTMPNet.forward(data)` with `data.edge_attr = None`): graph tables from the int64 `edge_index` (K0), edge features (K1, with
the first BatchNorm's moment sums taken in the GEMM epilogue), forward with fused decisions.
N = 1: BASELINE.json configs[1] — L=1 MPN, 4096 tracklets, 8 cameras, dense cross-camera edges, E = 14,680,064 directed edges
("~7M" undirected pairs).  N > 1: the same per-GPU work (weak scaling): a graph of 4096*sqrt(N) tracklets whose edges are
sharded by row block; the line also carries `c5_strong` (BASELINE configs[4]: 32,768 tracklets, L = 4, fixed graph).
Before any timing the outputs are checked (BASELINE.md section 4.3): `parity` in the line; a failed gate raises.
Prints ONE JSON line (rank 0).  `--impl reference` times the reference ITSELF (oracle/_ref: the reference's own Python files,
copied by __graft_entry__.build()) on the host cores, on the same configuration.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints a "NCCL version ..." banner through C stdio when
# the first communicator is created), so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to a
# private duplicate of the original stdout.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()

import torch  # noqa: E402

NODES_1GPU, CAMS, FEAT_DIM = 4096, 8, 2048
METRIC, UNIT = "mpn_inference_directed_edges_per_sec", "edges/s"
# algorithmic work per directed edge (SURVEY.md section 8d / DESIGN.md "Kernels")
# node_apply: y read 16 + logits 8 + the fused decisions this bench asks for (u8 prediction 1 + fp32 probability 4), SURVEY 8d row K4
BYTES_PER_EDGE = {"enc_moments": 8.0, "edge_update": 28.0, "node_moments": 16.0, "node_apply": 29.0, "forward": 81.0}
FLOP_PER_EDGE_GRAM = 4096.0


def shipped_params(L=1, n_cls=1):
    """GRAPH_NET_PARAMS of the reference's config/config_training.yaml:68-111 (the benchmark's model), restated."""
    return {"node_agg_fn": "sum", "num_enc_steps": L, "num_class_steps": n_cls, "reattach_initial_nodes": False,
            "reattach_initial_edges": False,
            "encoder_feats_dict": {"edges": {"edge_in_dim": 2, "edge_fc_dims": [4], "edge_out_dim": 4},
                                   "nodes": {"resnet101": {"node_in_dim": FEAT_DIM, "node_fc_dims": [1024, 512, 128],
                                                           "node_out_dim": 32, "dropout_p": 0.1, "use_batchnorm": True}}},
            "edge_model_feats_dict": {"fc_dims": [4], "dropout_p": 0.1, "use_batchnorm": True},
            "node_model_feats_dict": {"fc_dims": [32], "dropout_p": 0.1, "use_batchnorm": True},
            "classifier_feats_dict": {"edge_in_dim": 4, "edge_fc_dims": [], "edge_out_dim": 2, "dropout_p": 0,
                                      "use_batchnorm": False, "is_classifier": True}}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: an NVML polling thread (1 ms period), `nvidia-smi` as fallback."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        import threading
        self.samples, self.bits, self.max_mhz, self.power = [], 0, None, []
        self.stop_flag = threading.Event()
        self.thread = self.p = self.f = None
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                i = 0
                while not self.stop_flag.is_set():
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        if i % 4 == 0:
                            self.bits |= int(reasons_fn(h))
                            self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    except Exception:
                        pass
                    i += 1
                    time.sleep(0.001)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            self.how = "nvml thread, 1 ms period"
        except Exception:
            self.how = "nvidia-smi -lms 20"
            try:
                self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                           "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
                time.sleep(1.0)
            except Exception:
                self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "how": self.how}
        reasons = set()
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            reasons = {name for name, bit in self.REASONS if self.bits & bit}
            if self.power:
                out["power_w_max"] = max(self.power)
        elif self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.f.flush()
            rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
            os.unlink(self.f.name)
            for r in rows:
                try:
                    self.samples.append(float(r[0]))
                    out["sm_max_mhz"] = float(r[1])
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                        if v.strip().lower().startswith("active"):
                            reasons.add(name)
                except Exception:
                    pass
        sm = sorted(self.samples)
        if sm:
            out["sm_mhz"] = sm[len(sm) // 2]
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------- synthetic graph
def workload_shape(world):
    """(tracklets, directed edges) of the bench workload on ``world`` GPUs: configs[1] at 1 GPU, E per GPU ~ constant above."""
    if world == 1:
        n = NODES_1GPU
    else:
        n = int(round(NODES_1GPU * world ** 0.5 / (CAMS * world))) * CAMS * world           # weak scaling
    return n, n * (n - n // CAMS)                                                            # equal cameras, all cross-camera pairs


def workload_name(n_nodes, e_total, world):
    return ("BASELINE configs[1]: L=1 MPN (shipped config) + edge features + decisions, %d tracklets, %d cameras, dense "
            "cross-camera edges, E=%d directed edges%s" %
            (n_nodes, CAMS, e_total, "" if world == 1 else " row-block sharded over %d GPUs" % world))


def device_features(n_nodes, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n_nodes, FEAT_DIM, generator=g, device=dev), p=2, dim=0)   # inference.py:403-404


def device_graph(n_nodes, cams, seed, dev, row_block=None):
    """Graph(N,C,seed) of SURVEY.md section 8d built on the device.  row_block=(n0,n1) builds only that shard's edges."""
    x = device_features(n_nodes, seed, dev)
    cam = (torch.arange(n_nodes, device=dev) * cams // n_nodes)
    nodes = torch.arange(n_nodes, device=dev)
    n0, n1 = row_block if row_block is not None else (0, n_nodes)
    parts = []
    for c in range(cams):
        rows = nodes[(cam == c) & (nodes >= n0) & (nodes < n1)]
        if rows.numel():
            parts.append(torch.cartesian_prod(rows, nodes[cam != c]))         # inference.py:409-413
    ei = torch.cat(parts, dim=0).t().contiguous()
    return x, ei


def make_model(dev, L=1, n_cls=1, seed=0):
    """The benchmark's model: shipped configuration, default nn.Linear initialisation under a fixed seed, BatchNorm affine
    parameters jittered (weight ~ U(0.5,1.5), bias ~ N(0,0.1)) so that no BatchNorm is trivially the identity."""
    import gcn_mtmc_b200 as m
    torch.manual_seed(seed)
    net = m.MOTMPNet(copy.deepcopy(shipped_params(L, n_cls)), None, "resnet101")
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for mod in net.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.weight.copy_(torch.rand(mod.weight.shape, generator=g) + 0.5)
                mod.bias.copy_(torch.randn(mod.bias.shape, generator=g) * 0.1)
    net = net.to(dev).eval()
    net.fuse_decisions = True
    return net


class Batch:
    pass


def time_events(fn, flush, reps, warm=3):
    ts = []
    for i in range(reps + warm):
        if flush is not None:
            flush.fill_(i & 0xFF)
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        e.record()
        e.synchronize()
        if i >= warm:
            ts.append(a.elapsed_time(e))
    ts.sort()
    return ts


# ------------------------------------------------------------------------------------------------- reference arm (host cores)
def reference_sample(ef_edges=1_000_000, nodes=NODES_1GPU, cams=CAMS, model=None, cache={}):
    """One bounded sample of the configs[1] step on the host cores with the reference itself (oracle/_ref), else its port
    (oracle/mpn_oracle.py): the forward on the WHOLE graph (same N, C, E as the GPU arm), the reference's edge-feature statements
    on the first ``ef_edges`` edges, decisions.  The rate per directed edge adds the two per-edge costs."""
    from oracle import mpn_oracle as mo
    from oracle import ref_arm
    torch.set_num_threads(os.cpu_count() or 1)
    key = (nodes, cams)
    if key not in cache:
        x, ei, _, _ = mo.synth_graph(nodes, cams, 0)
        gen = torch.Generator().manual_seed(5)
        # edge features of the WHOLE graph for the forward's input: a filled-in stand-in with the right statistics (computing
        # them with the reference's statements takes ~40 s per pass; they are timed on a slice below)
        ea = torch.empty(ei.shape[1], 2)
        ea[:, 0] = 1.414 + 0.023 * torch.randn(ei.shape[1], generator=gen)
        ea[:, 1] = 1.0 + 0.022 * torch.randn(ei.shape[1], generator=gen)
        cache[key] = (x, ei, ea)
    x, ei, ea = cache[key]
    E = ei.shape[1]
    if ref_arm.available():
        kind = "reference"
        net = model if model is not None else ref_arm.make_model()
        r = ref_arm.timed_step(net, x, ei, ef_edges, edge_attr=ea)
        t_fwd, t_ef, n_ef, t_dec = r["t_forward"], r["t_edge_features"], r["ef_edges"], r["t_decisions"]
        what = "the reference itself (oracle/_ref: models/mpn.py, models/mlp.py, inference.py:453-456,475-479 verbatim)"
    else:
        kind = "port"
        params = mo.shipped_model_params(1, 1)
        sd = mo.init_weights(params, "resnet101", 0)
        n_ef = int(min(E, ef_edges))
        t0 = time.perf_counter()
        mo.edge_features(x, ei[:, :n_ef], chunk=200_000)
        t_ef = time.perf_counter() - t0
        with torch.no_grad():
            t0 = time.perf_counter()
            out, _ = mo.mpn_forward(sd, params, "resnet101", x, ei, ea)
            t_fwd = time.perf_counter() - t0
            t0 = time.perf_counter()
            mo.decide(out[-1])
            t_dec = time.perf_counter() - t0
        net = None
        what = "oracle/mpn_oracle.py (torch-CPU port of the reference; oracle/_ref is not built)"
    per_edge = (t_fwd + t_dec) / E + t_ef / n_ef
    return {"value": 1.0 / per_edge, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": kind,
            "sample": "%s on %d host threads: MOTMPNet.forward + softmax/argmax on the WHOLE configs[1] graph (N=%d C=%d E=%d: %.2f s) "
                      "+ the edge-feature statements on the first %d edges in 200k-edge chunks (%.2f us/edge; un-chunked they need "
                      "2 x E x 8 KB), per-edge costs added" % (what, os.cpu_count() or 1, nodes, cams, E, t_fwd + t_dec, n_ef, t_ef / n_ef * 1e6),
            "forward_edges_per_sec": E / (t_fwd + t_dec), "edge_feature_edges_per_sec": n_ef / t_ef, "same_config": True,
            "_model": net, "_seconds": t_fwd + t_dec + t_ef}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, info, model = [], None, None
    ef_edges = 1_000_000
    t_start = time.perf_counter()
    budget = 280.0                                              # the whole run stays within a few minutes
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        info = reference_sample(ef_edges=ef_edges if i >= args.warmup else 200_000, model=model)
        model = info.pop("_model")
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
        left = args.warmup + args.steps - i - 1
        if left > 0 and (time.perf_counter() - t_start) + left * dt > budget and ef_edges > 200_000:
            ef_edges = max(200_000, ef_edges // 2)              # shrink the edge-feature slice, never the graph of the forward
    v = info["value"]
    world = max(int(args.gpus), 1)
    n_nodes, e_total = workload_shape(1)
    info.pop("_seconds", None)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / max(len(times), 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(n_nodes, e_total, 1),
                       "sample": "each step = one bounded sample of that workload on the host cores (see cpu_baseline.sample); the "
                                 "rate is per directed edge, so it is the figure to set against the %d-GPU line as well" % world},
            "cpu_baseline": {k: info[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config")},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------- parity gate
def parity_gate(m, net, x, ei, dev):
    """BASELINE.md section 4.3 on the benchmark's own graph, before anything is timed.  Checker: oracle/mpn_oracle.py (the port
    of the reference that tests/ pin against the reference's outputs) evaluated in fp64 with torch ops on the device.
      * edge features (tcgen05 kernel) on 262,144 sampled edges vs fp64: rtol = atol = 1e-5
      * logits of the one-call forward vs the fp64 forward on our edge features: max |err| <= 1e-4 * max|logit|
      * decisions identical wherever the fp64 margin |l1 - l0| exceeds that bound; prob1 bit-identical to torch.softmax of our logits
    Raises on failure; returns the measured errors."""
    from oracle import mpn_oracle as mo
    N, E = x.shape[0], ei.shape[1]
    b = Batch()
    b.x, b.edge_index, b.num_nodes, b.edge_attr = x, ei, N, None
    out, h = net(b)
    logits = out["classified_edges"][-1]
    pred, prob1 = net.last_pred, net.last_prob1
    ea = b.edge_attr
    gen = torch.Generator(device=dev).manual_seed(11)
    idx = torch.randint(0, E, (262144,), generator=gen, device=dev)
    a, c = x.double()[ei[0, idx]], x.double()[ei[1, idx]]
    d = (a - c + 1e-6).norm(dim=1)
    cs = 1 - (a * c).sum(1) / (a.norm(dim=1) * c.norm(dim=1)).clamp_min(1e-8)
    ef_err = max((ea[idx, 0].double() - d).abs().max().item(), (ea[idx, 1].double() - cs).abs().max().item())
    ef_ok = bool(torch.allclose(ea[idx, 0].double(), d, rtol=1e-5, atol=1e-5) and torch.allclose(ea[idx, 1].double(), cs, rtol=1e-5, atol=1e-5))
    del a, c
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    ref, href = mo.mpn_forward(sd, shipped_params(int(net.num_enc_steps), int(net.num_class_steps)), "resnet101", x, ei, ea, dtype=torch.float64)
    ref = ref[-1]
    scale = ref.abs().max().item()
    err = (logits.double() - ref).abs().max().item()
    margin = (ref[:, 1] - ref[:, 0]).abs()
    wrong = (pred.long() != ref.argmax(1)) & (margin > 1e-4 * scale)
    n_wrong = int(wrong.sum().item())
    h_err = (h.double() - href).abs().max().item()
    h_tol = 1e-4 * max(1.0, href.abs().max().item())
    prob_same = bool(torch.equal(prob1, torch.softmax(logits, dim=1)[:, 1]))
    res = {"checked": True, "checker": "oracle/mpn_oracle.py in fp64 on the device (torch ops)", "edge_feature_max_abs_err": ef_err,
           "logit_max_abs_err": err, "logit_tolerance": 1e-4 * scale, "h_max_abs_err": h_err, "h_tolerance": h_tol,
           "decisions_differ_outside_margin_band": n_wrong, "decisions_differ_total": int((pred.long() != ref.argmax(1)).sum().item()),
           "prob1_bit_identical_to_torch_softmax": prob_same}
    del ref, href
    torch.cuda.empty_cache()
    if not (ef_ok and err <= 1e-4 * scale and n_wrong == 0 and h_err <= h_tol and prob_same):
        raise RuntimeError("parity gate failed: %s" % json.dumps(res))
    return res


# ------------------------------------------------------------------------------------------------- phases (N = 1)
def time_phases(m, net, x, ei, reps=5):
    """Per-kernel device times through the plan API (CUDA events on the launching stream), L2 flushed between repetitions."""
    dev = x.device
    g = m.TrackletGraph(ei, x.shape[0])
    ea = m.edge_features(x, ei, graph=g)
    W = net._weights(dev)
    logits = torch.empty(1, g.n_edges, 2, device=dev)
    pred = torch.empty(g.n_edges, dtype=torch.uint8, device=dev)
    prob1 = torch.empty(g.n_edges, device=dev)
    ph = m.CudaPhases(g, W, x, ea, 1, 1, g.n_edges, logits, pred, prob1, True, ws_kind="bench_plan")
    S = m._lib
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    seq = [("node_encoder", lambda: ph.node_encoder()),
           ("enc_moments0_sweep_not_in_the_step", lambda: ph.sweep(0, S.STAGE_ENC0)), ("fin0", lambda: ph.reduce(S.STAGE_ENC0, True)),
           ("enc_moments1", lambda: ph.sweep(0, S.STAGE_ENC1)), ("fin1", lambda: ph.reduce(S.STAGE_ENC1, True)),
           ("node_tables", lambda: ph.node_tables(1)),
           ("edge_update", lambda: ph.sweep(1, S.STAGE_EDGE)), ("fin2", lambda: ph.reduce(S.STAGE_EDGE, True)),
           ("node_moments", lambda: ph.sweep(1, S.STAGE_NODE)), ("fin3", lambda: ph.reduce(S.STAGE_NODE, True)),
           ("node_apply", lambda: ph.sweep(1, S.STAGE_APPLY, out_index=0, last=True)),
           ("node_finalize", lambda: ph.node_finalize(1))]
    acc = {}
    for name, fn in seq:
        ts = time_events(fn, flush, reps, warm=1)
        acc[name] = sum(ts) / len(ts)
    ph.close()
    ts = time_events(lambda: m.edge_features(x, ei, graph=g), flush, reps, warm=1)
    acc["edge_features"] = sum(ts) / len(ts)
    ts = time_events(lambda: m.TrackletGraph(ei, x.shape[0], validate="deferred"), flush, reps, warm=1)
    acc["graph_tables_from_edge_index"] = sum(ts) / len(ts)
    # the Gram GEMM with the distance epilogue alone: CUDA events recorded by the library around that one launch
    lib = S.lib()
    lib.mpn_profile_gram(1)
    ks = []
    for rep in range(reps + 1):
        flush.fill_(rep & 0xFF)
        m.edge_features(x, ei, graph=g)
        torch.cuda.synchronize()
        if rep > 0:
            ks.append(float(lib.mpn_profile_gram_ms()))
    lib.mpn_profile_gram(0)
    acc["gram_ef_kernel"] = sum(ks) / len(ks)
    return acc


def s02_latency(m, dev, reps=300):
    """Second half of BASELINE.json's metric: p50 latency of one S02-shaped graph (configs[0]: N=300, C=4, E=67,500, L=1):
    graph tables + edge features + forward + fused decisions per call (device time, CUDA events; host wall clock beside it),
    and the post-processing of its decisions (CUT / PRUNE / CUT / SPLIT + reference labels; host wall clock, it synchronises)."""
    net = make_model(dev)
    x, ei = device_graph(300, 4, 0, dev)
    b = Batch()
    b.x, b.edge_index, b.num_nodes = x, ei, 300

    def call():
        g = m.TrackletGraph(ei, 300, validate="deferred")
        b._mpn_b200_graph = ((ei.data_ptr(), tuple(ei.shape), ei._version, 300, None), g)
        b.edge_attr = m.edge_features(x, ei, graph=g)
        net(b)
        g.validate()
        return net.last_pred
    for _ in range(20):
        call()
    dts, hts = [], []
    for _ in range(reps):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a.record()
        call()
        e.record()
        e.synchronize()
        hts.append(1e3 * (time.perf_counter() - t0))
        dts.append(a.elapsed_time(e))
    dts.sort()
    hts.sort()
    # the whole call as ONE CUDA graph (GraphStream(graph_replay=True)): host features in, decisions out, copies included
    gs = m.GraphStream(net, dev, depth=1, graph_replay=True)
    hx = x.cpu().pin_memory()
    hp = torch.empty(ei.shape[1], dtype=torch.uint8).pin_memory()
    cam_host = (torch.arange(300) * 4 // 300).numpy()
    for _ in range(6):
        gs.submit(hx, cam_host, hp)
        gs.drain()
    rts, rhs = [], []
    for _ in range(reps):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a.record()
        gs.submit(hx, cam_host, hp)
        gs.drain(host_sync=False)
        e.record()
        e.synchronize()
        rhs.append(1e3 * (time.perf_counter() - t0))
        rts.append(a.elapsed_time(e))
    rts.sort()
    rhs.sort()
    replay = {"p50_ms": rts[len(rts) // 2], "p99_ms": rts[int(len(rts) * 0.99)], "host_wall_p50_ms": rhs[len(rhs) // 2],
              "how": "GraphStream(depth=1, graph_replay=True).submit + drain: H2D of the pinned features (2.4 MB), tables + edge features + "
                     "forward + decisions replayed as one CUDA graph, D2H of the decisions (67 KB); CUDA events around the whole call"}
    # post-processing of a planted S02-shaped prediction (the random-weight decisions above are ~50 % active: not a tracking output)
    import numpy as np
    rng = np.random.default_rng(0)
    ident = rng.integers(0, 110, 300)
    src, dst = ei[0].cpu().numpy(), ei[1].cpu().numpy()
    same = ident[src] == ident[dst]
    flip = rng.random(src.size)
    act = np.where(same, flip > 0.03, flip < 0.003)
    prob = np.where(act, rng.uniform(0.55, 1.0, src.size), rng.uniform(0.0, 0.45, src.size)).astype(np.float32)
    pred_d, prob_d = torch.from_numpy(act.astype(np.int64)).to(dev), torch.from_numpy(prob).to(dev)
    cfg = {"CUTTING": True, "PRUNING": True, "SPLITTING": True}
    pts = []
    for _ in range(25):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.post_processing(4, None, None, pred_d.clone(), None, dict(cfg), b, prob_d)
        torch.cuda.synchronize()
        pts.append(1e3 * (time.perf_counter() - t0))
    pts.sort()
    return {"config": "BASELINE configs[0] shape: 300 tracklets, 4 cameras, E=%d directed edges, L=1; K0 + K1 + forward + decisions per call "
                      "(forward replayed as one CUDA graph)" % ei.shape[1],
            "p50_ms": dts[len(dts) // 2], "p99_ms": dts[int(len(dts) * 0.99)], "host_wall_p50_ms": hts[len(hts) // 2], "calls": reps,
            "one_graph_replay_from_host": replay,
            "post_processing_ms": pts[len(pts) // 2],
            "post_processing": "CUT + PRUNE + CUT + SPLIT + reference label numbering of a planted prediction on the same graph "
                               "(%d active edges), host wall clock p50 of 25 calls" % int(act.sum())}


# ------------------------------------------------------------------------------------------------- other BASELINE configs
def extra_batched_graphs(m, dev, n_graphs=2000, n=300, cams=4):
    """BASELINE configs[2]: 2000 S02-shaped graphs packed into one launch, BatchNorm statistics per graph."""
    net = make_model(dev)
    gen = torch.Generator(device=dev).manual_seed(3)
    x = torch.randn(n_graphs, n, FEAT_DIM, generator=gen, device=dev)
    x = torch.nn.functional.normalize(x, p=2, dim=1).reshape(n_graphs * n, FEAT_DIM)      # per graph, per column
    _, tmpl = device_graph(n, cams, 0, dev)
    E1 = tmpl.shape[1]
    ei = (tmpl[None] + (torch.arange(n_graphs, device=dev) * n)[:, None, None]).permute(1, 0, 2).reshape(2, n_graphs * E1).contiguous()
    ptr = torch.arange(n_graphs + 1, device=dev) * n
    b = Batch()
    b.x, b.edge_index, b.num_nodes, b.ptr = x, ei, n_graphs * n, ptr

    def step():
        b.edge_attr = None
        b._mpn_b200_graph = None
        return net(b)
    out, _ = step()
    big = out["classified_edges"][-1]
    # >= 50 graphs checked against the single-graph path (the reference handles one graph per forward: inference.py:375,469)
    worst = 0.0
    for k in torch.linspace(0, n_graphs - 1, 50).long().tolist():
        s = Batch()
        s.x, s.edge_index, s.num_nodes, s.edge_attr = x[k * n:(k + 1) * n].contiguous(), tmpl, n, None
        o1, _ = net(s)
        l1 = o1["classified_edges"][-1]
        worst = max(worst, (l1 - big[k * E1:(k + 1) * E1]).abs().max().item() / l1.abs().max().item())
    if worst > 1e-4:
        raise RuntimeError("batched graphs differ from the single-graph path: %g" % worst)
    ts = time_events(step, None, 5, warm=1)
    ms = ts[len(ts) // 2]
    return {"config": "BASELINE configs[2]: %d graphs x (N=%d, C=%d, E=%d) in one call (tables + edge features + forward + decisions), "
                      "BatchNorm statistics per graph" % (n_graphs, n, cams, E1),
            "ms": ms, "us_per_graph": 1e3 * ms / n_graphs, "graphs_per_s": n_graphs / ms * 1e3, "edges_per_s": ei.shape[1] / ms * 1e3,
            "max_rel_logit_diff_vs_single_graph_path_50_graphs": worst}


def planted_prediction_device(n_nodes, cams, e_target, dev, seed=7):
    """Predicted graph of BASELINE configs[3] generated on the device: planted clusters of <= cams nodes (one per camera), their
    directed edges active with p in U(0.55,1) (2 % flipped off), plus random inter-cluster pairs (both directions) up to
    ``e_target`` edges, each direction flipped on with 2 % (p in U(0.5,0.6)) — ~4e-4 of the pairs end up mutual and merge
    clusters, which is what PRUNING and SPLITTING then undo; ~1 % of the active edges lose their reverse.  Edges are (row, col)-
    sorted and unique."""
    g = torch.Generator(device=dev).manual_seed(seed)
    # nodes are laid out cluster by cluster; node k of a cluster sits in camera k
    sizes = torch.randint(1, cams + 1, (int(n_nodes * 2 / (cams + 1)) + cams,), generator=g, device=dev)
    cs = torch.cumsum(sizes, 0)
    n_clusters = int((cs <= n_nodes).sum().item())
    sizes = sizes[:n_clusters]
    rest = n_nodes - int(sizes.sum().item())
    if rest > 0:
        sizes = torch.cat([sizes, torch.ones(rest, dtype=sizes.dtype, device=dev)])
    cluster = torch.repeat_interleave(torch.arange(sizes.numel(), device=dev), sizes)
    # intra-cluster ordered pairs
    first = torch.cumsum(sizes, 0) - sizes
    pos = torch.arange(n_nodes, device=dev) - first[cluster]
    parts_s, parts_d = [], []
    for k in range(1, cams):
        ok = pos + k < sizes[cluster]
        a = torch.nonzero(ok).reshape(-1)
        parts_s += [a, a + k]
        parts_d += [a + k, a]
    s_in, d_in = torch.cat(parts_s), torch.cat(parts_d)
    n_rand = max(0, (e_target - s_in.numel()) // 2)                          # random inter-cluster PAIRS, both directions present
    s_r = torch.randint(0, n_nodes, (n_rand,), generator=g, device=dev)
    d_r = torch.randint(0, n_nodes, (n_rand,), generator=g, device=dev)
    keep = (cluster[s_r] != cluster[d_r]) & (pos[s_r] != pos[d_r])          # different identities, different cameras
    s_r, d_r = s_r[keep], d_r[keep]
    key = torch.cat([s_in * n_nodes + d_in, s_r * n_nodes + d_r, d_r * n_nodes + s_r])
    intra = torch.cat([torch.ones(s_in.numel(), dtype=torch.bool, device=dev), torch.zeros(2 * s_r.numel(), dtype=torch.bool, device=dev)])
    key, order = torch.sort(key)
    intra = intra[order]
    uniq = torch.ones_like(intra)
    uniq[1:] = key[1:] != key[:-1]
    key, intra = key[uniq], intra[uniq]
    src, dst = key // n_nodes, key % n_nodes
    E = key.numel()
    u = torch.rand(E, generator=g, device=dev)
    act = torch.where(intra, u > 0.02, u < 0.02)
    p = torch.rand(E, generator=g, device=dev)
    prob = torch.where(act, torch.where(intra, 0.55 + 0.45 * p, 0.5 + 0.1 * p), 0.45 * p).float()
    drop = act & (torch.rand(E, generator=g, device=dev) < 0.01)              # single-direction edges
    act = act & ~drop
    prob = torch.where(drop, 0.45 * p, prob)
    return torch.stack([src, dst]), act.long(), prob


def extra_post_processing(m, dev, n_nodes=1_000_000, e_target=100_000_000, cams=8):
    """BASELINE configs[3]: post-processing only on a 1M-node, 100M-edge predicted graph."""
    import numpy as np
    ei, pred, prob = planted_prediction_device(n_nodes, cams, e_target, dev)
    E = ei.shape[1]
    d = Batch()
    d.x, d.edge_index, d.num_nodes = torch.zeros(n_nodes, 1, device=dev), ei, n_nodes
    m.graph_for(d, ei, n_nodes)
    cfg = {"CUTTING": True, "PRUNING": True, "SPLITTING": True}
    res = {}
    for numbering in ("canonical", "reference"):
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ID, P = m.post_processing(cams, None, None, pred.clone(), None, dict(cfg), d, prob, numbering=numbering)
            torch.cuda.synchronize()
            ts.append(1e3 * (time.perf_counter() - t0))
        res["ms_numbering_" + numbering] = min(ts)
    st = m.split_stats()
    sizes = np.bincount(ID.numpy())
    # size-independent properties: no cluster above the camera count; only active edges were switched off; SPLITTING again is a
    # no-op (nothing oversized is left) and gives the same label integers
    ID2, P2 = m.post_processing(cams, None, None, P.clone(), None, {"CUTTING": False, "PRUNING": False, "SPLITTING": True}, d, prob,
                                numbering="reference")
    idem = bool(torch.equal(P2, P)) and bool(np.array_equal(ID2.numpy(), ID.numpy()))
    subset = bool((P <= pred).all().item())
    if int(sizes.max()) > cams or not idem or not subset:
        raise RuntimeError("configs[3] property check failed: max cluster %d, SPLITTING idempotent %s, subset %s" % (int(sizes.max()), idem, subset))
    res.update({"config": "BASELINE configs[3]: CUT + PRUNE + CUT + SPLIT + labels on a predicted graph of %d nodes, %d directed edges "
                          "(%d active), %d cameras" % (n_nodes, E, int(pred.sum().item()), cams),
                "edges_per_s": E / (res["ms_numbering_reference"] * 1e-3), "clusters": int(sizes.size), "active_after": int(P.sum().item()),
                "max_cluster_size": int(sizes.max()), "splitting_idempotent": idem, "splitting": st,
                "timing": "host wall clock around the call (it synchronises), best of 3"})
    return res


def big_graph_step(m, dev, world, rank, sharded_cls, n_nodes=32768, L=4, steps=3, check=True):
    """BASELINE configs[4]: L=4, 32,768 tracklets, E = 939,524,096, row-block sharded over `world` GPUs (strong scaling: the graph
    is fixed).  Tables from the camera ids (the int64 edge_index alone would be 15 GB).  At world > 1 every rank also runs the
    unsharded forward once and compares its shard's decisions with it."""
    import torch.distributed as dist
    net = make_model(dev, L=L, n_cls=1)
    x = device_features(n_nodes, 0, dev)
    cam_host = (torch.arange(n_nodes) * CAMS // n_nodes).numpy()
    per = n_nodes // world
    blocks = [(r * per, (r + 1) * per) for r in range(world)]
    E_total = n_nodes * (n_nodes - n_nodes // CAMS)
    sharded = sharded_cls(net) if world > 1 else None
    batch = Batch()
    batch.num_nodes = n_nodes

    def step():
        if world == 1:
            batch.x, batch.mpn_graph, batch.edge_attr = x, m.TrackletGraph.from_cameras(cam_host, dev), None
            net(batch)
            return net.last_pred
        gr = m.TrackletGraph.from_cameras(cam_host, dev, row_block=blocks[rank])
        return sharded.forward(x, None, None, blocks, fuse_decisions=True, graph=gr, total_edges=E_total)[2]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    pred = step()
    barrier()
    times = []
    for _ in range(steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pred = step()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        times.append(float(ms.item()))
    times.sort()
    ms = times[len(times) // 2]            # median: a step that makes the caching allocator go back to cudaMalloc (tens of GB of
                                           # per-step tensors) is not the kernels' time
    res = {"config": "BASELINE configs[4]: N=%d C=%d L=%d E=%d directed edges, row-block sharded over %d GPU(s), tables from camera ids"
                     % (n_nodes, CAMS, L, E_total, world),
           "ms_per_step": ms, "ms_per_step_all": [round(t, 3) for t in times], "timing": "median of %d steps, CUDA events, max over ranks" % steps,
           "edges_per_s": E_total / (ms * 1e-3), "edge_steps_per_s": E_total * L / (ms * 1e-3),
           "peak_mem_gb_rank0": torch.cuda.max_memory_allocated(dev) / 1e9}
    if world > 1:
        res["path"] = sharded.path
        if check:
            pred_sh = pred.clone()
            del pred
            torch.cuda.empty_cache()
            batch.x, batch.mpn_graph, batch.edge_attr = x, m.TrackletGraph.from_cameras(cam_host, dev), None
            out, _ = net(batch)
            full_pred, lg = net.last_pred, out["classified_edges"][-1]
            g_full = batch.mpn_graph
            lo = int(g_full.rowptr[blocks[rank][0]].item())
            hi = int(g_full.rowptr[blocks[rank][1]].item())
            margin = (lg[lo:hi, 1] - lg[lo:hi, 0]).abs()
            diff = full_pred[lo:hi] != pred_sh
            bad = torch.tensor([float((diff & (margin > 1e-4 * lg.abs().max())).sum().item()), float(diff.sum().item()),
                                float(pred_sh.sum().item())], dtype=torch.float64, device=dev)
            dist.all_reduce(bad)
            res["vs_unsharded"] = {"decisions_differ_outside_margin_band": int(bad[0].item()), "decisions_differ_total": int(bad[1].item()),
                                   "active_edges": int(bad[2].item())}
            if int(bad[0].item()) != 0:
                raise RuntimeError("sharded decisions differ from the unsharded forward: %s" % json.dumps(res["vs_unsharded"]))
    return res


# ------------------------------------------------------------------------------------------------- GPU arm
DUMP_EDGES = 1 << 20        # per-edge outputs sampled for --dump-outputs: ~33 MB in all instead of ~470 MB at E = 14.7 M


def dump_outputs(path, res):
    """--dump-outputs: what one step handed its caller, as DIR/<name>.npy (float32; edge ids float64).  Per-edge arrays are taken
    at the same DUMP_EDGES edges on every run (a seeded sample, sorted, stored as edge_ids.npy) so that two builds compare edge
    for edge; h is stored whole."""
    import numpy as np
    logits = res["classified_edges"]
    E = logits[0].shape[0]
    ids = torch.randperm(E, generator=torch.Generator().manual_seed(0))[:DUMP_EDGES].sort().values
    idx = ids.to(logits[0].device)
    arrays = {"edge_ids": ids.double(), "classified_edges": torch.stack([l[idx] for l in logits]), "h": res["h"],
              "pred": res["pred"][idx].float(), "prob1": res["prob1"][idx], "edge_attr": res["edge_attr"][idx]}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())


def step_timeline(lib, step_fn, flush, barrier, dev, world, reps=5):
    """Where inside ONE step the time goes (mpn_profile_timeline: CUDA events at the phase boundaries of the step's forward call;
    each entry = ms since the forward began, median over ``reps`` steps, max over ranks).  Measured after the timed region: the
    events end the programmatic overlap between neighbouring kernels, so this step is a few percent slower than the timed ones."""
    import ctypes
    buf, names = (ctypes.c_float * 32)(), ctypes.create_string_buffer(2048)
    rows = []
    lib.mpn_profile_timeline(1)
    try:
        for r in range(reps):
            flush.fill_(r)
            barrier()
            step_fn()
            torch.cuda.synchronize(dev)
            n = lib.mpn_profile_timeline_read(buf, names, 2048)
            if n <= 0:
                return None
            rows.append([buf[i] for i in range(n)])
    finally:
        lib.mpn_profile_timeline(0)
    keys = names.value.decode().split("|")
    t = torch.tensor(rows, dtype=torch.float64, device=dev).median(dim=0).values
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {k: round(float(v), 4) for k, v in zip(keys, t.tolist())}


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import gcn_mtmc_b200 as m
    m._lib.require_device(local_rank)
    lib = m._lib.lib()
    peaks = load_peaks()
    net = make_model(dev)

    n_nodes, e_expected = workload_shape(world)
    per = n_nodes // world
    blocks = [(r * per, (r + 1) * per) for r in range(world)]
    x, ei = device_graph(n_nodes, CAMS, 0, dev, row_block=blocks[rank])
    E_local = ei.shape[1]
    tot = torch.tensor([E_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
    E_total = int(tot.item())
    sharded = m.ShardedMPN(net) if world > 1 else None
    batch = Batch()
    batch.x, batch.edge_index, batch.num_nodes = x, ei, n_nodes
    cam_host = (torch.arange(n_nodes) * CAMS // n_nodes).numpy()

    def step(x, ei):
        """One timed step -> the arrays its caller receives (logits per classified step, node embeddings, decisions, edge features)."""
        if world == 1:
            g = m.TrackletGraph(ei, n_nodes, validate="deferred")              # K0 (the edge-list check is read at the end)
            batch.x, batch.edge_index, batch.mpn_graph, batch.edge_attr = x, ei, g, None
            out, h = net(batch)                                                # K1 + K1b..K4 (+ fused decisions) in one call
            g.validate()                                                       # raises on an unsorted / out-of-range edge list
            return {"classified_edges": out["classified_edges"], "h": h, "pred": net.last_pred, "prob1": net.last_prob1,
                    "edge_attr": batch.edge_attr}
        n0, n1 = blocks[rank]
        g = m.TrackletGraph(ei, n_nodes, row_offset=n0, n_rows=n1 - n0, validate="deferred")
        out, h, pred, prob1 = sharded.forward(x, ei, None, blocks, fuse_decisions=True, graph=g)     # edge features inside the call
        g.validate()
        return {"classified_edges": out["classified_edges"], "h": h, "pred": pred, "prob1": prob1, "edge_attr": sharded.last_edge_attr}

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity gate before any timing
    parity = None
    if world == 1:
        parity = parity_gate(m, net, x, ei, dev)
    else:
        # the sharded decisions against the unsharded forward of the same graph run on every rank's own GPU
        pred_sh = step(x, ei)["pred"].clone()
        bfull = Batch()
        bfull.x, bfull.num_nodes, bfull.edge_attr = x, n_nodes, None
        bfull.mpn_graph = gfull = m.TrackletGraph.from_cameras(cam_host, dev)
        out, _ = net(bfull)
        lg, full_pred = out["classified_edges"][-1], net.last_pred
        lo, hi = int(gfull.rowptr[blocks[rank][0]].item()), int(gfull.rowptr[blocks[rank][1]].item())
        margin = (lg[lo:hi, 1] - lg[lo:hi, 0]).abs()
        diff = full_pred[lo:hi] != pred_sh
        cnt = torch.tensor([float((diff & (margin > 1e-4 * lg.abs().max())).sum().item()), float(diff.sum().item()),
                            float(pred_sh.sum().item()), float(full_pred[lo:hi].sum().item())], dtype=torch.float64, device=dev)
        dist.all_reduce(cnt)
        parity = {"checked": True, "checker": "the unsharded forward of the same graph on each rank's own GPU (itself gated against the "
                                              "fp64 oracle at N = 1)",
                  "decisions_differ_outside_margin_band": int(cnt[0].item()), "decisions_differ_total": int(cnt[1].item()),
                  "active_edges_sharded": int(cnt[2].item()), "active_edges_unsharded": int(cnt[3].item()), "path": sharded.path}
        del out, lg, full_pred, bfull, gfull, pred_sh
        torch.cuda.empty_cache()
        if parity["decisions_differ_outside_margin_band"] != 0:
            raise RuntimeError("parity gate failed: %s" % json.dumps(parity))

    clocks = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step(x, ei)
    barrier()
    launches0 = lib.mpn_kernel_launches()
    total_ms = 0.0
    for i in range(args.steps):
        last = None                                                            # the previous step's outputs are not kept alive
        flush.fill_(i & 0xFF)                                                  # L2 flush between timed iterations
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        last = step(x, ei)
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)                          # max over ranks
        total_ms += float(ms.item())
    launches = lib.mpn_kernel_launches() - launches0
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last = None
    ms_per_step = total_ms / args.steps
    value = E_total / (ms_per_step * 1e-3)
    timeline = step_timeline(lib, lambda: step(x, ei), flush, barrier, dev, world)

    # ---- e2e: the public API with HOST buffers (pinned), copies inside the timed region.  What the reference driver holds on
    # the host before it builds the graph (inference.py:383-414): the node features and the per-node camera ids; the graph tables
    # are built on the device (TrackletGraph.from_cameras, row f1).  N > 1: every rank copies only ITS rows of x and the ranks
    # all-gather them over NVLink.
    hx_all = x.cpu()
    hx = (hx_all if world == 1 else hx_all[blocks[rank][0]:blocks[rank][1]].contiguous()).pin_memory()
    hpred = torch.empty(E_local, dtype=torch.uint8).pin_memory()
    dx = torch.empty_like(x)
    n_e2e = max(3, min(args.steps, 11))

    def e2e_once():
        if world == 1:
            dx.copy_(hx, non_blocking=True)
            g = m.TrackletGraph.from_cameras(cam_host, dev)                # K0 from camera ids, on the device
            batch.x, batch.mpn_graph, batch.edge_attr = dx, g, None
            net(batch)
            return net.last_pred
        mine = dx[blocks[rank][0]:blocks[rank][1]]
        mine.copy_(hx, non_blocking=True)
        dist.all_gather_into_tensor(dx, mine)
        g = m.TrackletGraph.from_cameras(cam_host, dev, row_block=blocks[rank])
        return sharded.forward(dx, None, None, blocks, fuse_decisions=True, graph=g)[2]

    samples = []
    for i in range(n_e2e + 1):
        flush.fill_(i & 0xFF)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pred = e2e_once()
        hpred.copy_(pred, non_blocking=True)
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if i > 0:
            samples.append(float(ms.item()))
    samples.sort()
    e2e_ms = samples[len(samples) // 2]
    batch.mpn_graph = None
    # Throughput of a STREAM of host-resident graphs (the reference loops over one-graph batches, inference.py:375): GraphStream
    # keeps two graphs in flight so the PCIe copies of neighbouring graphs overlap the kernels.  Every graph still pays its own
    # H2D (features + camera ids) and D2H (decisions) inside the timed region; the region closes after the last D2H.
    pipe_depth, n_pipe = 2, max(min(args.steps, 200), 3)
    n_bits = 4 * ((E_local + 31) // 32)

    def time_pipe(packed):
        """ms per graph of the stream; packed: the decisions come back as a bit mask (1/8 of the D2H bytes)."""
        kw = dict(depth=pipe_depth, packed_decisions=packed)
        gs = m.GraphStream(net, dev, **kw) if world == 1 else m.ShardedGraphStream(sharded, blocks, dev, **kw)
        hpreds = [torch.empty(n_bits if packed else E_local, dtype=torch.uint8).pin_memory() for _ in range(pipe_depth + 1)]

        def run_pipe(k):
            for i in range(k):
                gs.submit(hx, cam_host, hpreds[i % len(hpreds)])
            gs.drain(host_sync=False)

        run_pipe(2 * pipe_depth)
        flush.fill_(1)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run_pipe(n_pipe)
        b.record()
        barrier()
        pipe = torch.tensor([a.elapsed_time(b) / n_pipe], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(pipe, op=dist.ReduceOp.MAX)                        # max over ranks
        gs.drain()
        last = hpreds[(n_pipe - 1) % len(hpreds)]
        got = torch.from_numpy(m.unpack_decisions(last, E_local)) if packed else last
        if not torch.equal(got, hpred):
            raise RuntimeError("GraphStream decisions differ from the one-at-a-time call")
        return float(pipe.item())

    pipe_ms_bytes = time_pipe(False)
    pipe_ms = time_pipe(True)
    h2d = hx.numel() * 4 + cam_host.size * 8
    d2h = n_bits

    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": workload_name(n_nodes, E_total, world),
                           "call": "graph tables from the int64 edge_index + ONE MOTMPNet.forward(data) with data.edge_attr = None "
                                   "(edge features inside the call) + fused decisions" if world == 1 else
                                   "per rank: graph tables of its row block, edge features of its rows, ShardedMPN.forward (%s)" % sharded.path,
                           "l2": "256 MiB flush between timed iterations; inputs (edge_index 235 MB) exceed L2",
                           "timing": "CUDA events per step on the launching stream, max over ranks, summed over steps"},
                "parity": parity,
                "e2e": {"value": E_total / ((pipe_ms or e2e_ms) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": pipe_ms or e2e_ms,
                        "inputs": "host node features f32 (N = 1: [N,2048]; N > 1: each rank its own rows, all-gathered over NVLink) + "
                                  "camera ids; graph tables built on the device; decisions copied back as a bit mask (1 bit per edge, "
                                  "mpn_pack_decisions / GraphStream(packed_decisions=True); unpacked on the host only for the check)",
                        "how": ("%s(depth=%d): %d graphs submitted back to back from pinned host memory, timed from the first "
                                "H2D to the last D2H (CUDA events, max over ranks); the H2D / D2H%s of neighbouring graphs overlap the "
                                "kernels, every graph pays its own copies; no L2 flush (each graph's ~600 MB of edge arrays exceed L2)"
                                % ("GraphStream" if world == 1 else "ShardedGraphStream", pipe_depth, n_pipe,
                                   "" if world == 1 else " / NVLink all-gather of the feature rows")) if pipe_ms else
                               "one graph at a time: H2D, kernels, D2H serial; median over the timed calls, max over ranks",
                        "decisions_as_bytes": {"value": E_total / (pipe_ms_bytes * 1e-3), "ms_per_step": pipe_ms_bytes,
                                               "d2h_bytes_per_step": hpred.numel(),
                                               "how": "the same stream with one uint8 per edge copied back"},
                        "one_at_a_time": {"value": E_total / (e2e_ms * 1e-3), "ms_per_step": e2e_ms,
                                          "how": "H2D, kernels, D2H (one uint8 per edge) serial per call, barrier + L2 flush between calls; median"}},
                "gpu_launches": int(launches), "clocks": clk}
    # ---- the Gram GEMM + distance epilogue alone (library-side CUDA events around that launch), every rank's own shard
    lib.mpn_profile_gram(1)
    ks = []
    for rep in range(6):
        flush.fill_(rep & 0xFF)
        if world == 1:
            m.edge_features(x, ei, graph=m.TrackletGraph.from_cameras(cam_host, dev))
        else:
            m.edge_features(x, None, graph=m.TrackletGraph.from_cameras(cam_host, dev, row_block=blocks[rank]))
        torch.cuda.synchronize()
        if rep > 0:
            ks.append(float(lib.mpn_profile_gram_ms()))
    lib.mpn_profile_gram(0)
    gram_ms = torch.tensor([sum(ks) / len(ks)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(gram_ms, op=dist.ReduceOp.MAX)
    gram_ms = float(gram_ms.item())
    tf32_peak = peaks["bf16_tflops"] / 2.0
    gram_roof = {"bound": "tensor", "achieved": FLOP_PER_EDGE_GRAM * E_local / (gram_ms * 1e-3) / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                 "ms": gram_ms, "traffic": None, "kernel": "gram_ef_kernel",
                 "peak_note": "peak = TF32 dense proxy = measured bf16 burst / 2 (SURVEY 8d; no TF32 measurement).  The kernel runs 3 fp16 "
                              "products per fp32 product (two tcgen05.mma per k-slice: N = 256 and N = 128) on the tiles that hold edges "
                              "(upper triangle at N = 1: both directions come from one tile); 'achieved' counts the algorithmic 4096 FLOP "
                              "per directed edge of the rank's shard; the time includes the distance epilogue and the moment sums"}
    gram_roof["frac"] = gram_roof["achieved"] / tf32_peak
    if world == 1:
        ph = time_phases(m, net, x, ei)
        in_step = [k for k in ph if k not in ("edge_features", "gram_ef_kernel", "enc_moments0_sweep_not_in_the_step", "graph_tables_from_edge_index")]
        fwd_ms = sum(ph[k] for k in in_step)
        hbm = peaks["hbm_gbs"]
        E = E_local
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "traffic_r2.json")
        if os.path.isfile(tp):
            traffic = json.load(open(tp))
        roof = {}
        for name, key in (("enc_moments", "enc_moments1"), ("edge_update", "edge_update"), ("node_moments", "node_moments"), ("node_apply", "node_apply")):
            t = ph[key]
            ach = BYTES_PER_EDGE[name] * E / (t * 1e-3) / 1e9
            roof[name] = {"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "ms": t,
                          "traffic": traffic.get(name)}
        ach = BYTES_PER_EDGE["forward"] * E / (fwd_ms * 1e-3) / 1e9
        roof["forward_all_kernels"] = {"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "ms": fwd_ms, "traffic": None,
                                       "note": "sum of the forward's kernels timed one by one (the node encoder runs on a side stream in the "
                                               "step); 81 B per edge: the 8 B ENC0 sweep is gone (moment sums come from the K1 epilogue)"}
        gram_roof["traffic"] = traffic.get("gram_ef_kernel")
        roof["gram_ef_kernel"] = gram_roof
        t = ph["edge_features"]
        roof["edge_features_all_kernels"] = {"bound": "tensor", "achieved": FLOP_PER_EDGE_GRAM * E / (t * 1e-3) / 1e12, "peak": tf32_peak,
                                             "unit": "TFLOP/s", "frac": FLOP_PER_EDGE_GRAM * E / (t * 1e-3) / 1e12 / tf32_peak, "ms": t, "traffic": None}
        t = ph["node_encoder"]
        roof["node_encoder"] = {"bound": "tensor", "achieved": 2 * 2691072.0 * n_nodes / (t * 1e-3) / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                                "frac": 2 * 2691072.0 * n_nodes / (t * 1e-3) / 1e12 / tf32_peak, "ms": t, "traffic": None,
                                "note": "5.38 MFLOP per node (SURVEY 8d K1b), four GEMMs + column statistics; latency bound at 4096 rows"}
        single = [k for k in roof if not k.endswith("all_kernels") and k != "node_encoder"]
        dominant = max(single, key=lambda k: roof[k]["ms"])
        line["roofline"] = dict(roof[dominant], kernel=dominant, peak_source=peaks["source"], traffic_source=traffic.get("_source"))
        line["roofline_all"] = roof
        line["phase_ms"] = ph
        line["step_timeline_ms"] = timeline
        line["s02_latency"] = s02_latency(m, dev)
        if not args.no_extras:
            extras = {}
            for name, fn in (("configs2_batched_graphs", lambda: extra_batched_graphs(m, dev)),
                             ("configs3_post_processing", lambda: extra_post_processing(m, dev)),
                             ("configs4_big_graph_1gpu", lambda: big_graph_step(m, dev, 1, 0, None))):
                try:
                    torch.cuda.empty_cache()
                    extras[name] = fn()
                except Exception as exc:                          # an extra must not take the headline line down with it
                    extras[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            line["extra"] = extras
        torch.cuda.empty_cache()
        cb = reference_sample(ef_edges=1_000_000)
        cb.pop("_model", None)
        cb.pop("_seconds", None)
        line["cpu_baseline"] = cb
    else:
        if rank == 0:
            line["roofline"] = dict(gram_roof, peak_source=peaks["source"])
        # coarse phases at N > 1 (CUDA events, max over ranks): tables, edge features, sharded forward
        n0, n1 = blocks[rank]
        phs = {}
        g = m.TrackletGraph(ei, n_nodes, row_offset=n0, n_rows=n1 - n0)
        ea = m.edge_features(x, ei, graph=g)
        for name, fn in (("graph_tables", lambda: m.TrackletGraph(ei, n_nodes, row_offset=n0, n_rows=n1 - n0, validate="deferred")),
                         ("edge_features", lambda: m.edge_features(x, ei, graph=g)),
                         ("sharded_forward", lambda: sharded.forward(x, ei, ea, blocks, fuse_decisions=True, graph=g))):
            acc = 0.0
            for rep in range(4):
                flush.fill_(rep)
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                barrier()
                t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                if rep > 0:
                    acc += float(t.item()) / 3
            phs[name] = acc
        del g, ea
        torch.cuda.empty_cache()
        c5 = None
        if not args.no_extras:
            try:
                c5 = big_graph_step(m, dev, world, rank, m.ShardedMPN)
            except Exception as exc:
                c5 = {"error": "%s: %s" % (type(exc).__name__, exc)}
        if rank == 0:
            line["phase_ms"] = phs
            line["step_timeline_ms"] = timeline
            line["c5_strong"] = c5
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE configs (extra / c5_strong blocks)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0; "
                                                           "per-edge arrays at a fixed sample of edges)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the timed GPU path; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
