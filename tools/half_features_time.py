"""fp32 / fp16 / bf16 node features, timed in one session with the dtypes alternated: outputs are first checked to be identical
to the fp32 widening of the same 16-bit features, then every figure is the median of CUDA-event timings after warm-up, with a
256 MiB L2 flush before each timed call (as bench.py).  Writes JSON (default profiles/r3_half_features.json).

  1. the configs[1] step (tables from the camera layout + fused forward with edge features + decisions), and the kernels that
     read x inside it (torch.profiler, separate pass): ge_col_mean + ge_center_split, absmax + split_f16_bn of encoder layer 0;
  2. the GraphStream end to end of configs[1] (pinned host features in, bit-mask decisions out, depth 2), per graph;
  3. a configs[2] batch (2000 graphs x 300 nodes, 4 cameras) from pinned host memory: H2D, normalize_columns(ptr=),
     from_cameras(ptr=), forward, post_processing_batched;
  4. with >= 2 GPUs, the ShardedGraphStream end to end of bench.py's sharded workload at 2 / 4 / 8 GPUs (each rank copies its
     16-bit or fp32 rows in, NVLink all-gather, shard forward, bit-mask decisions out), one torchrun process per GPU, max over
     ranks; with fewer GPUs the section records how many were visible.

    python tools/half_features_time.py [out.json]
"""
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import gcn_mtmc_b200 as m

dev = torch.device("cuda", 0)
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
NAMES = {torch.float32: "fp32", torch.float16: "fp16", torch.bfloat16: "bf16"}
CFG = {"CUTTING": True, "PRUNING": True, "SPLITTING": True}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def med(ts):
    ts = sorted(ts)
    return {"ms_median": ts[len(ts) // 2], "ms_min": ts[0], "ms_max": ts[-1], "reps": len(ts)}


def alternate(fns, flush, reps, warm=2):
    """{dtype: timings} of fns[dtype]() with the dtypes interleaved rep by rep."""
    ts = {k: [] for k in fns}
    for i in range(reps + warm):
        for k, fn in fns.items():
            flush.fill_(i & 0xFF)
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            e.record()
            e.synchronize()
            if i >= warm:
                ts[k].append(a.elapsed_time(e))
    return {NAMES[k]: med(v) for k, v in ts.items()}


def kernel_ms(fn, names, reps=3):
    """Mean device time per call of the kernels whose names contain one of `names` (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {n: 0.0 for n in names}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        t = ev.cuda_time_total if t is None else t
        for n in names:
            if n in ev.key:
                out[n] += t / 1e3 / reps
    return out


def step_section(net, flush):
    N, C = bench.NODES_1GPU, bench.CAMS
    x32 = bench.device_features(N, 0, dev)
    cam = (np.arange(N) * C // N)
    xs = {dt: x32.to(dt) for dt in DTYPES}

    def step(x):
        b = bench.Batch()
        b.x, b.num_nodes, b.edge_attr = x, N, None
        b.mpn_graph = m.TrackletGraph.from_cameras(cam, dev)
        out, h = net(b)
        return out["classified_edges"][-1], h, net.last_pred, b.edge_attr

    checks = {}
    for dt in (torch.float16, torch.bfloat16):
        a, b = step(xs[dt]), step(xs[dt].float())
        checks[NAMES[dt]] = all(torch.equal(u, v) for u, v in zip(a, b))
        if not checks[NAMES[dt]]:
            raise RuntimeError("configs[1] step on %s x differs from its fp32 widening" % NAMES[dt])
        del a, b
    res = {"nodes": N, "cameras": C, "D": x32.shape[1], "outputs_identical_to_fp32_widening": checks,
           "x_bytes": {NAMES[dt]: xs[dt].numel() * xs[dt].element_size() for dt in DTYPES}}
    res["step"] = alternate({dt: (lambda dt=dt: step(xs[dt])) for dt in DTYPES}, flush, reps=15)
    names = ["ge_col_mean_kernel", "ge_center_split_kernel", "absmax_kernel", "split_f16_bn_kernel"]
    res["x_reading_kernels_ms"] = {NAMES[dt]: kernel_ms(lambda dt=dt: step(xs[dt]), names) for dt in DTYPES}
    print("configs1 step", json.dumps(res), flush=True)
    return res


def stream_section(net, n_graphs=24):
    N, C = bench.NODES_1GPU, bench.CAMS
    cam = (np.arange(N) * C // N)
    x32 = bench.device_features(N, 0, dev)
    E = int(m.TrackletGraph.from_cameras(cam, dev).n_edges)
    hosts = {dt: x32.to(dt).cpu().pin_memory() for dt in DTYPES}
    ref = {}
    for dt in DTYPES:                                          # decisions of the direct call on the fp32 widening
        b = bench.Batch()
        b.x, b.num_nodes, b.edge_attr = hosts[dt].to(dev).float(), N, None
        b.mpn_graph = m.TrackletGraph.from_cameras(cam, dev)
        net(b)
        ref[dt] = torch.from_numpy(np.packbits(net.last_pred.cpu().numpy(), bitorder="little"))
    outs = [torch.zeros(4 * ((E + 31) // 32), dtype=torch.uint8).pin_memory() for _ in range(3)]
    ts = {dt: [] for dt in DTYPES}
    ok = {}
    for rnd in range(4):                                      # round 0 warms every dtype's slots
        for dt in DTYPES:
            gs = m.GraphStream(net, dev, depth=2, packed_decisions=True)
            for i in range(3):
                gs.submit(hosts[dt], cam, outs[i % 3])
            gs.drain()
            ok[NAMES[dt]] = all(torch.equal(o[:ref[dt].numel()], ref[dt]) for o in outs)
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n_graphs):
                gs.submit(hosts[dt], cam, outs[i % 3])
            gs.drain(host_sync=False)
            e.record()
            e.synchronize()
            if rnd > 0:
                ts[dt].append(a.elapsed_time(e) / n_graphs)
    if not all(ok.values()):
        raise RuntimeError("GraphStream decisions differ from the direct call: %s" % ok)
    res = {"graphs_per_timed_run": n_graphs, "depth": 2, "decisions": "bit mask", "decisions_identical_to_direct_call": ok,
           "h2d_bytes_per_graph": {NAMES[dt]: hosts[dt].numel() * hosts[dt].element_size() for dt in DTYPES},
           "ms_per_graph": {NAMES[dt]: med(v) for dt, v in ts.items()}}
    print("graphstream", json.dumps(res), flush=True)
    return res


def batch_section(net, flush, G=2000, n=300, C=4):
    cam = np.tile(np.arange(n) * C // n, G)
    ptr = np.arange(G + 1) * n
    g0 = torch.Generator(device=dev).manual_seed(3)
    x32 = torch.randn(G * n, bench.FEAT_DIM, generator=g0, device=dev)
    stages = ["h2d", "normalize_columns_ptr", "from_cameras_ptr", "forward", "post_processing_batched"]
    res = {"graphs": G, "nodes_per_graph": n, "cameras": C, "D": bench.FEAT_DIM}
    times = {dt: {s: [] for s in stages + ["total"]} for dt in DTYPES}
    decisions = {}
    for dt in DTYPES:
        res.setdefault("h2d_bytes", {})[NAMES[dt]] = x32.numel() * (4 if dt == torch.float32 else 2)
    for rep in range(4):                                       # rep 0: warm-up and the identity check
        for dt in DTYPES:
            host = x32.to(dt).cpu().pin_memory()
            xd = torch.empty(host.shape, dtype=dt, device=dev)
            flush.fill_(rep & 0xFF)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(stages) + 1)]
            ev[0].record()
            xd.copy_(host, non_blocking=True)
            ev[1].record()
            xn = m.normalize_columns(xd, ptr=ptr)
            ev[2].record()
            b = bench.Batch()
            b.x, b.num_nodes, b.edge_attr = xn, G * n, None
            b.mpn_graph = m.TrackletGraph.from_cameras(cam, dev, ptr=ptr)
            ev[3].record()
            net(b)
            ev[4].record()
            ID, P, ncl = m.post_processing_batched(C, net.last_pred, dict(CFG), b, net.last_prob1)
            ev[5].record()
            ev[5].synchronize()
            if rep == 0:
                ref_x = xd.float() if dt != torch.float32 else None
                decisions[dt] = (ID.clone(), P.clone())
                if ref_x is not None:                          # the same batch on the fp32 widening, on the device
                    b2 = bench.Batch()
                    b2.x, b2.num_nodes, b2.edge_attr = m.normalize_columns(ref_x, ptr=ptr), G * n, None
                    b2.mpn_graph = m.TrackletGraph.from_cameras(cam, dev, ptr=ptr)
                    net(b2)
                    ID2, P2, _ = m.post_processing_batched(C, net.last_pred, dict(CFG), b2, net.last_prob1)
                    same = bool(torch.equal(ID, ID2) and torch.equal(P, P2) and torch.equal(xn, b2.x))
                    res.setdefault("outputs_identical_to_fp32_widening", {})[NAMES[dt]] = same
                    if not same:
                        raise RuntimeError("configs[2] batch on %s x differs from its fp32 widening" % NAMES[dt])
                    del b2, ID2, P2, ref_x
            else:
                for i, s in enumerate(stages):
                    times[dt][s].append(ev[i].elapsed_time(ev[i + 1]))
                times[dt]["total"].append(ev[0].elapsed_time(ev[-1]))
            del host, xd, xn, b, ID, P, ncl
            torch.cuda.empty_cache()
    res["ms"] = {NAMES[dt]: {s: med(v)["ms_median"] for s, v in t.items()} for dt, t in times.items()}
    res["h2d_bytes_per_s"] = {NAMES[dt]: res["h2d_bytes"][NAMES[dt]] / (res["ms"][NAMES[dt]]["h2d"] * 1e-3) for dt in DTYPES}
    print("configs2 batch", json.dumps(res), flush=True)
    return res


def sharded_worker(out_path, n_graphs=48):
    """One rank of section 4 (launched by torchrun from sharded_section)."""
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    d = torch.device("cuda", local)
    torch.cuda.set_device(d)
    dist.init_process_group("nccl", device_id=d)
    net = bench.make_model(d)
    sh = m.ShardedMPN(net)
    n_nodes, _ = bench.workload_shape(world)
    per = n_nodes // world
    blocks = [(r * per, (r + 1) * per) for r in range(world)]
    n0, n1 = blocks[rank]
    cam = (np.arange(n_nodes) * bench.CAMS // n_nodes)
    x32 = bench.device_features(n_nodes, 0, d)
    rows = {dt: x32[n0:n1].to(dt).cpu().pin_memory() for dt in DTYPES}
    ref = {}
    for dt in DTYPES:                                          # decisions of the direct sharded call on the fp32 widening
        g = m.TrackletGraph.from_cameras(cam, d, row_block=blocks[rank])
        pred = sh.forward(x32.to(dt).float(), None, None, blocks, fuse_decisions=True, graph=g)[2]
        ref[dt] = torch.from_numpy(np.packbits(pred.cpu().numpy(), bitorder="little"))
    E = int(ref[torch.float32].numel() * 8)
    outs = [torch.zeros(4 * ((E + 31) // 32), dtype=torch.uint8).pin_memory() for _ in range(3)]
    ts, ok = {dt: [] for dt in DTYPES}, {}
    for rnd in range(4):                                       # round 0 warms every dtype's slots; dtypes alternated
        for dt in DTYPES:
            gs = m.ShardedGraphStream(sh, blocks, d, depth=2, packed_decisions=True)
            for i in range(4):
                gs.submit(rows[dt], cam, outs[i % 3])
            gs.drain()
            ok[NAMES[dt]] = all(torch.equal(o[:ref[dt].numel()], ref[dt]) for o in outs)
            dist.barrier()
            torch.cuda.synchronize()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n_graphs):
                gs.submit(rows[dt], cam, outs[i % 3])
            gs.drain(host_sync=False)
            e.record()
            e.synchronize()
            dist.barrier()
            t = torch.tensor([a.elapsed_time(e) / n_graphs], dtype=torch.float64, device=d)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if rnd > 0:
                ts[dt].append(float(t.item()))
    good = torch.tensor([float(all(ok.values()))], device=d)
    dist.all_reduce(good, op=dist.ReduceOp.MIN)
    if rank == 0:
        res = {"world": world, "nodes": n_nodes, "graphs_per_timed_run": n_graphs, "depth": 2, "decisions": "bit mask",
               "decisions_identical_to_direct_call_on_fp32_widening": bool(good.item() == 1.0),
               "h2d_bytes_per_rank_and_graph": {NAMES[dt]: rows[dt].numel() * rows[dt].element_size() for dt in DTYPES},
               "ms_per_graph_max_over_ranks": {NAMES[dt]: med(v) for dt, v in ts.items()}}
        with open(out_path, "w") as f:
            json.dump(res, f)
    dist.destroy_process_group()


def sharded_section():
    n = torch.cuda.device_count()
    worlds = [w for w in (2, 4, 8) if w <= n]
    if not worlds:
        return "not measured: %d GPU visible (the ShardedGraphStream needs at least 2)" % n
    res = {}
    for w in worlds:
        with tempfile.TemporaryDirectory() as tmp:
            out = os.path.join(tmp, "sharded.json")
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(w), "--master-addr",
                   "127.0.0.1", "--master-port", "29591", os.path.abspath(__file__), "--sharded-worker", out]
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
            if r.returncode != 0 or not os.path.isfile(out):
                raise RuntimeError("sharded section at %d GPUs failed:\n%s" % (w, (r.stdout + r.stderr)[-3000:]))
            with open(out) as f:
                res[str(w)] = json.load(f)
        if not res[str(w)]["decisions_identical_to_direct_call_on_fp32_widening"]:
            raise RuntimeError("ShardedGraphStream decisions at %d GPUs differ from the direct call" % w)
        print("sharded", w, json.dumps(res[str(w)]), flush=True)
    return res


def main():
    if len(sys.argv) > 2 and sys.argv[1] == "--sharded-worker":
        sharded_worker(sys.argv[2])
        return
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r3_half_features.json")
    m._lib.require_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = {"gpu": "%s (name, power limit, max SM clock; read in the same run)" % card(),
           "timing": "CUDA events, median over repetitions after warm-up, dtypes alternated; 256 MiB L2 flush before each timed call "
                     "(sections 1 and 3); ms"}
    net = bench.make_model(dev)
    res["configs1_step"] = step_section(net, flush)
    res["configs1_graphstream"] = stream_section(net)
    res["configs2_batch_from_host"] = batch_section(net, flush)
    del net
    torch.cuda.empty_cache()
    res["sharded_graphstream"] = sharded_section()
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
