"""post_processing_batched at BASELINE configs[2] scale: 2000 S02-shaped planted predicted graphs (300 nodes, 4 cameras, 67,500
edges each) in one call, against the per-graph post_processing loop over all 2000 graphs; then configs[2] end to end (batched
forward with fused decisions + batched post-processing).  Writes JSON (default profiles/r3_batched_post.json).

    python tools/batched_post_time.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import gcn_mtmc_b200 as m
from oracle import postproc_oracle as po

dev = torch.device("cuda", 0)
G, N, C = 2000, 300, 4
CFG = {"CUTTING": True, "PRUNING": True, "SPLITTING": True}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), r


def median_of(fn, reps=5):
    fn()                                                       # warm-up (workspace, pinned staging)
    ts = sorted(wall(fn)[0] for _ in range(reps))
    return ts[len(ts) // 2], ts


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r3_batched_post.json")
    res = {"gpu": card(), "graphs": G, "nodes_per_graph": N, "cameras": C}
    t0 = time.perf_counter()
    gen = [po.planted_prediction_graph(N, C, 20000 + k, dense=True) for k in range(G)]
    src, dst = gen[0][0], gen[0][1]
    E1 = src.size
    tmpl = torch.from_numpy(np.stack([src, dst])).to(dev)
    ei = (tmpl[None] + (torch.arange(G, device=dev) * N)[:, None, None]).permute(1, 0, 2).reshape(2, G * E1).contiguous()
    data = bench.Batch()
    data.x, data.edge_index, data.num_nodes, data.ptr = torch.zeros(G * N, 1, device=dev), ei, G * N, torch.arange(G + 1, device=dev) * N
    pred = torch.from_numpy(np.concatenate([g[3] for g in gen])).to(dev)
    prob = torch.from_numpy(np.concatenate([g[2] for g in gen])).to(dev)
    res["edges_per_graph"] = E1
    res["active_edges"] = int(pred.sum())
    del gen
    print("built %d graphs in %.1f s" % (G, time.perf_counter() - t0), flush=True)
    m.graph_for(data, ei, G * N)                               # tables built once, as after a batched forward
    for numbering in ("canonical", "reference"):
        ms, ts = median_of(lambda: m.post_processing_batched(C, pred.clone(), dict(CFG), data, prob, numbering=numbering))
        st = m.split_stats()
        res["batched_" + numbering] = {"ms_median": ms, "ms_runs": ts, "us_per_graph": 1e3 * ms / G,
                                       "host_order_graphs": st["host_order_graphs"], "tied_edges": st["tied_edges"],
                                       "rounds": st["rounds"]}
        print(numbering, res["batched_" + numbering], flush=True)
    # the per-graph loop over all 2000 graphs (one graph's tables reused: all graphs share the edge list)
    one = bench.Batch()
    one.x, one.edge_index, one.num_nodes = torch.zeros(N, 1, device=dev), tmpl, N
    m.graph_for(one, tmpl, N)
    ID_b, P_b, _ = m.post_processing_batched(C, pred.clone(), dict(CFG), data, prob)

    def loop():
        out = []
        for k in range(G):
            e0, e1 = k * E1, (k + 1) * E1
            out.append(m.post_processing(C, None, None, pred[e0:e1].clone(), None, dict(CFG), one, prob[e0:e1]))
        return out
    m.post_processing(C, None, None, pred[:E1].clone(), None, dict(CFG), one, prob[:E1])
    t_loop, outs = wall(loop)
    equal = all(torch.equal(P_b[k * E1:(k + 1) * E1], outs[k][1]) and torch.equal(ID_b[k * N:(k + 1) * N], outs[k][0]) for k in range(G))
    res["per_graph_loop_reference"] = {"ms": t_loop, "us_per_graph": 1e3 * t_loop / G}
    res["batched_equals_loop"] = bool(equal)
    res["speedup_vs_loop_reference"] = t_loop / res["batched_reference"]["ms_median"]
    print("loop %.1f ms, equal %s, speedup %.1fx" % (t_loop, equal, res["speedup_vs_loop_reference"]), flush=True)
    del outs
    # configs[2] end to end: batched forward with fused decisions, then the batched post-processing
    net = bench.make_model(dev)
    net.fuse_decisions = True
    g = torch.Generator(device=dev).manual_seed(3)
    x = torch.randn(G, N, bench.FEAT_DIM, generator=g, device=dev)
    x = torch.nn.functional.normalize(x, p=2, dim=1).reshape(G * N, bench.FEAT_DIM)
    b = bench.Batch()
    b.x, b.edge_index, b.num_nodes, b.ptr = x, ei, G * N, data.ptr

    def e2e():
        b.edge_attr = None
        b._mpn_b200_graph = None
        net(b)
        return m.post_processing_batched(C, net.last_pred, dict(CFG), b, net.last_prob1)

    def fwd():
        b.edge_attr = None
        b._mpn_b200_graph = None
        return net(b)
    ms_fwd, _ = median_of(fwd)
    ms_e2e, ts = median_of(e2e)
    st = m.split_stats()
    res["configs2_end_to_end"] = {"ms_median": ms_e2e, "ms_runs": ts, "forward_only_ms_median": ms_fwd, "us_per_graph": 1e3 * ms_e2e / G,
                                  "active_edges": int(net.last_pred.sum()), "host_order_graphs": st["host_order_graphs"],
                                  "tied_edges": st["tied_edges"]}
    print("e2e", res["configs2_end_to_end"], flush=True)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
