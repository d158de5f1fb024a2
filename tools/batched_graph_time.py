"""Batched graphs from camera layouts, timed with device events after warm-up: the tables of configs[2] (2000 graphs x N=300,
4 cameras) and of a mixed batch of ragged graphs with 3 to 8 cameras, built from the offset edge_index (today's route:
edge_index built on the device, then TrackletGraph(ei, N, ptr=)) and by TrackletGraph.from_cameras(cam, ptr=); the per-graph
normalize_columns loop against normalize_columns(x, ptr=); and the whole batched step both ways (tables, edge features, forward,
decisions, post_processing_batched).  Both routes are checked for identical tables and decisions before anything is timed.
Writes JSON (default profiles/r3_batched_graph_build.json).

    python tools/batched_graph_time.py [out.json]
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
import gcn_mtmc_b200 as m

dev = torch.device("cuda", 0)
CFG = {"CUTTING": True, "PRUNING": True, "SPLITTING": True}
HBM_BYTES_PER_S = 7.7e12              # HGX B200 data sheet, one GPU


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, reps=10, warm=2):
    ts = bench.time_events(fn, None, reps, warm=warm)
    return {"ms_median": ts[len(ts) // 2], "ms_min": ts[0], "ms_max": ts[-1], "reps": reps}


def uniform_batch(G, n, C):
    return np.tile(np.arange(n) * C // n, G), np.arange(G + 1) * n


def ragged_batch(G, seed):
    """G graphs of 3..8 cameras (ids drawn from 0..15), 20..80 nodes per camera."""
    rng = np.random.default_rng(seed)
    cams = []
    for _ in range(G):
        ids = np.sort(rng.choice(16, size=int(rng.integers(3, 9)), replace=False))
        cams.append(np.repeat(ids, rng.integers(20, 81, size=ids.size)))
    return np.concatenate(cams), np.cumsum([0] + [c.size for c in cams]), [int(np.unique(c).size) for c in cams]


def offset_edge_index_uniform(G, n, C):
    """configs[2] as bench.py builds it: one graph's edge_index on the device, offset by every graph's first node."""
    _, tmpl = bench.device_graph(n, C, 0, dev)
    E1 = tmpl.shape[1]
    return (tmpl[None] + (torch.arange(G, device=dev) * n)[:, None, None]).permute(1, 0, 2).reshape(2, G * E1).contiguous()


def offset_edge_index_ragged(cam_d, ptr):
    """inference.py:407-413 for every graph on the device (cartesian_prod per camera), offset by ptr[g] and concatenated."""
    parts = []
    for g in range(ptr.size - 1):
        c = cam_d[ptr[g]:ptr[g + 1]]
        nodes = torch.arange(int(ptr[g]), int(ptr[g + 1]), device=dev)
        for k in torch.unique(c).tolist():
            parts.append(torch.cartesian_prod(nodes[c == k], nodes[c != k]))
    return torch.cat(parts, dim=0).t().contiguous()


def same_tables(a, b):
    torch.cuda.synchronize()
    if (a.n_edges, a.chunk, a.max_tasks, a.n_graphs, a.max_graph_nodes) != (b.n_edges, b.chunk, b.max_tasks, b.n_graphs, b.max_graph_nodes):
        return False
    nt = int(a.n_tasks.item())
    return (all(torch.equal(getattr(a, k), getattr(b, k)) for k in ("rowptr", "taskptr", "n_tasks", "node_gid", "graph_nptr"))
            and torch.equal(a.col[:a.n_edges], b.col[:b.n_edges]) and torch.equal(a.task_row[:nt], b.task_row[:nt]))


def tables_section(name, cam, ptr, make_ei):
    ptr_d = torch.from_numpy(ptr).to(dev)
    N = int(cam.size)
    ei = make_ei()
    ref = m.TrackletGraph(ei, N, ptr=ptr_d)
    new = m.TrackletGraph.from_cameras(cam, dev, ptr=ptr)
    res = {"graphs": int(ptr.size - 1), "nodes": N, "edges": int(ei.shape[1]), "tables_identical": same_tables(ref, new)}
    if not res["tables_identical"]:
        raise RuntimeError("%s: from_cameras(ptr=) tables differ from the edge_index route" % name)
    del ref, new
    res["edge_index_build"] = timed(make_ei, reps=3 if name == "ragged" else 10, warm=1)
    res["tables_from_edge_index"] = timed(lambda: m.TrackletGraph(ei, N, ptr=ptr_d))
    res["from_cameras_ptr"] = timed(lambda: m.TrackletGraph.from_cameras(cam, dev, ptr=ptr))
    res["today_route_total_ms"] = res["edge_index_build"]["ms_median"] + res["tables_from_edge_index"]["ms_median"]
    res["col_write_floor_ms"] = 4.0 * res["edges"] / HBM_BYTES_PER_S * 1e3
    print(name, json.dumps(res), flush=True)
    return res


def normalize_section(G, n):
    x = torch.randn(G * n, bench.FEAT_DIM, generator=torch.Generator(device=dev).manual_seed(7), device=dev)
    ptr = np.arange(G + 1) * n
    out_loop, out = torch.empty_like(x), torch.empty_like(x)

    def loop():
        for g in range(G):
            m.normalize_columns(x[g * n:(g + 1) * n], out=out_loop[g * n:(g + 1) * n])
    loop()
    m.normalize_columns(x, out=out, ptr=ptr)
    torch.cuda.synchronize()
    d = (out.view(torch.int32).long() - out_loop.view(torch.int32).long()).abs().max().item()
    res = {"graphs": G, "nodes_per_graph": n, "D": bench.FEAT_DIM, "x_bytes": x.numel() * 4, "max_ulp_vs_loop": int(d)}
    res["per_graph_loop"] = timed(loop, reps=5, warm=1)
    res["batched"] = timed(lambda: m.normalize_columns(x, out=out, ptr=ptr))
    res["batched_bytes_per_s"] = 2 * res["x_bytes"] / (res["batched"]["ms_median"] * 1e-3)
    res["batched_fraction_of_hbm_datasheet"] = res["batched_bytes_per_s"] / HBM_BYTES_PER_S
    print("normalize", json.dumps(res), flush=True)
    return res


def step_section(name, cam, ptr, make_ei, n_cams):
    net = bench.make_model(dev)
    net.fuse_decisions = True
    x = torch.randn(int(cam.size), bench.FEAT_DIM, generator=torch.Generator(device=dev).manual_seed(3), device=dev)
    x = m.normalize_columns(x, ptr=ptr)
    ptr_d = torch.from_numpy(ptr).to(dev)

    def today():
        b = bench.Batch()
        b.x, b.edge_index, b.num_nodes, b.ptr, b.edge_attr = x, make_ei(), int(cam.size), ptr_d, None
        net(b)
        return m.post_processing_batched(n_cams, net.last_pred, dict(CFG), b, net.last_prob1)

    def new():
        b = bench.Batch()
        b.x, b.num_nodes, b.edge_attr = x, int(cam.size), None
        b.mpn_graph = m.TrackletGraph.from_cameras(cam, dev, ptr=ptr)
        net(b)
        return m.post_processing_batched(n_cams, net.last_pred, dict(CFG), b, net.last_prob1)
    ID_a, P_a, nc_a = today()
    ID_b, P_b, nc_b = new()
    res = {"decisions_identical": bool(torch.equal(ID_a, ID_b) and torch.equal(P_a, P_b) and torch.equal(nc_a, nc_b))}
    if not res["decisions_identical"]:
        raise RuntimeError("%s: the two routes give different decisions" % name)
    del ID_a, P_a, ID_b, P_b
    reps = 3 if name == "ragged" else 5
    res["edge_index_route"] = timed(today, reps=reps, warm=1)
    res["from_cameras_route"] = timed(new, reps=reps, warm=1)
    print(name, "step", json.dumps(res), flush=True)
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r3_batched_graph_build.json")
    m._lib.require_device(0)
    res = {"gpu": card(), "timing": "CUDA events around each call after warm-up, median of the repetitions; ms per call",
           "hbm_datasheet_bytes_per_s": HBM_BYTES_PER_S}
    G, n, C = 2000, 300, 4
    cam_u, ptr_u = uniform_batch(G, n, C)
    cam_r, ptr_r, ncam_r = ragged_batch(1000, 11)
    cam_r_d = torch.from_numpy(cam_r).to(dev)
    res["ragged_batch"] = {"graphs": 1000, "cameras": "3..8 per graph, ids from 0..15", "nodes_per_camera": "20..80"}
    res["tables_configs2"] = tables_section("configs2", cam_u, ptr_u, lambda: offset_edge_index_uniform(G, n, C))
    res["tables_ragged"] = tables_section("ragged", cam_r, ptr_r, lambda: offset_edge_index_ragged(cam_r_d, ptr_r))
    res["normalize_configs2"] = normalize_section(G, n)
    res["step_configs2"] = step_section("configs2", cam_u, ptr_u, lambda: offset_edge_index_uniform(G, n, C), C)
    res["step_ragged"] = step_section("ragged", cam_r, ptr_r, lambda: offset_edge_index_ragged(cam_r_d, ptr_r), ncam_r)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
