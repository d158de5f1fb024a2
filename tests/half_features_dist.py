"""Multi-GPU check of 16-bit node features, launched by torchrun (one rank per GPU, NCCL):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29583 tests/half_features_dist.py

Each rank runs its row-block shard through ShardedMPN (fused collectives, shared symmetric Gram; and the NCCL schedule) with fp16
and bf16 x, and compares every output bit for bit with the same call on x.float().  ShardedGraphStream then takes 16-bit host rows
(all-gathered in half) and must give the decisions of the direct sharded call on the fp32 widening.
"""
import copy
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gcn_mtmc_b200 as m                      # noqa: E402
from oracle import mpn_oracle as mo            # noqa: E402


def model(dev, L):
    params = mo.shipped_model_params(L, 1, 128, (96, 64))
    net = m.MOTMPNet(copy.deepcopy(params), None, "resnet101")
    net.load_state_dict(mo.init_weights(params, "resnet101", 2), strict=True)
    return net.to(dev).eval()


def check_forward(rank, world, dev, dt):
    net = model(dev, 2)
    N, C = 600, 4
    x, ei, cam, _ = mo.synth_graph(N, C, 3, D=128, planted=True)
    per = N // world
    blocks = [(r * per, (r + 1) * per if r + 1 < world else N) for r in range(world)]
    g = m.TrackletGraph.from_cameras(cam, dev, row_block=blocks[rank])
    xh = x.to(dev).to(dt)
    xf = xh.float()
    for fused in (True, False):
        sh = m.ShardedMPN(net, fused=fused)
        outs = []
        for xx in (xh, xf):
            out, h, pred, prob1 = sh.forward(xx, None, None, blocks, fuse_decisions=True, graph=g)
            torch.cuda.synchronize()
            outs.append(([o.clone() for o in out["classified_edges"]], h.clone(), pred.clone(), prob1.clone(),
                         sh.last_edge_attr.clone()))
        if fused:
            assert sh.shared_gram_used(), "the shared-Gram path was not taken"
        a, b = outs
        assert all(torch.equal(u, v) for u, v in zip(a[0], b[0])), "sharded logits differ (fused=%s)" % fused
        for u, v in zip(a[1:], b[1:]):
            assert torch.equal(u, v), "sharded h / decisions / edge features differ (fused=%s)" % fused


def check_stream(rank, world, dev, dt):
    net = model(dev, 2)
    sh = m.ShardedMPN(net)
    N, C = 128 * world * 4, 4
    per = N // world
    blocks = [(r * per, (r + 1) * per) for r in range(world)]
    cam = np.arange(N) * C // N
    rows, refs = [], []
    for seed in range(4):
        x, _, _, _ = mo.synth_graph(N, C, seed, D=128, planted=True)
        xh = x.to(dt)
        g = m.TrackletGraph.from_cameras(cam, dev, row_block=blocks[rank])
        refs.append(sh.forward(xh.float().to(dev), None, None, blocks, fuse_decisions=True, graph=g)[2].cpu())
        rows.append(xh[blocks[rank][0]:blocks[rank][1]].contiguous().pin_memory())
    gs = m.ShardedGraphStream(sh, blocks, dev, depth=2)
    outs = [torch.zeros(refs[0].numel(), dtype=torch.uint8).pin_memory() for _ in rows]
    for xr, o in zip(rows, outs):
        gs.submit(xr, cam, o)
    gs.drain()
    for o, r in zip(outs, refs):
        assert torch.equal(o, r), "ShardedGraphStream decisions on 16-bit rows differ from the fp32 call"
    assert all(s.x_dev.dtype == dt for s in gs.slots if s.x_dev is not None)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    for dt in (torch.float16, torch.bfloat16):
        check_forward(rank, world, dev, dt)
        check_stream(rank, world, dev, dt)
    dist.barrier()
    if rank == 0:
        print("half_features_dist ok: world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
