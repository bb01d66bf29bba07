#!/usr/bin/env python
"""Multi-process check of the fused data-parallel update (csrc/peer_adam.cu) on real peer GPUs.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/peer_check.py

(1) flat buffers: PeerAdam over CUDA-IPC-mapped arenas vs NCCL all-reduce(AVG) + torch.optim.Adam on every rank --
    replicas bitwise identical across ranks, values within fp32 rounding of the library path;
(2) the gbm-shape train step: Trainer(peer_update=True) vs Trainer(peer_update=False), eager and as a CUDA graph --
    same loss trajectory, same parameters.
Prints one JSON line on rank 0; exits non-zero on any mismatch or on a peer wait that timed out."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def same_on_all_ranks(t, world):
    got = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(got, t.contiguous())
    return all(torch.equal(g, got[0]) for g in got)


def flat_check(dev, world, rank):
    from multilevel_gnn_b200.train import GradBucket, PeerAdam, PeerArena
    shapes = [(257, 33), (1000,), (64, 64), (3,), (500001,)]
    g0 = torch.Generator().manual_seed(5)
    init = [torch.randn(s, generator=g0) for s in shapes]
    params = [torch.nn.Parameter(t.clone().to(dev)) for t in init]
    arena = PeerArena(GradBucket.padded_size(params, 4 * world), world, rank, dev)
    bucket = GradBucket(params, flat=arena.grad, align=4 * world)
    opt = PeerAdam(bucket, arena, lr=1e-2, betas=(0.9, 0.999), weight_decay=1e-2)
    ref = [torch.nn.Parameter(t.clone().to(dev)) for t in init]
    ref_opt = torch.optim.Adam(ref, lr=1e-2, betas=(0.9, 0.999), weight_decay=1e-2)
    g = torch.Generator().manual_seed(100 + rank)
    dist.barrier()
    for step in range(6):
        grads = [torch.randn(s, generator=g).to(dev) for s in shapes]
        for p, x in zip(ref, grads):
            p.grad = x.clone()
            dist.all_reduce(p.grad, op=dist.ReduceOp.AVG)
        ref_opt.step()
        bucket.store(grads)
        opt.step()
    torch.cuda.synchronize()
    assert arena.status() == 0, "rank %d: a peer wait timed out" % rank
    err = 0.0
    for p, q in zip(params, ref):
        assert same_on_all_ranks(p.data, world), "replicas differ across ranks"
        torch.testing.assert_close(p.data, q.data, rtol=2e-5, atol=2e-6)
        err = max(err, float((p.data - q.data).abs().max()))
    assert float(opt.step_dev.item()) == 6.0 and not opt.failed()
    return err


def trainer_check(dev, world, rank, graph):
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200.train import Trainer
    args = m.configs.make_args("gbm")
    B = 4
    out = {}
    for mode in ("peer", "nccl"):
        torch.manual_seed(0)
        model = m.MultilevelGNN(args)
        m.synth.multilevel_params(model)
        model.to(dev)
        model.pathway_indexs = model.pathway_indexs.to(dev)
        batch = m.synth.multilevel_batch(batch_size=B, seed=100 + rank).to(dev)
        batch.topology_key = "fold0"

        weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(dev)
        tr = Trainer(model, args, weight, world_size=world, peer_update=(mode == "peer"))
        assert (tr.peer is not None) == (mode == "peer")
        losses = []
        for _ in range(3):
            losses.append(float(tr.step(batch).item()))
        if graph:
            tr.capture(batch)
            for _ in range(4):
                losses.append(float(tr.step().item()))
        torch.cuda.synchronize()
        if tr.peer is not None:
            assert tr.peer.status() == 0, "rank %d: a peer wait timed out" % rank
        ids = {id(p) for p in tr.params}
        flat = torch.cat([p.data.reshape(-1) for p in model.parameters() if id(p) in ids])
        assert same_on_all_ranks(flat, world), "%s: parameters differ across ranks" % mode
        out[mode] = (losses, flat.clone())
        dist.barrier()
    lp, ln = out["peer"][0], out["nccl"][0]
    for a, b in zip(lp, ln):
        assert abs(a - b) <= 1e-4 * max(1.0, abs(b)), "loss trajectories differ: %r vs %r" % (lp, ln)
    torch.testing.assert_close(out["peer"][1], out["nccl"][1], rtol=1e-3, atol=2e-5)
    return lp, float((out["peer"][1] - out["nccl"][1]).abs().max())


def main():
    world = int(os.environ["WORLD_SIZE"])
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)
    res = {"world": world}
    res["flat_max_abs_diff_vs_nccl_adam"] = flat_check(dev, world, rank)
    losses, d = trainer_check(dev, world, rank, graph=False)
    res["trainer_eager"] = {"losses": losses, "param_max_abs_diff_vs_nccl": d}
    losses, d = trainer_check(dev, world, rank, graph=True)
    res["trainer_graph"] = {"losses": losses, "param_max_abs_diff_vs_nccl": d}
    if rank == 0:
        print(json.dumps(res))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
