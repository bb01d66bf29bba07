#!/usr/bin/env python
"""Multi-process check of the sharded split evaluation (train.Evaluator) on real GPUs.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        tools/eval_check.py [--out FILE.json]

Every rank builds the same model and the same splits (n = 45, 100 and 7 at B = 16: padded tails, and with 8 ranks ranks whose
last batch is empty), evaluates each split once on its shard and once alone on the full split (world_size=1, no collective),
and checks that the sharded EvalResult -- auc, acc, bce and the pred array -- equals the single-GPU one exactly, on every rank.
Prints one JSON line on rank 0; exits non-zero on any mismatch."""
import argparse
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def split(m, n, seed):
    raw = m.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * m.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = m.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    return [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(n)], topo


def same(a, b):
    return a == b or (a != a and b != b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch", type=int, default=16)
    a = ap.parse_args()
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200.train import Evaluator
    world = int(os.environ["WORLD_SIZE"])
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)
    args = m.configs.make_args("gbm")
    torch.manual_seed(0)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model)
    model.to(dev)
    model.pathway_indexs = model.pathway_indexs.to(dev)
    B = a.batch
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1)
    out, ok = {"world": world, "batch": B, "splits": []}, True
    for n, seed in ((45, 3), (100, 4), (7, 5)):
        pts, topo = split(m, n, seed)
        ex = m.data.to_device(m.data.collate((pts * B)[:B], topo, pin=False), topo, dev)
        sharded = Evaluator(model, args, batch_size=B, criterion_weight=weight, world_size=world).capture(ex)
        alone = Evaluator(model, args, batch_size=B, criterion_weight=weight, world_size=1).capture(ex)
        r_dp = sharded.evaluate(pts, topo)
        r_1 = alone.evaluate(pts, topo)
        good = (all(same(getattr(r_dp, k), getattr(r_1, k)) for k in ("auc", "acc", "bce", "n"))
                and torch.equal(r_dp.pred, r_1.pred))
        flags = torch.tensor([1 if good else 0], device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        # and the same on every rank: rank 0's numbers against everyone's
        mine = torch.tensor([r_dp.auc, r_dp.acc, r_dp.bce], dtype=torch.float64, device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        across = all(torch.equal(t.nan_to_num(-1.0), allr[0].nan_to_num(-1.0)) for t in allr)
        ok = ok and bool(flags.item()) and across
        out["splits"].append({"n": n, "auc": r_dp.auc, "acc": r_dp.acc, "bce": r_dp.bce,
                              "equal_to_single_gpu": bool(flags.item()), "equal_across_ranks": across})
    out["ok"] = ok
    if rank == 0:
        line = json.dumps(out)
        print(line)
        if a.out:
            os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
            with open(a.out, "w") as f:
                f.write(line + "\n")
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
