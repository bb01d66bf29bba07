"""Host side of the split evaluation (train.Evaluator), no GPU: the NumPy metric reference the kernel is checked against, and
the sharded evaluation plan -- every sample evaluated exactly once, and the gathered per-rank rows reassembled in dataset
order, also through a real gloo all_gather."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import eval_ref


def test_auc_reference_matches_mannwhitneyu():
    from scipy.stats import mannwhitneyu
    rng = np.random.default_rng(0)
    for n, levels in ((50, None), (400, None), (400, 5), (1000, 2), (7, 3)):
        labels = rng.integers(0, 2, n)
        labels[:2] = (0, 1)
        s = rng.random(n)
        if levels:                                     # heavy ties
            s = np.floor(s * levels) / levels
        pos, neg = s[labels == 1], s[labels == 0]
        u = mannwhitneyu(pos, neg, alternative="two-sided").statistic
        assert eval_ref.auc(labels, s) == pytest.approx(u / (len(pos) * len(neg)), rel=1e-12, abs=0)
    assert np.isnan(eval_ref.auc(np.ones(5, int), rng.random(5)))
    assert eval_ref.auc([0, 1], [0.3, 0.3]) == 0.5


def test_metric_reference_bce_matches_torch():
    g = torch.Generator().manual_seed(1)
    pred = torch.softmax(torch.randn(33, 2, generator=g), 1)
    pred[0] = torch.tensor([1.0, 0.0])                 # log(0): clamped at -100
    y = torch.nn.functional.one_hot(torch.randint(0, 2, (33,), generator=g), 2).float()
    w = torch.tensor([0.8, 1.3])
    bce, acc, _ = eval_ref.metrics(pred.numpy(), y.numpy(), w.numpy())
    want = torch.nn.BCELoss(weight=w.expand(33, 2))(pred.double(), y.double())
    assert bce == pytest.approx(float(want), rel=1e-12)
    assert acc == float((pred.argmax(1) == y.argmax(1)).double().mean())


def _plans(n, B, world):
    from multilevel_gnn_b200.data import TopologyLoader
    return [TopologyLoader(list(range(n)), None, B, shuffle=False, drop_last=False, rank=r, world=world).index_batches()
            for r in range(world)]


def _gathered(plans, B):
    """[world, steps, B] of dataset indices as the Evaluator's per-rank buffers hold them (padding slots: -1)."""
    steps = len(plans[0])
    out = torch.full((len(plans), steps, B), -1, dtype=torch.int64)
    for r, plan in enumerate(plans):
        for s, idx in enumerate(plan):
            out[r, s, :idx.numel()] = idx
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_sharded_plan_covers_each_sample_once(world):
    from multilevel_gnn_b200.train import reassemble
    for n in (1, 5, 31, 32, 33, 45, 100, 257, 400):
        for B in (1, 4, 32):
            plans = _plans(n, B, world)
            assert len({len(p) for p in plans}) == 1, "every rank must step the same number of times"
            seen = torch.cat([i for p in plans for i in p])
            assert sorted(seen.tolist()) == list(range(n))
            assert all(i.numel() <= B for p in plans for i in p)
            got = reassemble(_gathered(plans, B), n)
            assert torch.equal(got, torch.arange(n)), (n, B, world)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n, B, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from multilevel_gnn_b200.data import TopologyLoader
    from multilevel_gnn_b200.train import reassemble
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    plan = TopologyLoader(list(range(n)), None, B, shuffle=False, drop_last=False, rank=rank, world=world).index_batches()
    # per step [pred | y] rows of the B slots, as the Evaluator copies them out of its static buffers; the "prediction" of
    # sample i is (i, -i), its label (i % 2, 1 - i % 2); padding slots hold garbage
    out = torch.full((len(plan), 2, B, 2), 1e9)
    for s, idx in enumerate(plan):
        f = idx.double()
        out[s, 0, :idx.numel()] = torch.stack([f, -f], 1)
        out[s, 1, :idx.numel()] = torch.stack([f % 2, 1 - f % 2], 1)
    got = [torch.empty_like(out) for _ in range(world)]
    dist.all_gather(got, out)
    rows = reassemble(torch.stack(got).permute(0, 1, 3, 2, 4), n)
    q.put((rank, rows.tolist()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,n,B", [(2, 45, 8), (3, 100, 16)])
def test_gloo_all_gather_reassembles_dataset_order(world, n, B):
    port = _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, B, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    f = torch.arange(n, dtype=torch.float32)
    want = torch.stack([torch.stack([f, -f], 1), torch.stack([f % 2, 1 - f % 2], 1)], 1)
    for _, rows in res:
        assert torch.equal(torch.tensor(rows), want)
