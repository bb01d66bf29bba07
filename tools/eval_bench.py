#!/usr/bin/env python
"""Evaluation speed on one GPU: the reference's per-epoch eval() (train.py:71-109) three ways, and a synthetic epoch.

    python tools/eval_bench.py [--out-dir profiles] [--windows 7] [--steps 50]

(1) graphs/s of a forward-only pass at gbm B = 32 over a device-resident batch: (a) today's eager route, model.eval() +
    torch.no_grad() + model(batch); (b) eager MultilevelGNN.predict; (c) the captured train.Evaluator graph (replays only);
    plus (a) and (c) over a whole 400-sample split from host records -- collate, upload, forward, metrics (eager: pred to the
    host and NumPy metrics; Evaluator: evaluate());
(2) the captured Evaluator for kirc and lgg at B = 64 (replays, and a 400-sample split);
(3) the wall time of a synthetic gbm epoch: 400 training samples through the captured Trainer (prefetched batches, every loss
    read back), then eval of splits of 400 / 50 / 50 samples -- Trainer + eager eval against Trainer + Evaluator.
Every number is the median of --windows repeated windows, with min and max.  The device name and power limit are read in
the same run.  Writes r03_eval_<part>.json under --out-dir and prints one JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def device_info(idx=0):
    info = {"torch_name": torch.cuda.get_device_name(idx)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = [s.strip() for s in q.split(",")]
        info.update(name=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:          # the query is informative only
        info["nvidia_smi_error"] = repr(e)
    return info


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs), "all": xs}


def make_split(m, n, seed, topo_seed=0):
    """n patient records on ONE gene network (a fold of the reference's dataset) + its FoldTopology."""
    raw = m.synth.multilevel_batch(batch_size=1, seed=topo_seed)
    n1 = 3 * m.MultilevelGNN.GENES
    topo = m.data.FoldTopology(raw.edge_index, raw.edge_attr, raw.gene_pca_match[0], raw.raw_indice[0], n1)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, n1, generator=g)
    age = torch.rand(n, generator=g)
    lab = (torch.rand(n, generator=g) < 0.5).long()
    y = torch.nn.functional.one_hot(lab, 2).float()
    return [types.SimpleNamespace(x=x[i], age=age[i], y=y[i]) for i in range(n)], topo


def np_metrics(pred, y, w=None):
    """What a user computes on the host after an eager pass: BCELoss(weight), argmax accuracy, ROC AUC (Mann-Whitney)."""
    p, t = pred.astype(np.float64), y.astype(np.float64)
    w = np.ones(2) if w is None else np.asarray(w, dtype=np.float64)
    with np.errstate(divide="ignore"):
        bce = float((w * ((t - 1) * np.maximum(np.log1p(-p), -100) - t * np.maximum(np.log(p), -100))).mean())
    lab = t.argmax(1)
    acc = float((p.argmax(1) == lab).mean())
    pos, neg = p[lab == 1, 1], np.sort(p[lab == 0, 1])
    if len(pos) == 0 or len(neg) == 0:
        return bce, acc, float("nan")
    lo = np.searchsorted(neg, pos, "left")
    hi = np.searchsorted(neg, pos, "right")
    return bce, acc, float((2 * lo.sum() + (hi - lo).sum()) / (2.0 * len(pos) * len(neg)))


def eager_split(m, model, pts, topo, B, dev, w=None):
    """Today's evaluation of a split: unshuffled batches, eval() + no_grad forward, predictions to the host, host metrics."""
    was = model.training
    model.eval()
    preds = []
    with torch.no_grad():
        for hb in m.data.TopologyLoader(pts, topo, B, shuffle=False, drop_last=False):
            pred, _ = model(m.data.to_device(hb, topo, dev))
            preds.append(pred.cpu())
    model.train(was)
    pred = torch.cat(preds).numpy()
    y = torch.stack([p.y for p in pts]).numpy()
    return np_metrics(pred, y, w)


def timed(fn, windows, reps):
    """Host wall time of ``reps`` calls of fn() ending in a device synchronise, per window (ms)."""
    out = []
    for _ in range(windows):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def model_for(m, cfg, dev):
    args = m.configs.make_args(cfg)
    torch.manual_seed(0)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model)
    model.to(dev)
    model.pathway_indexs = model.pathway_indexs.to(dev)
    return model, args


def forward_rates(m, cfg, B, dev, a, ways):
    model, args = model_for(m, cfg, dev)
    pts, topo = make_split(m, a.split, seed=1)
    batch = m.data.to_device(m.data.collate(pts[:B], topo, pin=False), topo, dev)
    ev = m.train.Evaluator(model, args, batch_size=B).capture(batch)
    res = {"config": cfg, "batch": B}

    def eager():
        model.eval()
        with torch.no_grad():
            model(batch)

    calls = {"a_eager_eval_no_grad": eager, "b_eager_predict": lambda: model.predict(batch), "c_evaluator_replay": ev.graph.replay}
    for k in ways:
        fn = calls[k]
        for _ in range(3):
            fn()
        ms = timed(fn, a.windows, a.steps)
        res[k] = {"graphs_per_s": spread([B * a.steps / (t / 1e3) for t in ms]),
                  "ms_per_batch": spread([t / a.steps for t in ms])}
    # whole split from host records
    ev.evaluate(pts, topo)
    ms = timed(lambda: ev.evaluate(pts, topo, with_pred=False), a.windows, 1)
    res["c_evaluator_split"] = {"n": len(pts), "ms": spread(ms), "graphs_per_s": spread([len(pts) / (t / 1e3) for t in ms])}
    if "a_eager_eval_no_grad" in ways:
        eager_split(m, model, pts, topo, B, dev)
        ms = timed(lambda: eager_split(m, model, pts, topo, B, dev), a.windows, 1)
        res["a_eager_split"] = {"n": len(pts), "ms": spread(ms), "graphs_per_s": spread([len(pts) / (t / 1e3) for t in ms])}
        r = ev.evaluate(pts, topo)
        e = eager_split(m, model, pts, topo, B, dev)
        res["metrics_evaluator_vs_eager"] = {"evaluator": [r.bce, r.acc, r.auc], "eager_host": list(e)}
    return res


def epoch_wall(m, dev, a):
    """Synthetic gbm epoch: train on 400 samples (captured Trainer, prefetched host batches, losses read back), then eval of the
    train / valid / test splits (400 / 50 / 50), eager or through the Evaluator."""
    B = 32
    model, args = model_for(m, "gbm", dev)
    train_pts, topo = make_split(m, 400, seed=11)
    valid_pts, _ = make_split(m, 50, seed=12)
    test_pts, _ = make_split(m, 50, seed=13)
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(dev)
    tr = m.train.Trainer(model, args, weight)
    first = m.data.to_device(m.data.collate(train_pts[:B], topo, pin=False), topo, dev)
    tr.capture(first)
    ev = m.train.Evaluator(model, args, batch_size=B, criterion_weight=weight).capture(first)
    loader = m.data.TopologyLoader(train_pts, topo, B)

    def train_epoch(epoch):
        loader.set_epoch(epoch)
        pend = []
        for hb in loader:
            tr.prefetch(hb)
            pend.append(tr.loss_to_host(tr.step_prefetched()))
        return [h.get() for h in pend]

    def eval_eager():
        return [eager_split(m, model, s, topo, B, dev, [0.8, 1.3] if args.weight_balance else None)
                for s in (train_pts, valid_pts, test_pts)]

    def eval_graph():
        return [ev.evaluate(s, topo, with_pred=False) for s in (train_pts, valid_pts, test_pts)]

    out = {"train_samples": 400, "eval_samples": [400, 50, 50], "batch": B}
    train_epoch(0)
    eval_eager()
    eval_graph()
    for name, fn in (("trainer_plus_eager_eval", eval_eager), ("trainer_plus_evaluator", eval_graph)):
        tot, tr_ms, ev_ms = [], [], []
        for e in range(a.windows):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            train_epoch(e + 1)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            tot.append((t2 - t0) * 1e3)
            tr_ms.append((t1 - t0) * 1e3)
            ev_ms.append((t2 - t1) * 1e3)
        out[name] = {"epoch_ms": spread(tot), "train_ms": spread(tr_ms), "eval_ms": spread(ev_ms)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--split", type=int, default=400)
    ap.add_argument("--parts", default="gbm,kirc_lgg,epoch")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench.py needs a CUDA device")
    import multilevel_gnn_b200 as m
    m._cabi.lib()
    dev = torch.device("cuda", 0)
    os.makedirs(a.out_dir, exist_ok=True)
    dev_info = device_info(0)
    results = {}
    parts = a.parts.split(",")
    if "gbm" in parts:
        results["gbm"] = forward_rates(m, "gbm", 32, dev, a, ["a_eager_eval_no_grad", "b_eager_predict", "c_evaluator_replay"])
        r = results["gbm"]
        r["speedup_c_over_a"] = (r["c_evaluator_replay"]["graphs_per_s"]["median"]
                                 / r["a_eager_eval_no_grad"]["graphs_per_s"]["median"])
        r["speedup_c_split_over_a_split"] = r["a_eager_split"]["ms"]["median"] / r["c_evaluator_split"]["ms"]["median"]
    if "kirc_lgg" in parts:
        results["kirc_lgg"] = [forward_rates(m, cfg, 64, dev, a, ["c_evaluator_replay"]) for cfg in ("kirc", "lgg")]
    if "epoch" in parts:
        results["epoch"] = epoch_wall(m, dev, a)
    for k, v in results.items():
        with open(os.path.join(a.out_dir, "r03_eval_%s.json" % k), "w") as f:
            json.dump({"device": dev_info, "windows": a.windows, "steps": a.steps, "result": v}, f, indent=1)
    summary = {"device": dev_info}
    if "gbm" in results:
        g = results["gbm"]
        summary["gbm_b32_graphs_per_s"] = {k: g[k]["graphs_per_s"]["median"] for k in
                                           ("a_eager_eval_no_grad", "b_eager_predict", "c_evaluator_replay")}
        summary["speedup_c_over_a"] = g["speedup_c_over_a"]
        summary["split400_ms"] = {"eager": g["a_eager_split"]["ms"]["median"], "evaluator": g["c_evaluator_split"]["ms"]["median"]}
    if "kirc_lgg" in results:
        summary["b64_replay_graphs_per_s"] = {r["config"]: r["c_evaluator_replay"]["graphs_per_s"]["median"]
                                              for r in results["kirc_lgg"]}
    if "epoch" in results:
        summary["epoch_ms"] = {k: results["epoch"][k]["epoch_ms"]["median"]
                               for k in ("trainer_plus_eager_eval", "trainer_plus_evaluator")}
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
