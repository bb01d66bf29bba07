"""Attribution speed on the GPU: captured saliency per batch against the eager route (model forward + autograd.grad w.r.t. x on
the same kernels, launched from the host) and against the captured training step; integrated gradients (32 points) in
patients per second per config.  Median of several timed windows (CUDA events), card name and power limit recorded.

    python tools/attribution_bench.py --out r04_attribution.json
"""
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

import torch  # noqa: E402

import multilevel_gnn_b200 as mlg  # noqa: E402

DEV = "cuda:0"


def _split(n, seed):
    raw = mlg.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * mlg.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = mlg.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(n)]
    return pts, topo


def _model(cfg, seed=1):
    args = mlg.configs.make_args(cfg)
    torch.manual_seed(seed)
    model = mlg.MultilevelGNN(args)
    mlg.synth.multilevel_params(model, seed=seed)
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    return model, args


def _time(fn, iters, windows):
    """Median over windows of the mean time per call (ms), device events around ``iters`` calls."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return statistics.median(out), out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--iters", type=int, default=200)
    a = ap.parse_args()
    res = {"card": card(), "torch": torch.__version__}
    # --- gbm B = 32: captured saliency, eager route, training step
    B = 32
    model, args = _model("gbm")
    pts, topo = _split(64, seed=2)
    batch = mlg.data.to_device(mlg.data.collate(pts[:B], topo, pin=False), topo, DEV)
    at = mlg.Attributor(model, args, batch_size=B, method="saliency").capture(batch)
    med, win = _time(at.graph.replay, a.iters, a.windows)
    res["gbm_b32_saliency_captured_ms"] = {"median": med, "windows": win}
    med, win = _time(at.eager, a.iters // 4, a.windows)
    res["gbm_b32_saliency_eager_ms"] = {"median": med, "windows": win}
    # per-kernel spans of one eager pass (CUDA events around each native call; the pass is host bound, the spans are not)
    from multilevel_gnn_b200 import _cabi
    timer = _cabi.KernelTimer()
    _cabi.TIMER = timer
    try:
        at.eager()
        torch.cuda.synchronize()
        res["gbm_b32_saliency_eager_spans"] = timer.summary()
    finally:
        _cabi.TIMER = None
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(DEV)
    tr = mlg.train.Trainer(model, args, weight)
    tr.capture(batch)
    med, win = _time(tr.step, a.iters, a.windows)
    res["gbm_b32_train_step_ms"] = {"median": med, "windows": win}
    # whole attribute() call over 256 patients (host collate + staging + replays + accumulation + one sync)
    ds = pts * 4
    at = mlg.Attributor(model, args, batch_size=B, method="saliency").capture(batch)
    at.attribute(ds, topo)
    t = []
    for _ in range(a.windows):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        at.attribute(ds, topo)
        t.append(time.perf_counter() - t0)
    res["gbm_b32_saliency_attribute_256_patients_s"] = {"median": statistics.median(t), "windows": t}
    del tr, at
    # --- integrated gradients, 32 points: patients per second (replay + accumulation per replay)
    for cfg in ("gbm", "kirc", "lgg"):
        model, args = _model(cfg)
        Bc = args.batch_size
        pts, topo = _split(Bc, seed=3)
        batch = mlg.data.to_device(mlg.data.collate(pts, topo, pin=False), topo, DEV)
        at = mlg.Attributor(model, args, batch_size=Bc, method="integrated_gradients", points=32).capture(batch)
        med, win = _time(at.graph.replay, a.iters // 2, a.windows)
        per_replay = Bc // 32
        res["%s_ig32_b%d" % (cfg, Bc)] = {"replay_ms": med, "windows": win, "patients_per_replay": per_replay,
                                          "patients_per_s": per_replay / (med * 1e-3)}
        ds = pts * 2
        at.attribute(ds, topo)
        t = []
        for _ in range(a.windows):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            at.attribute(ds, topo)
            t.append(time.perf_counter() - t0)
        res["%s_ig32_b%d" % (cfg, Bc)]["attribute_%d_patients_s" % len(ds)] = statistics.median(t)
        del at
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
