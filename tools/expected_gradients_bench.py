"""Expected-gradients speed on the GPU: patients per second of whole ``Attributor.attribute`` calls with
method="expected_gradients" at S = 32 samples (without and with ``completeness``), against integrated gradients at 32 points,
the three alternated window by window in one run; the replay of each captured graph alone; and the two expected-gradients
kernels (mlg_attr_eg_interp, mlg_attr_eg_accumulate) alone.  gbm, kirc and lgg at their configured batch sizes.  Median of
``--windows`` windows (CUDA events for device-only timings, a host clock around calls that end in a synchronisation);
card name and power limit recorded in each file.

    python tools/expected_gradients_bench.py --out-dir profiles --prefix r06_expected_gradients
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
from multilevel_gnn_b200 import _cabi  # noqa: E402

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


def _events(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def _wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def bench_config(cfg, a):
    model, args = _model(cfg)
    B = args.batch_size
    pts, topo = _split(a.patients + a.background, seed=3)
    data = pts[:a.patients]
    bank = torch.stack([p.x.reshape(-1) for p in pts[a.patients:]])
    batch = mlg.data.to_device(mlg.data.collate((data * B)[:B], topo, pin=False), topo, DEV)
    arms = {
        "ig32": mlg.Attributor(model, args, batch_size=B, method="integrated_gradients", points=32),
        "eg32": mlg.Attributor(model, args, batch_size=B, method="expected_gradients", background=bank, samples=32),
        "eg32_completeness": mlg.Attributor(model, args, batch_size=B, method="expected_gradients", background=bank,
                                            samples=32, completeness=True),
    }
    for at in arms.values():
        at.capture(batch)
        at.attribute(data, topo)                         # warm-up of every shape the windows use
    res = {"card": card(), "torch": torch.__version__, "config": cfg, "batch_size": B, "patients": a.patients,
           "background_rows": bank.shape[0], "windows": a.windows}
    # whole attribute() calls, the arms alternated within every window
    wall = {k: [] for k in arms}
    for _ in range(a.windows):
        for k, at in arms.items():
            wall[k].append(_wall(lambda: at.attribute(data, topo)))
    # the captured graph alone (forward + input-only backward of B slots), alternated the same way
    for at in arms.values():
        for _ in range(3):
            at.graph.replay()
    replay = {k: [] for k in arms}
    for _ in range(a.windows):
        for k, at in arms.items():
            replay[k].append(_events(at.graph.replay, a.iters))
    for k in arms:
        med = statistics.median(wall[k])
        res[k] = {"attribute_s": {"median": med, "windows": wall[k]}, "patients_per_s": a.patients / med,
                  "replay_ms": {"median": statistics.median(replay[k]), "windows": replay[k]}}
    res["eg32_over_ig32_time"] = res["eg32"]["attribute_s"]["median"] / res["ig32"]["attribute_s"]["median"]
    # the two kernels alone at this batch: interpolation of B slots, accumulation of one replay's patients
    at = arms["eg32"]
    N = at.out_g.shape[1]
    M = at._bank.shape[0]
    per = max(1, B // 32)
    w = torch.full((B,), 1.0 / 32, device=DEV)
    ptr = torch.arange(0, per * 32 + 1, 32, dtype=torch.int32, device=DEV)
    acc = torch.zeros(per, N, device=DEV)
    xs = at.static_batch.x.view(B, N)
    xin = torch.empty(B, N, device=DEV)
    L = _cabi.lib()

    def interp():
        L.mlg_attr_eg_interp(_cabi.fptr(xs), _cabi.fptr(at._bank), M, _cabi.iptr(at.j), _cabi.fptr(at.alpha), B, N,
                             _cabi.fptr(xin), _cabi.iptr(at._bad), _cabi.stream_ptr())

    def accumulate():
        L.mlg_attr_eg_accumulate(_cabi.fptr(at.out_g), _cabi.fptr(xs), _cabi.fptr(at._bank), M, _cabi.iptr(at.j),
                                 _cabi.fptr(w), _cabi.iptr(ptr), per, N, 1, _cabi.fptr(acc), _cabi.iptr(at._bad),
                                 _cabi.stream_ptr())

    for name, fn, nbytes in (("eg_interp", interp, 3 * B * N * 4), ("eg_accumulate", accumulate, (3 * B + 2 * per) * N * 4)):
        fn()
        t = [_events(fn, 500) for _ in range(a.windows)]
        med = statistics.median(t)
        res["kernel_" + name] = {"us": med * 1e3, "windows_ms": t, "algorithmic_bytes": nbytes,
                                 "GB_per_s": nbytes / (med * 1e-3) / 1e9}
    assert int(at._bad.item()) == 0
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--prefix", default="r06_expected_gradients")
    ap.add_argument("--configs", default="gbm,kirc,lgg")
    ap.add_argument("--patients", type=int, default=32)
    ap.add_argument("--background", type=int, default=32)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("expected_gradients_bench.py measures on the GPU; no CUDA device found")
    os.makedirs(a.out_dir, exist_ok=True)
    for cfg in a.configs.split(","):
        res = bench_config(cfg, a)
        with open(os.path.join(a.out_dir, "%s_%s.json" % (a.prefix, cfg)), "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({k: v for k, v in res.items() if k in ("config", "card", "eg32_over_ig32_time")} |
                         {k: res[k]["patients_per_s"] for k in ("ig32", "eg32", "eg32_completeness")}))
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
