"""Pathway Shapley speed on the GPU: patients per second of whole ``PathwayShapley.explain`` calls (64 synthetic patients, a
background of 64, players="pathway", S = 32), the chain kernel (mlg_shap_chains) per launch, and the same estimator by brute
force on a few patients: the same draws, every chain's 147 prefix grids built on the device and evaluated by a captured
``post_pool`` replay (the fused head) of 64 rows.  Also players="omic", samples="exact".  gbm, kirc and lgg at their
configured batch sizes.  Median of ``--windows`` windows (a host clock around calls that end in a synchronisation, CUDA events
for the kernel); card name and power limit recorded in each file.

    python tools/pathway_shapley_bench.py --out-dir profiles --prefix r07_pathway_shapley
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
from multilevel_gnn_b200 import shapley as S  # noqa: E402

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
    if args.reorder_pathway:
        model.set_reorder_idxs(torch.randperm(146, generator=torch.Generator().manual_seed(seed)).tolist())
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    return model, args


def _wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def _chain_ms(sh, data, topo):
    """Device time of the chain kernel inside one explain call (CUDA events around the launch)."""
    _cabi.TIMER = _cabi.KernelTimer()
    try:
        sh.explain(data, topo)
        return _cabi.TIMER.summary()["shap_chains"]["ms"]
    finally:
        _cabi.TIMER = None


def _grids(model, pts, topo, B):
    out = []
    for s in range(0, len(pts), B):
        chunk = [types.SimpleNamespace(x=p.x, age=0.0, y=torch.zeros(2)) for p in pts[s:s + B]]
        m = len(chunk)
        chunk = chunk + [chunk[-1]] * (B - m)
        with torch.no_grad():
            out.append(model.predict(mlg.data.to_device(mlg.data.collate(chunk, topo, pin=False), topo, DEV))[1][:m].clone())
    return torch.cat(out)


class BruteForce:
    """The sampled estimator evaluated grid by grid: captured post_pool replays of ROWS head-input grids."""
    ROWS = 64

    def __init__(self, model, args, groups):
        self.model, self.args = model, args
        kh, kw, _, _, _ = S.head_geometry(model)
        reorder = model.reorder_idxs if args.reorder_pathway else None
        self.Wg = 3 * model.pca_dim
        self.owner = S.player_tables(groups, model.pca_dim, kh, kw, reorder)[0].view(146, self.Wg).long().to(DEV)
        self.row = S.segment_row(reorder).to(DEV) if reorder is not None else None
        self.K = len(groups)
        self.static = torch.zeros(self.ROWS, 32, 146, self.Wg, device=DEV)
        self.age = torch.zeros(self.ROWS, device=DEV)
        model.eval()
        with torch.no_grad():
            for _ in range(2):
                self._body()
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._body()

    def _body(self):
        g = self.static if self.row is None else self.static[:, :, self.row]
        pred, _ = self.model.post_pool(g.reshape(self.ROWS, 32, 438, self.model.pca_dim), self.age, require_grad=False)
        self.out = pred[:, 1]

    def patient(self, xg, bgs, age, perm, j):
        """phi [K] (float64, device) of one patient from its S chains' (K + 1)-prefix grids."""
        K, Sn, R = self.K, perm.shape[0], self.ROWS
        rank = torch.empty(Sn, K, dtype=torch.int64, device=DEV)
        rank.scatter_(1, perm.to(DEV), torch.arange(K, device=DEV).expand(Sn, K).contiguous())
        own = self.owner
        orank = torch.where(own >= 0, rank[:, own.clamp(min=0)], torch.full_like(own, -1))           # [S, 146, Wg]
        total = Sn * (K + 1)
        chain = torch.arange(total, device=DEV) // (K + 1)
        t = torch.arange(total, device=DEV) % (K + 1)
        jd = j.to(DEV)
        f = torch.empty(total, dtype=torch.float32, device=DEV)
        self.age.fill_(age)
        for s in range(0, total, R):
            c, tt = chain[s:s + R], t[s:s + R]
            m = c.numel()
            mask = orank[c] < tt.view(-1, 1, 1)
            self.static[:m].copy_(torch.where(mask.unsqueeze(1), xg.unsqueeze(0), bgs[jd[c]]))
            self.graph.replay()
            f[s:s + m].copy_(self.out[:m])
        f = f.double().view(Sn, K + 1)
        return ((f.gather(1, rank + 1) - f.gather(1, rank)).mean(0)), f[:, 0].mean()


def bench_config(cfg, a):
    model, args = _model(cfg)
    B = args.batch_size
    pts, topo = _split(a.patients + a.background, seed=3)
    data = pts[:a.patients]
    bank = torch.stack([p.x.reshape(-1) for p in pts[a.patients:]])
    batch = mlg.data.to_device(mlg.data.collate((data * B)[:B], topo, pin=False), topo, DEV)
    arms = {
        "pathway_s32": mlg.PathwayShapley(model, args, background=bank, players="pathway", samples=32, batch_size=B),
        "omic_exact": mlg.PathwayShapley(model, args, background=bank, players="omic", samples="exact", batch_size=B),
    }
    res = {"card": card(), "torch": torch.__version__, "config": cfg, "batch_size": B, "patients": a.patients,
           "background_rows": bank.shape[0], "windows": a.windows}
    out = {}
    for k, sh in arms.items():
        sh.capture(batch)
        out[k] = sh.explain(data, topo)                     # warm-up of every shape the windows use
    wall = {k: [] for k in arms}
    chain = {k: [] for k in arms}
    for _ in range(a.windows):
        for k, sh in arms.items():
            wall[k].append(_wall(lambda: sh.explain(data, topo))[0])
    for _ in range(a.windows):
        for k, sh in arms.items():
            chain[k].append(_chain_ms(sh, data, topo))
    for k, sh in arms.items():
        med = statistics.median(wall[k])
        res[k] = {"explain_s": {"median": med, "windows": wall[k]}, "patients_per_s": a.patients / med,
                  "chain_kernel_ms": {"median": statistics.median(chain[k]), "windows": chain[k]},
                  "max_abs_delta": float(out[k].delta.abs().max())}
    res["w1_packed_MB"] = 4 * model.head[0].weight[:, :64 * arms["pathway_s32"].Ho * arms["pathway_s32"].Wo].numel() / 1e6
    # brute force of the same estimator on a few patients
    sh = arms["pathway_s32"]
    bf = BruteForce(model, args, sh.groups)
    few = data[:a.brute_patients]
    xg, bgs = _grids(model, few, topo, B), _grids(model, pts[a.patients:], topo, B)
    times, errs = [], []
    for i, p in enumerate(few):
        perm, j = S.shapley_draws(sh.seed, i, sh.samples, bank.shape[0], sh.K)
        bf.patient(xg[i], bgs, float(p.age), perm, j)               # warm-up
        dt, (phi, base) = _wall(lambda: bf.patient(xg[i], bgs, float(p.age), perm, j))
        times.append(dt)
        errs.append(max(float((phi.cpu() - out["pathway_s32"].values[i].double()).abs().max()),
                        abs(float(base) - float(out["pathway_s32"].base[i]))))
    per_patient = statistics.median(times)
    res["brute_force"] = {"patients": len(few), "s_per_patient": {"median": per_patient, "patients": times},
                          "grids_per_patient": sh.samples * (sh.K + 1), "rows_per_replay": bf.ROWS,
                          "max_abs_diff_vs_explain": max(errs)}
    res["speedup_explain_vs_brute_force"] = per_patient / (res["pathway_s32"]["explain_s"]["median"] / a.patients)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--prefix", default="r07_pathway_shapley")
    ap.add_argument("--configs", default="gbm,kirc,lgg")
    ap.add_argument("--patients", type=int, default=64)
    ap.add_argument("--background", type=int, default=64)
    ap.add_argument("--brute-patients", type=int, default=3)
    ap.add_argument("--windows", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pathway_shapley_bench.py measures on the GPU; no CUDA device found")
    os.makedirs(a.out_dir, exist_ok=True)
    for cfg in a.configs.split(","):
        res = bench_config(cfg, a)
        with open(os.path.join(a.out_dir, "%s_%s.json" % (a.prefix, cfg)), "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({k: res[k] for k in ("config", "card", "speedup_explain_vs_brute_force")} |
                         {k: (res[k]["patients_per_s"], res[k]["chain_kernel_ms"]["median"]) for k in ("pathway_s32", "omic_exact")}))
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
