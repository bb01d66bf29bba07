"""Knockout-screen timing on the B200: ``Knockout.screen`` against brute force, per config.

Brute force is ``model.predict`` captured over a static batch of 64 knocked-out copies built on the device (each replay
gathers the patients' rows and writes the group's nodes to the baseline inside the graph), one replay per 64 knockouts.
Both routes screen the same synthetic cohort with the same groups, alternating, ``--windows`` times; the medians go to
``<out>/r05_knockout_<cfg>.json`` with the card's name and power limit.  ``--profile`` adds a torch.profiler run of one
gene screen that splits the device time between the incremental trunk, the base forward and the head.

    python tools/knockout_bench.py --configs gbm,kirc,lgg --patients 64 --windows 5 --out profiles
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # the measurement stands without it; say why it is missing
        q = "unavailable (%s)" % e
    return q


def setup(m, cfg, n, seed=0):
    args = m.configs.make_args(cfg)
    torch.manual_seed(seed)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model, seed=seed)
    model.to("cuda")
    model.pathway_indexs = model.pathway_indexs.to("cuda")
    raw = m.synth.multilevel_batch(batch_size=n, seed=seed + 1)
    n1 = 3 * m.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = m.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(n)]
    return model, args, topo, pts


class BruteForce:
    """predict on 64 device-built knocked-out copies per replay (captured), groups as a padded node matrix."""
    ROWS = 64

    def __init__(self, m, model, topo, pts, groups):
        from multilevel_gnn_b200 import knockout as K
        n1 = topo.n_nodes
        ptr, nodes = K.parse_groups(groups, n1)
        lens = ptr[1:] - ptr[:-1]
        width = int(lens.max())
        pad = torch.empty(len(lens), width, dtype=torch.int64)
        for k in range(len(lens)):                   # pad with the group's first node: the same value written again
            g = nodes[ptr[k]:ptr[k + 1]]
            pad[k] = torch.cat([g, g[:1].expand(width - g.numel())])
        self.K = len(lens)
        self.model = model
        self.nodes = pad.cuda()
        self.xs = torch.stack([p.x.reshape(-1) for p in pts]).float().cuda()
        self.ages = torch.stack([torch.as_tensor(p.age, dtype=torch.float32) for p in pts]).cuda()
        dev = topo.on_device(self.ROWS, "cuda")
        self.static = m.synth.GraphBatch(x=torch.zeros(self.ROWS * n1, 1, device="cuda"), age=torch.zeros(self.ROWS, device="cuda"),
                                         **dev)
        self.static.topology_key = "%s-b%d" % (topo.key, self.ROWS)
        self.plan = torch.zeros(2, self.ROWS, dtype=torch.int64, device="cuda")
        for _ in range(2):
            self._body()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._body()

    def _body(self):
        R = self.ROWS
        x = self.xs.index_select(0, self.plan[0])
        idx = self.nodes.index_select(0, self.plan[1])
        x.scatter_(1, idx, torch.zeros_like(idx, dtype=x.dtype))
        self.static.x.view(R, -1).copy_(x)
        self.static.age.copy_(self.ages.index_select(0, self.plan[0]))
        self.out = self.model.predict(self.static)[0][:, 1]

    def screen(self):
        n = self.xs.shape[0]
        total = n * self.K
        items = torch.arange(total, device="cuda")
        plan = torch.stack([items // self.K, items % self.K])
        out = torch.empty(-(-total // self.ROWS) * self.ROWS, device="cuda")
        for s in range(0, total, self.ROWS):
            m = min(self.ROWS, total - s)
            self.plan[:, :m].copy_(plan[:, s:s + m])
            self.graph.replay()
            out[s:s + self.ROWS].copy_(self.out)
        return out[:total].view(n, self.K).cpu()


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, r


def pathway_sets(topo):
    """One group per pathway: the nodes its 3 segments' slots read."""
    match, seg = topo.gene_pca_match, topo.raw_indice
    return [sorted(set(match[((seg // 3) == p) & (match >= 0)].tolist())) for p in range(146)]


def run_config(m, cfg, n, windows, rows_list, out_dir):
    model, args, topo, pts = setup(m, cfg, n)
    res = {"config": cfg, "patients": n, "card": card(), "windows": windows}
    for gname, groups in (("gene", "gene"), ("pathway", pathway_sets(topo))):
        kos = {}
        for rows in rows_list if gname == "gene" else rows_list[:1]:
            ko = m.Knockout(model, args, groups=groups, batch_size=32)
            ko.ROWS = rows
            ko.capture(m.data.to_device(m.data.collate(pts[:32], topo), topo, "cuda"))
            kos[rows] = ko
        bf = BruteForce(m, model, topo, pts, groups)
        K = bf.K
        ts = {r: [] for r in kos}
        tb = []
        outs = {}
        for w in range(windows + 1):                   # window 0 warms every shape up and is not counted
            for r, ko in kos.items():
                dt, outs[r] = timed(lambda: ko.screen(pts, topo))
                if w:
                    ts[r].append(dt)
            dt, ob = timed(bf.screen)
            if w:
                tb.append(dt)
        med = lambda v: sorted(v)[len(v) // 2]
        entry = {"groups": K, "knockouts": n * K, "brute_force_ms_per_patient": 1e3 * med(tb) / n,
                 "brute_force_knockouts_per_s": n * K / med(tb)}
        base = outs[rows_list[0]]
        ko_prob = base.pred[:, 1:2] + base.delta
        entry["max_abs_diff_vs_brute_force"] = float((ko_prob - ob).abs().max())
        for r in kos:
            entry["rows_%d" % r] = {"ms_per_patient": 1e3 * med(ts[r]) / n, "knockouts_per_s": n * K / med(ts[r]),
                                    "speedup_vs_brute_force": med(tb) / med(ts[r]),
                                    "windows_s": ts[r],
                                    "max_abs_delta_diff_vs_rows_%d" % rows_list[0]: float((outs[r].delta - base.delta).abs().max())}
        entry["brute_force_windows_s"] = tb
        res[gname] = entry
        print(cfg, gname, json.dumps({k: v for k, v in entry.items() if not k.endswith("windows_s")}), flush=True)
    with open(os.path.join(out_dir, "r05_knockout_%s.json" % cfg), "w") as f:
        json.dump(res, f, indent=1)


def profile(m, out_dir, n=8):
    model, args, topo, pts = setup(m, "gbm", n)
    ko = m.Knockout(model, args, groups="gene", batch_size=8)
    ko.capture(m.data.to_device(m.data.collate(pts[:8], topo), topo, "cuda"))
    ko.screen(pts, topo)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ko.screen(pts, topo)
        torch.cuda.synchronize()
    cats = {}
    kern = {}
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if us <= 0:
            continue
        name = e.key
        if name.startswith(("ko_layer1", "ko_layer2")) or "ko_layer" in name:
            c = "incremental layers (ko_layer1 / ko_layer2)"
        elif "ko_pool" in name or "ko_copy" in name:
            c = "incremental pool + pooled copies (ko_pool)"
        elif "head" in name or "maxpool" in name:
            c = "head"
        elif "index" in name.lower() or "copy" in name.lower() or "Memcpy" in name:
            c = "plan / result copies"
        else:
            c = "base forward and other"
        cats[c] = cats.get(c, 0.0) + us / 1e3
        kern[name] = us / 1e3
    res = {"card": card(), "config": "gbm", "patients": n, "groups": "gene", "device_ms_by_category": cats,
           "device_ms_by_kernel": dict(sorted(kern.items(), key=lambda kv: -kv[1])[:25])}
    print(json.dumps(res, indent=1))
    with open(os.path.join(out_dir, "r05_knockout_profile.json"), "w") as f:
        json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="gbm,kirc,lgg")
    ap.add_argument("--patients", type=int, default=64)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--rows", default="128,64", help="head rows per replay to compare (the first is the shipped Knockout.ROWS)")
    ap.add_argument("--out", default="profiles", help="directory for the JSON results")
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("knockout_bench: needs a CUDA device")
    import multilevel_gnn_b200 as m
    os.makedirs(a.out, exist_ok=True)
    print("card:", card(), flush=True)
    for cfg in a.configs.split(","):
        run_config(m, cfg, a.patients, a.windows, [int(r) for r in a.rows.split(",")], a.out)
    if a.profile:
        profile(m, a.out)


if __name__ == "__main__":
    main()
