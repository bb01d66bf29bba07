"""Knockout screens (multilevel_gnn_b200.Knockout) against ``model.predict`` on explicitly knocked-out copies of the patients,
in batches of 64.

Tolerance: atol 1e-5 on the delta and on the knocked-out probability.  The screen recomputes the reached rows of the two
SAGE layers in plain fp32 row arithmetic, while ``predict`` computes them with the 3xTF32 tensor-core GEMM and the fused
kernels' own summation orders; the two agree to a few fp32 ulps per layer, i.e. ~1e-7 on the probabilities.

* gbm at full size, every one of the 5 135 gene groups for two patients;
* kirc and lgg (reorder_pathway, pca_dim 3, max-pool 1x1 / 4x2): the highest-degree genes and random genes, node groups,
  pathway gene sets (large T2) and a cohort-mean baseline;
* a synthetic hub gene read by thousands of rows (the largest tables and workspaces);
* exactness: a group already at the baseline and an empty group give delta == 0.0 exactly; a (patient, group) result has
  the same bits in another dataset, position or company; a replay equals an eager pass;
* after a Trainer step the screen reflects the new parameters, and the Trainer's state is untouched by a screen;
* routes the incremental trunk does not cover raise NotImplementedError;
* structure: a screen runs no weight-gradient kernel and writes no .grad; a training step launches the same kernels before
  and after a screen."""
import types

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ATOL = 1e-5


@pytest.fixture(scope="module")
def mlg():
    import multilevel_gnn_b200 as m
    m._cabi.lib()
    return m


def _model(mlg, cfg, seed):
    args = mlg.configs.make_args(cfg)
    torch.manual_seed(seed)
    model = mlg.MultilevelGNN(args)
    mlg.synth.multilevel_params(model, seed=seed)
    if args.reorder_pathway:
        model.set_reorder_idxs(torch.randperm(146, generator=torch.Generator().manual_seed(seed)).tolist())
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    return model, args


def _split(mlg, n, seed, hub=None):
    """n patients on the synthetic topology; ``hub`` = (gene, fan-out): that gene's mRNA node is also read by the mRNA rows of
    ``fan-out`` other genes."""
    raw = mlg.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * mlg.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    ei, ea = raw.edge_index[:, :e1], raw.edge_attr[:e1]
    if hub is not None:
        h, fan = hub
        dst = torch.randperm(mlg.MultilevelGNN.GENES, generator=torch.Generator().manual_seed(seed))[:fan]
        dst = dst[dst != h]
        ei = torch.cat([ei, torch.stack([torch.full_like(dst, 3 * h), 3 * dst])], 1)
        ea = torch.cat([ea, torch.full((dst.numel(), 1), 0.5)])
    topo = mlg.data.FoldTopology(ei, ea, raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1].clone(), age=raw.age[i], y=raw.y[2 * i:2 * i + 2])
           for i in range(n)]
    return pts, topo


def _batch(mlg, pts, topo):
    return mlg.data.to_device(mlg.data.collate(pts, topo, pin=False), topo, DEV)


def _knockout(mlg, model, args, pts, topo, B, **kw):
    ko = mlg.Knockout(model, args, batch_size=B, **kw)
    batch = _batch(mlg, (pts * B)[:B], topo)
    return ko.capture(batch)


def _groups_list(groups, n_nodes):
    from multilevel_gnn_b200 import knockout as K
    ptr, nodes = K.parse_groups(groups, n_nodes)
    return [nodes[ptr[k]:ptr[k + 1]] for k in range(ptr.numel() - 1)]


def _reference(mlg, model, pts, topo, groups, baseline=None, target=1):
    """(delta [n, K], knocked-out probability [n, K], base pred [n, 2]) from model.predict on knocked-out copies, 64 per call."""
    n1 = topo.n_nodes
    glist = _groups_list(groups, n1)
    base_x = torch.zeros(n1) if baseline is None else torch.as_tensor(baseline, dtype=torch.float32)
    dev_topo = topo.on_device(64, DEV)

    def predict(xs, ages):
        out = []
        for s in range(0, xs.shape[0], 64):
            x, a = xs[s:s + 64], ages[s:s + 64]
            m = x.shape[0]
            if m < 64:
                x = torch.cat([x, x[-1:].expand(64 - m, -1)])
                a = torch.cat([a, a[-1:].expand(64 - m)])
            b = mlg.synth.GraphBatch(x=x.reshape(-1, 1).to(DEV), age=a.to(DEV), **dev_topo)
            b.topology_key = "%s-b64" % topo.key
            out.append(model.predict(b)[0][:m].cpu())
        return torch.cat(out)

    deltas, kos, bases = [], [], []
    for p in pts:
        x = p.x.reshape(-1).float()
        copies = x.repeat(len(glist) + 1, 1)
        for k, g in enumerate(glist):
            copies[k + 1, g] = base_x[g]
        pr = predict(copies, torch.full((copies.shape[0],), float(p.age)))
        bases.append(pr[0])
        kos.append(pr[1:, target])
        deltas.append(pr[1:, target] - pr[0, target])
    return torch.stack(deltas), torch.stack(kos), torch.stack(bases)


def _check(res, ref, what, target=1):
    d, ko, base = ref
    assert res.delta.shape == d.shape, what
    err_d = (res.delta - d).abs().max().item()
    err_p = (res.pred[:, target:target + 1] + res.delta - ko).abs().max().item()
    err_b = (res.pred - base).abs().max().item()
    assert err_d <= ATOL and err_p <= ATOL and err_b <= ATOL, "%s: delta %.2e, knocked-out prob %.2e, base %.2e" % (
        what, err_d, err_p, err_b)


def test_gbm_full_size_every_gene(mlg):
    model, args = _model(mlg, "gbm", seed=51)
    pts, topo = _split(mlg, 2, seed=51)
    ko = _knockout(mlg, model, args, pts, topo, 32)
    res = ko.screen(pts, topo)
    assert res.delta.shape == (2, mlg.MultilevelGNN.GENES)
    _check(res, _reference(mlg, model, pts, topo, "gene"), "gbm genes")
    assert (res.delta != 0).float().mean() > 0.5          # knockouts do move the prediction


def _top_genes(topo, count):
    """Genes whose mRNA node is read by the most rows (highest out-degree in the edge list)."""
    deg = torch.bincount(topo.edge_index[0] // 3, minlength=topo.n_nodes // 3)
    return torch.argsort(deg, descending=True)[:count].tolist()


@pytest.mark.parametrize("cfg", ["kirc", "lgg"])
def test_kirc_lgg_genes_nodes_pathways_cohort_mean(mlg, cfg):
    model, args = _model(mlg, cfg, seed=52)
    pts, topo = _split(mlg, 3, seed=52)
    n1 = topo.n_nodes
    g = torch.Generator().manual_seed(5)
    genes = sorted(set(_top_genes(topo, 40) + torch.randint(0, n1 // 3, (160,), generator=g).tolist()))
    gene_groups = [[3 * q, 3 * q + 1, 3 * q + 2] for q in genes]
    node_groups = [[int(i)] for i in torch.randint(0, n1, (150,), generator=g)]
    match, seg = topo.gene_pca_match, topo.raw_indice
    pathways = []
    for s in torch.randint(0, 438, (12,), generator=g).tolist():
        nd = match[(seg == s) & (match >= 0)]
        pathways.append(sorted(set(nd.tolist())))
    mean = torch.stack([p.x.reshape(-1) for p in pts]).mean(0)
    for groups, baseline, what in ((gene_groups, None, "genes"), (node_groups, None, "nodes"), (pathways, None, "pathways"),
                                   (gene_groups, mean, "genes, cohort mean")):
        ko = _knockout(mlg, model, args, pts, topo, 8, groups=groups, baseline=baseline)
        res = ko.screen(pts, topo)
        _check(res, _reference(mlg, model, pts, topo, groups, baseline), "%s %s" % (cfg, what))
        if what == "pathways":
            assert ko._tables["max_t2"] > 1000


def test_hub_gene(mlg):
    hub = 11
    model, args = _model(mlg, "gbm", seed=53)
    pts, topo = _split(mlg, 2, seed=53, hub=(hub, 3000))
    groups = [[3 * q, 3 * q + 1, 3 * q + 2] for q in (hub, 0, 1, 2, 4000)] + [list(range(3 * hub, 3 * hub + 3)) + [5, 6]]
    ko = _knockout(mlg, model, args, pts, topo, 4, groups=groups)
    assert ko._tables["max_t1"] > 2900 and ko._tables["max_t2"] > 4000      # CNV / methylation rows read only themselves
    res = ko.screen(pts, topo)
    _check(res, _reference(mlg, model, pts, topo, groups), "hub")


def test_exactness_and_determinism(mlg):
    model, args = _model(mlg, "lgg", seed=54)
    pts, topo = _split(mlg, 5, seed=54)
    for q in (3, 4):                                     # genes 3 and 4 of patient 1 already at the (zero) baseline
        pts[1].x[3 * q:3 * q + 3] = 0.0
    groups = [[9, 10, 11], [], [30, 31, 32], [0], list(range(3000, 3300)), [12, 13, 14]]
    ko = _knockout(mlg, model, args, pts, topo, 4, groups=groups)
    full = ko.screen(pts, topo)
    assert full.delta[1, 0].item() == 0.0 and full.delta[1, 5].item() == 0.0 and torch.all(full.delta[:, 1] == 0.0)
    assert (full.delta[:, 2] != 0).all()
    rev = ko.screen(pts[::-1], topo)
    assert torch.equal(rev.delta.flip(0), full.delta) and torch.equal(rev.pred.flip(0), full.pred)
    for i in (0, 4):
        alone = ko.screen([pts[i]], topo)
        assert torch.equal(alone.delta[0], full.delta[i]) and torch.equal(alone.pred[0], full.pred[i])
    ko2 = _knockout(mlg, model, args, pts, topo, 4, groups=groups[::-1] + groups[:2])
    other = ko2.screen(pts[2:] + pts[:2], topo)
    assert torch.equal(other.delta[:, :len(groups)].flip(1), torch.cat([full.delta[2:], full.delta[:2]]))
    assert torch.equal(other.delta[:, len(groups):], torch.cat([full.delta[2:], full.delta[:2]])[:, :2])
    # a replay equals an eager pass of the same plan
    ko._plan.copy_(torch.tensor([[0, 0, 1, 1] + [0] * (ko.ROWS - 4), [-1, 2, -1, 4] + [-1] * (ko.ROWS - 4),
                                 [0, 0, 2, 2] + list(range(4, ko.ROWS))], device=DEV))
    ko.graph.replay()
    ko.graph_chunk.replay()
    d_graph, p_graph = ko.out_delta.clone(), ko.out_pred.clone()
    ko.eager()
    assert torch.equal(ko.out_delta, d_graph) and torch.equal(ko.out_pred, p_graph)
    assert d_graph[0].item() == 0.0 and d_graph[1].item() != 0.0


def test_trainer_step_then_screen(mlg):
    """Trainer step -> screen -> Trainer step: the screen (captured before the Trainer re-homed the parameters) re-captures
    and matches predict with the updated parameters; the flat parameters and Adam moments equal those of two plain steps."""
    B = 8
    pts, topo = _split(mlg, 16, seed=55)
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(DEV)
    groups = [[3 * q, 3 * q + 1, 3 * q + 2] for q in range(0, 5135, 97)]
    states = []
    for with_ko in (False, True):
        model, args = _model(mlg, "gbm", seed=55)
        ko = _knockout(mlg, model, args, pts, topo, B, groups=groups) if with_ko else None
        tr = mlg.train.Trainer(model, args, weight)
        tr.capture(_batch(mlg, pts[:B], topo))
        torch.manual_seed(1)
        tr.step(_batch(mlg, pts[:B], topo))
        if with_ko:
            old = ko.graph
            res = ko.screen(pts[:3], topo)
            assert ko.graph is not old
            _check(res, _reference(mlg, model, pts[:3], topo, groups), "after a Trainer step")
        tr.step(_batch(mlg, pts[B:], topo))
        torch.cuda.synchronize()
        states.append([t.clone() for t in (tr.opt.flat_p, tr.opt.exp_avg, tr.opt.exp_avg_sq)])
    for a, c in zip(*states):
        assert torch.equal(a, c)


def test_unsupported_routes_raise(mlg):
    from multilevel_gnn_b200 import functional as Fn
    model, args = _model(mlg, "gbm", seed=56)
    pts, topo = _split(mlg, 2, seed=56)
    for flag in ("TRANSFORM_FIRST", "FACTORED_RANK1", "H1_NODE_MAJOR"):
        old = getattr(Fn, flag)
        setattr(Fn, flag, False)
        try:
            with pytest.raises(NotImplementedError):
                _knockout(mlg, model, args, pts, topo, 4)
        finally:
            setattr(Fn, flag, old)
    args2 = mlg.configs.make_args("gbm", gnn_name="rsage")
    with pytest.raises(NotImplementedError):
        mlg.Knockout(mlg.MultilevelGNN(args2), args2)


class _Recorder:
    """Stands in for the loaded library: records the name and arguments of every C call."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            self.calls.append((name, a))
            return fn(*a)
        return call


def _step_calls(mlg, model, args, batch, monkeypatch):
    from multilevel_gnn_b200 import _cabi
    tr = mlg.train.Trainer(model, args, torch.tensor([[0.8, 1.3]]).repeat(4, 1).to(DEV))
    tr.step(batch)                                         # eager: builds the topology caches
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    torch.manual_seed(2)
    tr.step(batch)
    torch.cuda.synchronize()
    monkeypatch.setattr(_cabi, "_lib", rec._lib)
    return [c[0] for c in rec.calls]


def test_zz_knockout_structure(mlg, monkeypatch):
    from multilevel_gnn_b200 import _cabi
    model, args = _model(mlg, "kirc", seed=57)
    pts, topo = _split(mlg, 4, seed=57)
    batch = _batch(mlg, pts, topo)
    before = _step_calls(mlg, model, args, batch, monkeypatch)
    for p in model.parameters():
        p.grad = None
    ko = _knockout(mlg, model, args, pts, topo, 4, groups=[[0, 1, 2], [60, 61, 62]])
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        ko.eager()
        torch.cuda.synchronize()
    monkeypatch.setattr(_cabi, "_lib", rec._lib)
    names = [c[0] for c in rec.calls]
    banned = ("mlg_xty", "mlg_sage_fold_stacked_bwd", "mlg_sage_fold_bwd", "mlg_wcolsum", "mlg_pool_bwd",
              "mlg_sage_rank1_bwd", "mlg_head_conv_pool_bwd", "mlg_head_mlp_bwd", "mlg_adam", "mlg_peer")
    assert not [n for n in names if n.startswith(banned) and not n.endswith("_supported")], names
    assert "mlg_knockout_trunk" in names and "mlg_sage_rank1_fwd_rows_nm" in names
    ops = {e.key for e in prof.key_averages()}
    assert not {o for o in ops if "backward" in o}, ops
    assert all(p.grad is None for p in model.parameters())
    ko.screen(pts, topo)
    after = _step_calls(mlg, model, args, batch, monkeypatch)
    assert after == before
