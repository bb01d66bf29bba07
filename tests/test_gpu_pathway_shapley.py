"""Pathway Shapley values (multilevel_gnn_b200.PathwayShapley) against references built from ``model.post_pool`` on explicitly
built head-input grids (the patient's and the background rows' ``pca_feature`` from ``model.predict``, mixed per cell).

Tolerance: atol 1e-5 on values, base and delta.  The chains update the first Linear's pre-activation incrementally in fp32
(one window difference at a time) where the reference evaluates every grid from scratch; the two agree to ~1e-7 on the
probabilities.

* exact mode against the enumeration of all 2^K coalitions x M background rows with float64 Shapley weights ("omic" and a
  6-group segment partition, gbm / kirc with reorder / lgg);
* sampled mode against the same estimator by brute force: every chain's K + 1 prefix grids rebuilt from shapley_draws
  (S = 2 and 8, "pathway" and "segment", the three configs);
* efficiency at S = 32 (|delta| <= 1e-5) with pred equal to model.predict bitwise;
* exactness: a patient equal to every background row gets values == 0.0; gbm pathways 144 / 145 (grid rows the floor-mode
  pool never reads) get 0.0 in every mode; a patient's values have the same bits with another batch_size and company at
  the same dataset index; a replay equals an eager pass; a background row index outside [0, M) is flagged, not read;
* after a Trainer step the values reflect the new parameters and the Trainer's state is untouched by an explain call;
* structure (last): explain runs no weight-gradient kernel and writes no .grad; a training step launches the same kernels
  before and after."""
import math
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
    g = torch.Generator().manual_seed(seed + 100)
    with torch.no_grad():                   # biases away from 0 so that the probabilities are not all near 0.5
        model.head[0].bias.copy_(torch.randn(model.head[0].bias.shape, generator=g) * 0.05)
        model.head[3].bias.copy_(torch.randn(2, generator=g) * 0.3)
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    return model, args


def _split(mlg, n, seed):
    raw = mlg.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * mlg.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = mlg.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1].clone(), age=raw.age[i], y=raw.y[2 * i:2 * i + 2])
           for i in range(n)]
    return pts, topo


def _batch(mlg, pts, topo):
    return mlg.data.to_device(mlg.data.collate(pts, topo, pin=False), topo, DEV)


def _shapley(mlg, model, args, pts, topo, B, background, **kw):
    sh = mlg.PathwayShapley(model, args, background=background, batch_size=B, **kw)
    return sh.capture(_batch(mlg, (pts * B)[:B], topo))


class _Ref:
    """Head-input grids of patients and background rows (model.predict, 8 per call) and F on mixed grids (post_pool)."""

    def __init__(self, mlg, model, args, topo, players):
        from multilevel_gnn_b200 import shapley as S
        self.mlg, self.model, self.args, self.topo = mlg, model, args, topo
        self.groups = S.parse_players(players)
        kh, kw, _, _, _ = S.head_geometry(model)
        reorder = model.reorder_idxs if args.reorder_pathway else None
        owner = S.player_tables(self.groups, model.pca_dim, kh, kw, reorder)[0]
        self.Wg = 3 * model.pca_dim
        self.owner = owner.view(146, self.Wg).long().to(DEV)
        self.row = S.segment_row(reorder).to(DEV) if reorder is not None else None

    def grids(self, xs):
        out = []
        for s in range(0, len(xs), 8):
            chunk = [types.SimpleNamespace(x=x, age=0.0, y=torch.zeros(2)) for x in xs[s:s + 8]]
            m = len(chunk)
            chunk = chunk + [chunk[-1]] * (8 - m)
            with torch.no_grad():
                out.append(self.model.predict(_batch(self.mlg, chunk, self.topo))[1][:m].clone())
        return torch.cat(out)

    def F(self, grids, age, target):
        """pred[:, target] (float64, host) of head-input grids [R, 32, 146, Wg] at one age, 64 rows per post_pool call."""
        was = self.model.training
        self.model.eval()
        out = []
        try:
            for s in range(0, grids.shape[0], 64):
                g = grids[s:s + 64]
                if self.row is not None:
                    g = g[:, :, self.row]
                g = g.reshape(g.shape[0], 32, 438, self.model.pca_dim)
                with torch.no_grad():
                    pred, _ = self.model.post_pool(g, torch.full((g.shape[0],), float(age), device=DEV), require_grad=False)
                out.append(pred[:, target].double().cpu())
        finally:
            self.model.train(was)
        return torch.cat(out)

    def mixed(self, xg, bg, from_pat):
        """from_pat [R, 146, Wg] bool: the patient's cell, else the background grid's."""
        return torch.where(from_pat.unsqueeze(1), xg.unsqueeze(0), bg)

    def exact(self, xg, bgs, age, target):
        """(phi [K] float64, base, F(x)) by enumeration of the 2^K coalitions x M rows."""
        K, M = len(self.groups), bgs.shape[0]
        own = self.owner
        v = torch.empty(2 ** K, dtype=torch.float64)
        for c in range(2 ** K):
            bits = torch.tensor([(c >> k) & 1 for k in range(K)], dtype=torch.bool, device=DEV)
            fp = (own < 0) | bits[own.clamp(min=0)]
            v[c] = self.F(self.mixed(xg, bgs, fp.expand(M, -1, -1)), age, target).mean()
        phi = torch.zeros(K, dtype=torch.float64)
        for c in range(2 ** K):
            size = bin(c).count("1")
            for k in range(K):
                if not (c >> k) & 1:
                    w = math.factorial(size) * math.factorial(K - size - 1) / math.factorial(K)
                    phi[k] += w * (v[c | (1 << k)] - v[c])
        return phi, float(v[0]), float(v[-1])

    def sampled(self, xg, bgs, age, target, perm, j):
        """(phi [K], base) of the sampled estimator: every chain's K + 1 prefix grids."""
        K = len(self.groups)
        phi = torch.zeros(K, dtype=torch.float64)
        base = 0.0
        own = self.owner
        for g in range(perm.shape[0]):
            rank = torch.empty(K, dtype=torch.int64, device=DEV)
            rank[perm[g].to(DEV)] = torch.arange(K, device=DEV)
            orank = torch.where(own >= 0, rank[own.clamp(min=0)], torch.full_like(own, -1))
            f = torch.cat([self.F(self.mixed(xg, bgs[int(j[g])].unsqueeze(0),
                                             orank.unsqueeze(0) < torch.arange(t0, min(K + 1, t0 + 64), device=DEV).view(-1, 1, 1)),
                                  age, target) for t0 in range(0, K + 1, 64)])
            r = rank.cpu()
            phi += (f[r + 1] - f[r]) / perm.shape[0]
            base += float(f[0]) / perm.shape[0]
        return phi, base


def _xs(pts):
    return [p.x.reshape(-1) for p in pts]


def _partition6():
    g = torch.Generator().manual_seed(6)
    segs = torch.randperm(438, generator=g)[:300]
    return [segs[k::6].tolist() for k in range(6)]


@pytest.mark.parametrize("cfg", ["gbm", "kirc", "lgg"])
def test_exact_mode_vs_enumeration(mlg, cfg):
    model, args = _model(mlg, cfg, seed=61)
    pts, topo = _split(mlg, 6, seed=61)
    data, bgp = pts[:2], pts[2:]
    for players in ("omic", _partition6()):
        for target in (1, 0):
            sh = _shapley(mlg, model, args, data, topo, 4, torch.stack(_xs(bgp)), players=players, samples="exact",
                          target=target)
            res = sh.explain(data, topo)
            ref = _Ref(mlg, model, args, topo, players)
            xg, bgs = ref.grids(_xs(data)), ref.grids(_xs(bgp))
            for i, p in enumerate(data):
                phi, base, fx = ref.exact(xg[i], bgs, float(p.age), target)
                what = "%s %s target %d patient %d" % (cfg, "omic" if players == "omic" else "6 groups", target, i)
                assert (res.values[i].double() - phi).abs().max() <= ATOL, (what, res.values[i], phi)
                assert abs(float(res.base[i]) - base) <= ATOL, what
                assert abs(float(res.delta[i])) <= ATOL and abs(float(res.pred[i, target]) - fx) <= ATOL, what
            assert (res.values.abs() > 1e-6).float().mean() > 0.5


@pytest.mark.parametrize("cfg", ["gbm", "kirc", "lgg"])
def test_sampled_mode_vs_brute_force(mlg, cfg):
    from multilevel_gnn_b200 import shapley as S
    model, args = _model(mlg, cfg, seed=62)
    pts, topo = _split(mlg, 6, seed=62)
    data, bgp = pts[:2], pts[2:]
    bank = torch.stack(_xs(bgp))
    for players in ("pathway", "segment"):
        ref = _Ref(mlg, model, args, topo, players)
        xg, bgs = ref.grids(_xs(data)), ref.grids(_xs(bgp))
        for samples in (2, 8):
            sh = _shapley(mlg, model, args, data, topo, 4, bank, players=players, samples=samples, seed=5)
            res = sh.explain(data, topo)
            for i, p in enumerate(data):
                perm, j = S.shapley_draws(5, i, samples, bank.shape[0], len(ref.groups))
                phi, base = ref.sampled(xg[i], bgs, float(p.age), 1, perm, j)
                what = "%s %s S=%d patient %d" % (cfg, players, samples, i)
                err = (res.values[i].double() - phi).abs().max().item()
                assert err <= ATOL and abs(float(res.base[i]) - base) <= ATOL, (what, err)
                assert abs(float(res.delta[i])) <= ATOL, what


def test_efficiency_and_pred(mlg):
    model, args = _model(mlg, "lgg", seed=63)
    pts, topo = _split(mlg, 12, seed=63)
    data, bgp = pts[:8], pts[8:]
    sh = _shapley(mlg, model, args, data, topo, 8, torch.stack(_xs(bgp)), samples=32)
    res = sh.explain(data, topo)
    assert res.values.shape == (8, 146) and res.values.dtype == torch.float32
    assert float(res.delta.abs().max()) <= ATOL, res.delta
    with torch.no_grad():
        want = model.predict(_batch(mlg, data, topo))[0].cpu()
    assert torch.equal(res.pred, want)
    assert float((res.pred[:, 1].double() - res.base).abs().max()) > 1e-4       # the patients differ from the cohort


def test_exactness_and_determinism(mlg):
    model, args = _model(mlg, "gbm", seed=64)
    pts, topo = _split(mlg, 9, seed=64)
    data, bgp = pts[:6], pts[6:]
    bank = torch.stack(_xs(bgp))
    # a patient equal to every background row: every value is exactly 0
    same = _shapley(mlg, model, args, data, topo, 4, torch.stack([data[1].x.reshape(-1)] * 3), samples=4)
    r0 = same.explain(data, topo)
    assert torch.all(r0.values[1] == 0.0) and (r0.values[0] != 0).any()
    # gbm pathways 144 and 145 sit on grid rows the floor-mode (4, 2) pool never reads
    dead = [[3 * 144, 3 * 144 + 1, 3 * 144 + 2], [3 * 145, 3 * 145 + 1, 3 * 145 + 2], [0, 1, 2], [30, 31], [200]]
    for kw in (dict(samples=8), dict(players="segment", samples=2), dict(players=dead, samples="exact"),
               dict(players=dead, samples=4)):
        r = _shapley(mlg, model, args, data, topo, 4, bank, **kw).explain(data, topo)
        cols = [0, 1] if kw.get("players") is dead else ([144, 145] if "players" not in kw else list(range(3 * 144, 438)))
        assert torch.all(r.values[:, cols] == 0.0), kw
        assert (r.values != 0).float().mean() > 0.3, kw
    # the same dataset index gives the same bits with another batch_size and other company
    full = _shapley(mlg, model, args, data, topo, 4, bank, samples=8).explain(data, topo)
    other = [data[0], pts[7], data[2], pts[6], data[4], data[5], pts[8]]
    alt = _shapley(mlg, model, args, data, topo, 8, bank, samples=8).explain(other, topo)
    for i in (0, 2, 4, 5):
        assert torch.equal(alt.values[i], full.values[i]) and torch.equal(alt.base[i], full.base[i])
        assert torch.equal(alt.pred[i], full.pred[i])
    assert not torch.equal(alt.values[1], full.values[1])
    again = _shapley(mlg, model, args, data, topo, 4, bank, samples=8).explain(data, topo)
    assert torch.equal(again.values, full.values) and torch.equal(again.delta, full.delta)
    # a replay equals an eager pass
    sh = _shapley(mlg, model, args, data, topo, 4, bank, samples=8)
    sh.graph.replay()
    p_graph, c_graph = sh.out_pred.clone(), sh.out_cells.clone()
    sh.eager()
    assert torch.equal(sh.out_pred, p_graph) and torch.equal(sh.out_cells, c_graph)


def test_bad_background_index_is_flagged(mlg):
    """mlg_shap_chains never reads a chain's background row outside [0, M): its outputs are NaN, the flag is raised, and the
    other chains of the CTA are unchanged."""
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()
    g = torch.Generator().manual_seed(7)
    Hg, Wg, kh, kw, H, K, M, n = 8, 6, 2, 2, 64, 5, 3, 4
    cells = Hg * Wg
    nwin = (Hg // kh) * (Wg // kw)
    pat = torch.rand(n, 64 * cells, generator=g).to(DEV)
    bgt = torch.rand(M, 64 * cells, generator=g).to(DEV)
    w1p = (torch.randn(nwin, 64, H, generator=g) * 0.05).to(DEV)
    b1, w3, b3 = (torch.randn(H, generator=g) * 0.1).to(DEV), (torch.randn(2, H, generator=g) * 0.1).to(DEV), torch.zeros(2, device=DEV)
    owner = (torch.arange(cells) % K).to(torch.int32).to(DEV)
    wins = [sorted({(c // Wg // kh) * (Wg // kw) + (c % Wg) // kw for c in range(cells) if c % K == k}) for k in range(K)]
    win_ptr = torch.tensor([0] + [len(w) for w in wins], dtype=torch.int32).cumsum(0).to(torch.int32).to(DEV)
    win_idx = torch.tensor(sum(wins, []), dtype=torch.int32).to(DEV)
    perm = torch.stack([torch.randperm(K, generator=g) for _ in range(2)]).to(torch.int32).to(DEV)
    chain_pat = torch.arange(n, dtype=torch.int32, device=DEV)
    bad = torch.zeros(1, dtype=torch.int32, device=DEV)

    def run(chain_bg):
        out = [torch.empty(n * 2, K, device=DEV), torch.empty(n * 2, device=DEV), torch.empty(n * 2, device=DEV)]
        _cabi.check(L.mlg_shap_chains(_cabi.fptr(pat), n, _cabi.fptr(bgt), M, 64 * cells, Hg, Wg, kh, kw, _cabi.fptr(w1p),
                                      _cabi.fptr(b1), None, None, _cabi.fptr(w3), _cabi.fptr(b3), 1, H, _cabi.iptr(owner),
                                      _cabi.iptr(win_ptr), _cabi.iptr(win_idx), K, _cabi.iptr(perm), 2, _cabi.iptr(chain_pat),
                                      _cabi.iptr(chain_bg), n, _cabi.fptr(out[0]), _cabi.fptr(out[1]), _cabi.fptr(out[2]),
                                      _cabi.iptr(bad), _cabi.stream_ptr()), "mlg_shap_chains")
        return [t.cpu() for t in out]

    ok = torch.tensor([[0, 1, 2, 0], [2, 2, 1, 0]], dtype=torch.int32, device=DEV)
    good = run(ok)
    assert int(bad.item()) == 0 and all(bool(torch.isfinite(t).all()) for t in good)
    # per chain, the contributions add up to pT - p0
    assert float((good[0].double().sum(1) - (good[2] - good[1]).double()).abs().max()) < 1e-6
    badj = ok.clone()
    badj[0, 1] = M
    badj[1, 3] = -1
    got = run(badj)
    assert int(bad.item()) == 1
    rows_bad = [1 * 2 + 0, 3 * 2 + 1]                       # row = s * G + g
    keep = [r for r in range(n * 2) if r not in rows_bad]
    for t_good, t_got in zip(good, got):
        assert bool(t_got[rows_bad].isnan().all()) and torch.equal(t_got[keep], t_good[keep])
    assert L.mlg_shap_chains(None, n, None, M, 0, Hg, Wg, kh, kw, None, None, None, None, None, None, 1, H, None, None, None,
                             K, None, 2, None, None, n, None, None, None, None, None) < 0


def test_trainer_step_then_explain(mlg):
    """Trainer step -> explain -> Trainer step: the explain call (captured before the Trainer re-homed the parameters)
    re-captures and matches the enumeration with the updated parameters; the flat parameters and Adam moments equal those
    of two plain steps."""
    B = 8
    pts, topo = _split(mlg, 16, seed=65)
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(DEV)
    bank = torch.stack(_xs(pts[13:16]))
    states = []
    for with_shap in (False, True):
        model, args = _model(mlg, "gbm", seed=65)
        sh = _shapley(mlg, model, args, pts[:2], topo, 4, bank, players="omic", samples="exact") if with_shap else None
        tr = mlg.train.Trainer(model, args, weight)
        tr.capture(_batch(mlg, pts[:B], topo))
        torch.manual_seed(1)
        tr.step(_batch(mlg, pts[:B], topo))
        if with_shap:
            old = sh.graph
            res = sh.explain(pts[:2], topo)
            assert sh.graph is not old
            ref = _Ref(mlg, model, args, topo, "omic")
            xg, bgs = ref.grids(_xs(pts[:2])), ref.grids(_xs(pts[13:16]))
            for i in range(2):
                phi, base, _ = ref.exact(xg[i], bgs, float(pts[i].age), 1)
                assert (res.values[i].double() - phi).abs().max() <= ATOL and abs(float(res.base[i]) - base) <= ATOL
        tr.step(_batch(mlg, pts[B:2 * B], topo))
        torch.cuda.synchronize()
        states.append([t.clone() for t in (tr.opt.flat_p, tr.opt.exp_avg, tr.opt.exp_avg_sq)])
    for a, c in zip(*states):
        assert torch.equal(a, c)


class _Recorder:
    """Stands in for the loaded library: records the name of every C call."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            self.calls.append(name)
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
    return rec.calls


def test_zz_shapley_structure(mlg, monkeypatch):
    from multilevel_gnn_b200 import _cabi
    model, args = _model(mlg, "kirc", seed=66)
    pts, topo = _split(mlg, 6, seed=66)
    batch = _batch(mlg, pts[:4], topo)
    before = _step_calls(mlg, model, args, batch, monkeypatch)
    for p in model.parameters():
        p.grad = None
    sh = _shapley(mlg, model, args, pts[:4], topo, 4, torch.stack(_xs(pts[4:])), samples=2)
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        sh.eager()
        sh.explain(pts[:4], topo)
        torch.cuda.synchronize()
    monkeypatch.setattr(_cabi, "_lib", rec._lib)
    banned = ("mlg_xty", "mlg_sage_fold_stacked_bwd", "mlg_sage_fold_bwd", "mlg_wcolsum", "mlg_pool_bwd",
              "mlg_sage_rank1_bwd", "mlg_head_conv_pool_bwd", "mlg_head_mlp_bwd", "mlg_adam", "mlg_peer")
    assert not [n for n in rec.calls if n.startswith(banned) and not n.endswith("_supported")], rec.calls
    assert "mlg_shap_chains" in rec.calls and "mlg_head_conv_pool_fwd" in rec.calls and "mlg_attr_accumulate" in rec.calls
    ops = {e.key for e in prof.key_averages()}
    assert not {o for o in ops if "backward" in o}, ops
    assert all(p.grad is None for p in model.parameters())
    after = _step_calls(mlg, model, args, batch, monkeypatch)
    assert after == before
