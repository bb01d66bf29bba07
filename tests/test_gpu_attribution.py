"""Gradients with respect to the node values (batch.x) on the fused kernels, and the captured Attributor.

* dL/dx, dL/dage and dL/dpca_feature of the default route against autograd through the CPU oracle at full size
  (N = 15 405 nodes, G = 25 015 gene slots), at the tolerances of test_gpu_fullsize.py;
* every route of the layers (generic / gather first layer, buffered second layer, unfused activation backward, additive
  value mask, no value mask, an explicit ``x=`` argument) gives the same gradient;
* asking for dL/dx leaves every parameter gradient bitwise as it was, and a training step without it runs none of the new
  kernels;
* the Attributor: a replay is bit-identical to the eager pass and to a second call, and a patient's result does not depend
  on its batch company or slot; integrated gradients against a float64 oracle trapezoid sum, with a completeness gap that
  shrinks with the number of points; a Trainer's parameters and Adam state are untouched by attribution;
* structure (last): an attribution pass launches no weight-gradient kernel, no LeakyReLU backward / cat / library GEMM, and
  writes no .grad."""
import types

import pytest
import torch

from conftest import assert_close_flips as _check
from oracle import restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def mlg():
    import multilevel_gnn_b200 as m
    m._cabi.lib()
    return m


def _model(mlg, cfg, seed, **overrides):
    args = mlg.configs.make_args(cfg, **overrides)
    torch.manual_seed(seed)
    model = mlg.MultilevelGNN(args)
    mlg.synth.multilevel_params(model, seed=seed)
    return model, args


def _to_dev(model):
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    return model


def _split(mlg, n, seed=7):
    raw = mlg.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * mlg.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = mlg.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(n)]
    return pts, topo


def _batch(mlg, pts, topo):
    return mlg.data.to_device(mlg.data.collate(pts, topo, pin=False), topo, DEV)


def _input_grads(model, batch, Rw, explicit=False):
    """(g_x, g_age, g_feat) of pred[:, 1].sum() + (pca_feature * Rw).sum() w.r.t. batch.x, batch.age and pca_feature."""
    x = batch.x.detach().clone().requires_grad_()
    age = batch.age.detach().clone().requires_grad_()
    b = types.SimpleNamespace(**vars(batch))
    b.x, b.age = x, age
    if explicit:
        pred, feat = model(b, x=x, gene_pca_match=b.gene_pca_match, raw_indice=b.raw_indice, age=age)
    else:
        pred, feat = model(b)
    loss = pred[:, 1].sum() + (feat * Rw).sum()
    return torch.autograd.grad(loss, [x, age, feat], allow_unused=True)


FULL = [("gbm", 3), ("kirc", 3), ("lgg", 3), ("gbm", 40), ("lgg", 64)]


@pytest.mark.parametrize("cfg,bsz", FULL, ids=["gbm_b3", "kirc_b3", "lgg_b3", "gbm_b40", "lgg_b64"])
def test_input_gradients_full_size_vs_oracle(mlg, cfg, bsz):
    model, args = _model(mlg, cfg, seed=41 + bsz)
    model.eval()
    batch = mlg.synth.multilevel_batch(batch_size=bsz, seed=41 + bsz)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    cb = types.SimpleNamespace(**vars(batch))
    cb.x = batch.x.clone().requires_grad_()
    cb.age = batch.age.clone().requires_grad_()
    pred_r, feat_r = R.multilevel_forward(sd, cb, args)
    Rw = torch.randn(feat_r.shape, generator=torch.Generator().manual_seed(bsz))
    g_r = torch.autograd.grad(pred_r[:, 1].sum() + (feat_r * Rw).sum(), [cb.x, cb.age, feat_r], allow_unused=True)
    _to_dev(model)
    g = _input_grads(model, batch.to(DEV), Rw.to(DEV))
    tag = "%s B=%d" % (cfg, bsz)
    for name, a, c in zip(("x", "age", "pca_feature"), g, g_r):
        if c is None:
            assert a is None, tag + " g_" + name
            continue
        _check(a, c, tag + " g_" + name, rtol=2e-4, atol=1e-5, l2=1e-3, outliers=1e-3)


ROUTES = [("factored_off", dict(FACTORED_RANK1=False)), ("factored_gather", dict(FACTORED_RANK1="gather")),
          ("transform_first_off", dict(TRANSFORM_FIRST=False)), ("act_fusion_off", dict(FUSE_ACT_BACKWARD=False)),
          ("explicit_x", {})]


@pytest.mark.parametrize("name,flags", ROUTES, ids=[r[0] for r in ROUTES])
def test_every_route_gives_the_input_gradient(mlg, name, flags):
    from multilevel_gnn_b200 import functional as Fn
    model, args = _model(mlg, "gbm", seed=12)
    _to_dev(model).eval()
    batch = mlg.synth.multilevel_batch(batch_size=40, seed=12).to(DEV)
    Rw = torch.randn(40, 32, 146, 6, generator=torch.Generator().manual_seed(3)).to(DEV)
    g0 = _input_grads(model, batch, Rw)
    saved = {k: (getattr(Fn, k) if hasattr(Fn, k) else getattr(mlg.MultilevelGNN, k)) for k in flags}
    try:
        for k, v in flags.items():
            setattr(Fn if hasattr(Fn, k) else mlg.MultilevelGNN, k, v)
        g1 = _input_grads(model, batch, Rw, explicit=(name == "explicit_x"))
    finally:
        for k, v in saved.items():
            setattr(Fn if hasattr(Fn, k) else mlg.MultilevelGNN, k, v)
    for what, a, c in zip(("x", "age", "pca_feature"), g1, g0):
        sc = float(c.abs().max().clamp_min(1e-30))
        _check(a / sc, c / sc, name + " g_" + what, rtol=1e-4, atol=5e-5, l2=1e-4, outliers=1e-3)


@pytest.mark.parametrize("over", [dict(merge_mode="add"), dict(value_att_mask=False)], ids=["merge_add", "no_value_mask"])
def test_mask_variants_vs_oracle(mlg, over):
    """The additive value mask and the unmasked pool (plain torch around the pool kernel) against the oracle."""
    model, args = _model(mlg, "gbm", seed=13, **over)
    model.eval()
    batch = mlg.synth.multilevel_batch(batch_size=3, seed=13)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    cb = types.SimpleNamespace(**vars(batch))
    cb.x = batch.x.clone().requires_grad_()
    cb.age = batch.age.clone().requires_grad_()
    pred_r, feat_r = R.multilevel_forward(sd, cb, args)
    Rw = torch.randn(feat_r.shape, generator=torch.Generator().manual_seed(4))
    g_r = torch.autograd.grad(pred_r[:, 1].sum() + (feat_r * Rw).sum(), [cb.x, feat_r])
    _to_dev(model)
    g = _input_grads(model, batch.to(DEV), Rw.to(DEV))
    _check(g[0], g_r[0], "g_x", rtol=2e-4, atol=1e-5, l2=1e-3, outliers=1e-3)
    _check(g[2], g_r[1], "g_pca_feature", rtol=2e-4, atol=1e-5, l2=1e-3, outliers=1e-3)


def _param_grads(model, batch, Rw, with_x):
    b = types.SimpleNamespace(**vars(batch))
    if with_x:
        b.x = batch.x.detach().clone().requires_grad_()
    pred, feat = model(b)
    params = [p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]
    return torch.autograd.grad(pred[:, 1].sum() + (feat * Rw).sum(), params, allow_unused=True)


class _Recorder:
    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            self.calls.append((name, a))
            return fn(*a)
        return call


NEW_TAGS = {"sage_rank1_bwd_xs", "pool_bwd_vm", "embed_scale_bwd_xs"}
NEW_CALLS = {"mlg_sage_rank1_bwd_xs", "mlg_pool_bwd_vm", "mlg_embed_scale_bwd_xs", "mlg_attr_accumulate"}


def test_training_gradients_unchanged(mlg, monkeypatch):
    from multilevel_gnn_b200 import _cabi
    model, args = _model(mlg, "gbm", seed=14)
    _to_dev(model).eval()
    batch = mlg.synth.multilevel_batch(batch_size=32, seed=14).to(DEV)
    Rw = torch.randn(32, 32, 146, 6, generator=torch.Generator().manual_seed(5)).to(DEV)
    g_plain = _param_grads(model, batch, Rw, False)
    g_x = _param_grads(model, batch, Rw, True)
    for a, c in zip(g_x, g_plain):
        assert (a is None and c is None) or torch.equal(a, c)
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    timer = _cabi.KernelTimer()
    _cabi.TIMER = timer
    try:
        model.train()
        _param_grads(model, batch, Rw, False)
        torch.cuda.synchronize()
        tags = timer.summary()
    finally:
        _cabi.TIMER = None
    assert not (set(tags) & NEW_TAGS), tags
    assert not ({c[0] for c in rec.calls} & NEW_CALLS)


def _attributor(mlg, model, args, pts, topo, B, **kw):
    return mlg.Attributor(model, args, batch_size=B, **kw).capture(_batch(mlg, pts[:B] if len(pts) >= B else
                                                                             (pts * B)[:B], topo))


def test_replay_matches_eager_and_repeats(mlg):
    model, args = _model(mlg, "gbm", seed=15)
    _to_dev(model).train()
    pts, topo = _split(mlg, 16, seed=15)
    at = _attributor(mlg, model, args, pts, topo, 16, method="saliency")
    assert model.training and all(p.grad is None for p in model.parameters())
    at.graph.replay()
    g_graph, pw_graph = at.out_g.clone(), at.out_pw.clone()
    at.eager()
    assert torch.equal(at.out_g, g_graph) and torch.equal(at.out_pw, pw_graph)
    r1 = at.attribute(pts, topo)
    r2 = at.attribute(pts, topo)
    assert torch.equal(r1.nodes, g_graph.cpu()) and torch.equal(r1.nodes, r2.nodes)
    assert torch.equal(r1.pathways, r2.pathways) and torch.equal(r1.pred, r2.pred)
    assert r1.genes.shape == (16, mlg.MultilevelGNN.GENES, 3) and r1.pathways.shape == (16, 146, 3)


@pytest.mark.parametrize("method,points,B", [("saliency", 1, 8), ("integrated_gradients", 4, 8)], ids=["saliency", "ig"])
def test_result_does_not_depend_on_company_or_slot(mlg, method, points, B):
    """n = 11 patients: full batches and a tail; each patient again alone (a tail batch of one) and in reversed order."""
    model, args = _model(mlg, "gbm", seed=16)
    _to_dev(model)
    pts, topo = _split(mlg, 11, seed=16)
    at = _attributor(mlg, model, args, pts, topo, B, method=method, points=points)
    full = at.attribute(pts, topo)
    rev = at.attribute(pts[::-1], topo)
    for i in (0, 5, 10):
        alone = at.attribute([pts[i]], topo)
        assert torch.equal(alone.nodes[0], full.nodes[i]), i
        assert torch.equal(alone.pathways[0], full.pathways[i]), i
        assert torch.equal(rev.nodes[10 - i], full.nodes[i]), i


def test_integrated_gradients_vs_oracle(mlg):
    """Two gbm patients, points = 8: the trapezoid sum of oracle float64 gradients at the same interpolants; then the
    completeness gap shrinks from 8 to 64 points (64 points at B = 32: two replays per patient, accumulated on the device)."""
    from multilevel_gnn_b200 import attribution as A
    model, args = _model(mlg, "gbm", seed=17)
    sd = {k: v.detach().clone().double() for k, v in model.state_dict().items()}
    pts, topo = _split(mlg, 2, seed=17)
    m = 8
    al = A.ig_alphas(m)
    tw = A.trapezoid_weights(m)
    xs = torch.stack([pts[i].x.reshape(-1).double() for i in range(2)])                 # [2, N]
    xin = (al.view(1, m, 1) * xs.view(2, 1, -1)).reshape(2 * m, -1).clone().requires_grad_()
    cb = mlg.data.collate([pts[0]] * m + [pts[1]] * m, topo, pin=False)
    cb = types.SimpleNamespace(**{k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v)
                                  for k, v in vars(cb).items()})
    cb.x = xin.reshape(-1, 1)
    pred_r, _ = R.multilevel_forward(sd, cb, args)
    g_r, = torch.autograd.grad(pred_r[:, 1].sum(), [xin])
    ig_r = xs * (g_r.view(2, m, -1) * tw.view(1, m, 1)).sum(1)
    _to_dev(model)
    at = _attributor(mlg, model, args, pts, topo, 16, method="integrated_gradients", points=m)
    res = at.attribute(pts, topo)
    sc = float(ig_r.abs().max())
    # a LeakyReLU unit within fp32 rounding of 0 moves its fan-in (DESIGN section 2); the sum runs over 8 fp32 gradients, each
    # held to the full-size tests' bounds (1e-3 of the entries outside the element-wise bound, relative L2 1e-3) by
    # test_input_gradients_full_size_vs_oracle, against a float64 oracle here: twice the norm-wise bound (measured 1.2e-3)
    _check(res.nodes.double() / sc, ig_r / sc, "IG nodes", rtol=2e-4, atol=5e-5, l2=2e-3, outliers=8e-3)
    gap = {}
    for pts_m, B in ((8, 16), (64, 32)):
        at = _attributor(mlg, model, args, pts, topo, B, method="integrated_gradients", points=pts_m)
        r = at.attribute(pts, topo)
        f = at.attribute(pts, topo)
        assert torch.equal(r.nodes, f.nodes)
        span = (r.delta.double() + r.nodes.double().sum(1)).abs()          # F(x) - F(x')
        gap[pts_m] = (r.delta.double().abs() / span.clamp_min(1e-12)).max().item()
    assert gap[64] < gap[8] and gap[64] < 0.05, gap


def test_trainer_state_untouched(mlg):
    """Trainer step -> attribute -> Trainer step leaves the flat parameters and Adam moments bitwise equal to two plain
    steps; an Attributor captured before the Trainer re-homed the parameters re-captures and reads the updated values."""
    B = 8
    pts, topo = _split(mlg, 16, seed=18)
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(DEV)
    states = []
    for with_attr in (False, True):
        model, args = _model(mlg, "gbm", seed=18)
        _to_dev(model)
        at = _attributor(mlg, model, args, pts, topo, B, method="saliency") if with_attr else None
        tr = mlg.train.Trainer(model, args, weight)
        tr.capture(_batch(mlg, pts[:B], topo))
        torch.manual_seed(1)
        tr.step(_batch(mlg, pts[:B], topo))
        if with_attr:
            old = at.graph
            r = at.attribute(pts, topo)
            assert at.graph is not old
            at.eager()        # static buffers hold the last replay's patients: pts[8:16]
            assert torch.equal(r.nodes[B:], at.out_g.cpu())
        tr.step(_batch(mlg, pts[B:], topo))
        torch.cuda.synchronize()
        states.append([t.clone() for t in (tr.opt.flat_p, tr.opt.exp_avg, tr.opt.exp_avg_sq)])
    for a, c in zip(*states):
        assert torch.equal(a, c)


def test_zz_attribution_structure(mlg, monkeypatch):
    """An attribution pass: no weight-gradient kernel (xty / fold backward / wcolsum / pool weight gradient / rank-1 rows h /
    head weight gradients), no LeakyReLU backward, cat or library GEMM, and no .grad written."""
    from multilevel_gnn_b200 import _cabi
    model, args = _model(mlg, "kirc", seed=19)
    _to_dev(model)
    pts, topo = _split(mlg, 8, seed=19)
    at = _attributor(mlg, model, args, pts, topo, 8, method="integrated_gradients", points=8)
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        at.eager()
        torch.cuda.synchronize()
    names = [c[0] for c in rec.calls]
    banned = ("mlg_xty", "mlg_sage_fold_stacked_bwd", "mlg_sage_fold_bwd", "mlg_wcolsum", "mlg_pool_bwd_w",
              "mlg_pool_bwd_layout", "mlg_sage_rank1_bwd_rows", "mlg_sage_rank1_bwd")
    assert not [n for n in names if n.startswith(banned) and not n.startswith("mlg_sage_rank1_bwd_xs")
                and not n.endswith("_supported")], names
    assert "mlg_sage_rank1_bwd_xs" in names and "mlg_pool_bwd_vm" in names
    for n, a in rec.calls:
        if n == "mlg_head_mlp_bwd":
            assert all(v is None for v in a[16:20])
        if n == "mlg_head_conv_pool_bwd":
            assert all(v is None for v in a[15:20])
        if n == "mlg_pool_bwd_vm":
            assert a[15] is None and a[16] is None
    ops = {e.key for e in prof.key_averages()}
    bad = {o for o in ops if o in ("aten::leaky_relu_backward", "aten::cat", "aten::mm", "aten::addmm", "aten::bmm",
                                    "aten::matmul", "aten::linear")}
    assert not bad, bad
    assert all(p.grad is None for p in model.parameters())
