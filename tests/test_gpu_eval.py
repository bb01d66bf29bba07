"""Forward-only evaluation: MultilevelGNN.predict on the fused training kernels, the captured train.Evaluator over a split, and
the split metrics kernel mlg_eval_metrics.

* predict against the CPU oracle at full size (N = 15 405 nodes, G = 25 015 gene slots), at the tolerances of
  test_gpu_fullsize.py, and against today's eager ``model.eval()`` + ``no_grad`` route;
* a captured replay is bit-identical to eager predict; so is every row of a padded tail batch to the same sample evaluated in
  another batch composition (the graphs of a batch do not interact in any forward kernel);
* the Evaluator follows the Trainer's in-place parameter updates (fused FlatAdam) and re-captures when storage moved;
* the metrics kernel against NumPy and torch.nn.BCELoss;
* structure: predict launches the fused forward kernels only -- no backward kernel, no sign-bit words, no library GEMM / cat /
  LeakyReLU, and nothing that outlives the call but its two outputs."""
import types

import numpy as np
import pytest
import torch

import eval_ref
from conftest import assert_close
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
    """n patient records sharing one gene network (as one fold of the reference's dataset) and its FoldTopology."""
    raw = mlg.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * mlg.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = mlg.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(n)]
    return pts, topo


def _batch(mlg, pts, topo):
    return mlg.data.to_device(mlg.data.collate(pts, topo, pin=False), topo, DEV)


FULL = [("gbm", 3), ("kirc", 3), ("lgg", 3), ("gbm", 40), ("gbm", 32), ("kirc", 64), ("gbm", 256)]
CHUNKED = 32       # from this width on: the float64 oracle over chunks of graphs (test_gpu_batch_widths.py)


@pytest.mark.parametrize("cfg,bsz", FULL, ids=["gbm_b3", "kirc_b3", "lgg_b3", "gbm_b40", "gbm_b32", "kirc_b64", "gbm_b256"])
def test_predict_full_size_vs_oracle(mlg, cfg, bsz):
    """pred and pca_feature of predict against oracle.multilevel_forward on the CPU; the model is left in TRAINING mode
    (predict must not apply dropout) and comes back in it."""
    from test_gpu_batch_widths import ORACLE_CHUNK, forward_chunks, oracle_params
    model, args = _model(mlg, cfg, seed=31 + bsz)
    batch = mlg.synth.multilevel_batch(batch_size=bsz, seed=31 + bsz)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    _to_dev(model).train()
    pred, feat = model.predict(batch.to(DEV))
    assert model.training
    assert not pred.requires_grad and pred.grad_fn is None and feat.grad_fn is None
    tag = "%s B=%d predict" % (cfg, bsz)
    chunked = bsz >= CHUNKED
    dtype = torch.float64 if chunked else torch.float32
    with torch.no_grad():
        for g0, g1, _, pred_r, feat_r, _ in forward_chunks(oracle_params(sd, (), dtype), batch, args, 3 * mlg.MultilevelGNN.GENES,
                                                           chunk=ORACLE_CHUNK if chunked else bsz, dtype=dtype):
            _check(pred[g0:g1], pred_r, "%s graphs %d..%d pred" % (tag, g0, g1 - 1))
            _check(feat[g0:g1], feat_r, "%s graphs %d..%d pca_feature" % (tag, g0, g1 - 1))


def test_predict_matches_eager_eval(mlg):
    """predict against the route ``model(batch)`` takes under eval() + no_grad (generic layers, materialised first-layer
    input), which stays as it was."""
    model, _ = _model(mlg, "gbm", seed=3)
    _to_dev(model).eval()
    batch = mlg.synth.multilevel_batch(batch_size=8, seed=3).to(DEV)
    with torch.no_grad():
        pred_e, feat_e = model(batch)
    pred, feat = model.predict(batch)
    assert_close(pred, pred_e, rtol=1e-4, what="pred")
    assert_close(feat, feat_e, rtol=1e-4, what="pca_feature")


def test_captured_replay_is_bit_identical_to_predict(mlg):
    model, args = _model(mlg, "gbm", seed=4)
    _to_dev(model)
    pts, topo = _split(mlg, 32, seed=4)
    batch = _batch(mlg, pts, topo)
    ev = mlg.train.Evaluator(model, args, batch_size=32).capture(batch)
    assert model.training                                  # capture restores the mode
    ev.graph.replay()
    want = model.predict(batch)[0]
    assert torch.equal(ev.static_pred, want)
    res = ev.evaluate(pts, topo)
    assert res.n == 32 and torch.equal(res.pred, want.cpu())


def test_padded_tail_rows_do_not_depend_on_the_batch(mlg):
    """n = 45 at B = 32: the second batch holds 13 samples in the first slots, the rest of the static buffers are stale.  Each
    prediction equals (bitwise) that sample evaluated in another slot of a full batch with other company."""
    model, args = _model(mlg, "gbm", seed=5)
    _to_dev(model).eval()
    pts, topo = _split(mlg, 45, seed=5)
    ev = mlg.train.Evaluator(model, args, batch_size=32).capture(_batch(mlg, pts[:32], topo))
    res = ev.evaluate(pts, topo)
    assert res.n == 45 and res.pred.shape == (45, 2)
    # two full batches that put every sample in another slot and other company: [13..44] and [44..26] + [0..12]
    got = torch.empty(45, 2)
    a = list(range(13, 45))
    got[a] = model.predict(_batch(mlg, [pts[i] for i in a], topo))[0].cpu()
    b = list(range(44, 25, -1)) + list(range(13))
    got[:13] = model.predict(_batch(mlg, [pts[i] for i in b], topo))[0].cpu()[19:]
    diff = float((got - res.pred).abs().max())
    assert torch.equal(got, res.pred), "max |diff| %.3e" % diff
    bce, acc, auc = eval_ref.metrics(res.pred.numpy(), torch.stack([torch.as_tensor(p.y) for p in pts]).numpy())
    assert res.acc == np.float32(acc) and res.auc == np.float32(auc)
    assert res.bce == pytest.approx(bce, rel=1e-5)


def test_evaluator_follows_trainer_updates(mlg):
    """Capture first, then a Trainer re-homes the parameters into its flat FlatAdam buffer (storage moves: evaluate must
    re-capture) and takes 3 captured steps; a 4th step updates them in place (the graph must read the new values)."""
    model, args = _model(mlg, "gbm", seed=6)
    _to_dev(model)
    B = 8
    pts, topo = _split(mlg, 24, seed=6)
    batch = _batch(mlg, pts[:B], topo)
    ev = mlg.train.Evaluator(model, args, batch_size=B).capture(batch)
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(DEV)
    tr = mlg.train.Trainer(model, args, weight)
    assert isinstance(tr.opt, mlg.train.FlatAdam)
    tr.capture(_batch(mlg, pts[B:2 * B], topo))
    for _ in range(3):
        tr.step()
    old_graph = ev.graph
    res = ev.evaluate(pts, topo)
    assert ev.graph is not old_graph
    want = torch.cat([model.predict(_batch(mlg, pts[i:i + B], topo))[0] for i in range(0, 24, B)]).cpu()
    assert torch.equal(res.pred, want)
    tr.step()
    graph = ev.graph
    res2 = ev.evaluate(pts, topo)
    assert ev.graph is graph
    want2 = torch.cat([model.predict(_batch(mlg, pts[i:i + B], topo))[0] for i in range(0, 24, B)]).cpu()
    assert torch.equal(res2.pred, want2) and not torch.equal(want2, want)


def _metric_cases():
    rng = np.random.default_rng(11)
    out = []
    p1 = rng.random(1000)
    out.append(("random", np.stack([1 - p1, p1], 1), rng.integers(0, 2, 1000), None))
    p1 = np.floor(rng.random(5000) * 4) / 4                 # heavy ties, exact 0 and 1 scores included
    out.append(("ties", np.stack([1 - p1, p1], 1), rng.integers(0, 2, 5000), [0.8, 1.3]))
    p1 = rng.random(300)
    out.append(("one_class", np.stack([1 - p1, p1], 1), np.ones(300, int), None))
    out.append(("n1", np.array([[0.3, 0.7]]), np.array([1]), None))
    p1 = rng.random(70000)[:65536]
    out.append(("max_n", np.stack([1 - p1, p1], 1), rng.integers(0, 2, 65536), [2.0, 0.5]))
    return out


@pytest.mark.parametrize("case", _metric_cases(), ids=lambda c: c[0])
def test_eval_metrics_kernel(mlg, case):
    name, pred, labels, w = case
    y = np.eye(2)[labels]
    pd, yd = torch.tensor(pred, dtype=torch.float32, device=DEV), torch.tensor(y, dtype=torch.float32, device=DEV)
    wd = None if w is None else torch.tensor(w, dtype=torch.float32, device=DEV)
    out = mlg.train.eval_metrics(pd, yd, wd)
    again = mlg.train.eval_metrics(pd, yd, wd)
    assert torch.equal(out, again) or (torch.isnan(out[2]) and torch.equal(out[:2], again[:2]))
    bce, acc, auc = eval_ref.metrics(pd.double().cpu().numpy(), y, w)
    got = out.cpu().numpy()
    assert got[1] == np.float32(acc), name
    assert (np.isnan(got[2]) and np.isnan(auc)) or got[2] == np.float32(auc), (name, got[2], auc)
    assert got[0] == pytest.approx(bce, rel=1e-5), name
    crit = torch.nn.BCELoss(weight=None if wd is None else wd.expand(len(labels), 2))
    assert float(got[0]) == pytest.approx(float(crit(pd, yd)), rel=1e-5), name


def test_eval_metrics_rejects_oversized_split(mlg):
    pd = torch.full((65537, 2), 0.5, device=DEV)
    with pytest.raises(RuntimeError, match="n <= 65536"):
        mlg.train.eval_metrics(pd, pd)


class _Recorder:
    """Stands in for the loaded library: records every call's name and arguments."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            self.calls.append((name, a))
            return fn(*a)
        return call


def test_predict_structure(mlg, monkeypatch):
    from multilevel_gnn_b200 import _cabi
    model, _ = _model(mlg, "gbm", seed=8)
    _to_dev(model).train()
    batch = mlg.synth.multilevel_batch(batch_size=8, seed=8).to(DEV)
    model.predict(batch)                                    # builds the cached CSR / pool layouts
    torch.cuda.synchronize()
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    timer = _cabi.KernelTimer()
    _cabi.TIMER = timer
    before = torch.cuda.memory_allocated()
    try:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
            pred, feat = model.predict(batch)
        tags = timer.summary()
    finally:
        _cabi.TIMER = None
    kept = torch.cuda.memory_allocated() - before
    for t in ("sage_rank1_fwd", "sage_aggr_fwd", "pool_fwd", "head_conv_pool_fwd", "head_mlp_fwd"):
        assert tags.get(t, {}).get("launches", 0) >= 1, (t, sorted(tags))
    assert not [t for t in tags if t.endswith("_bwd") or "_bwd_" in t], sorted(tags)
    names = {e.name for e in prof.events()}
    bad = [nm for nm in names if nm in ("aten::cat", "aten::addmm", "aten::mm") or "leaky_relu" in nm]
    assert not bad, bad
    called = [c for c, _ in rec.calls]
    assert "mlg_sage_rank1_fwd_rows_nm" in called and "mlg_gather_sum_nm_ex" in called, called
    for name, a in rec.calls:
        if name in ("mlg_sage_rank1_fwd_rows", "mlg_sage_rank1_fwd_rows_nm"):
            assert a[16] is None, "predict asked the first layer for sign-bit words"
    # nothing outlives the call but pred and the pooled buffer pca_feature views
    def block(nbytes):
        return -(-nbytes // 512) * 512
    assert kept == block(pred.numel() * 4) + block(feat.untyped_storage().nbytes()), kept
