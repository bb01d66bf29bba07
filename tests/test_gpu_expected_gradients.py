"""Expected gradients against a background cohort on the fused kernels (Attributor(method="expected_gradients")).

* the two kernels: mlg_attr_eg_interp equals the header's fmaf formula evaluated on the host, bit for bit, is exact at
  alpha in {0, 1} and flags (without reading) a bank row index outside [0, M); mlg_attr_eg_accumulate against float64;
* exactness: a background of one row equal to the patient gives attributions and a completeness gap of exactly 0;
* the attributions against a float64 oracle (autograd through oracle/restated.py at the same interpolants and draws);
* a patient's nodes / pred / delta have the same bits at batch_size 8 and 32 (other slots and companies), on repeat, and a
  replay equals the eager pass; the completeness gap shrinks from S = 4 to S = 64;
* a Trainer's state is untouched; structure (last): no weight-gradient kernel or library GEMM runs, no .grad is written, and
  the training step's launches are unchanged."""
import types

import pytest
import torch

from conftest import assert_close_flips as _check
from oracle import restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EG = "expected_gradients"


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
    return model, args


def _to_dev(model):
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    return model


def _split(mlg, n, seed):
    raw = mlg.synth.multilevel_batch(batch_size=n, seed=seed)
    n1 = 3 * mlg.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // n
    topo = mlg.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    pts = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(n)]
    return pts, topo


def _bank(pts):
    return torch.stack([p.x.reshape(-1) for p in pts])


def _attributor(mlg, model, args, pts, topo, B, **kw):
    batch = mlg.data.to_device(mlg.data.collate((pts * B)[:B], topo, pin=False), topo, DEV)
    return mlg.Attributor(model, args, batch_size=B, method=EG, **kw).capture(batch)


def _fma32(a, x, t):
    """fmaf(a, x, t) of fp32 tensors on the host, correctly rounded: a * x is exact in float64; the float64 sum's rounding
    error (TwoSum) breaks the ties that rounding the float64 sum to fp32 would resolve blindly."""
    p, t = a.double() * x.double(), t.double()
    s = p + t
    bp = s - t
    err = (p - bp) + (t - (s - bp))
    r = s.float()
    d = s - r.double()
    nb = torch.nextafter(r, torch.where(d > 0, torch.full_like(r, float("inf")), torch.full_like(r, float("-inf"))))
    tie = (d != 0) & (s == (r.double() + nb.double()) / 2) & (err != 0)
    return torch.where(tie & ((err > 0) == (d > 0)), nb, r)


def _interp_host(alpha, x, bank, j):
    """The header's formula: fmaf(alpha_s, x[s, :], (1 - alpha_s) * bank[j_s, :]) in fp32."""
    a = alpha.view(-1, 1).expand_as(x)
    return _fma32(a, x, (1 - a) * bank[j.long()])


def test_interp_kernel_bitwise(mlg):
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()
    g = torch.Generator().manual_seed(1)
    B, N, M = 12, 15405, 5
    x = torch.randn(B, N, generator=g) * torch.rand(B, N, generator=g).pow(3) * 40
    bank = torch.randn(M, N, generator=g)
    j = torch.randint(0, M, (B,), generator=g, dtype=torch.int32)
    alpha = torch.cat([mlg.attribution.eg_draws(2, 0, B - 2, M)[1].float(), torch.tensor([0.0, 1.0])])
    dx, db, dj, da = (t.to(DEV) for t in (x, bank, j, alpha))
    out = torch.empty(B, N, device=DEV)
    bad = torch.zeros(1, dtype=torch.int32, device=DEV)
    _cabi.check(L.mlg_attr_eg_interp(_cabi.fptr(dx), _cabi.fptr(db), M, _cabi.iptr(dj), _cabi.fptr(da), B, N, _cabi.fptr(out),
                                     _cabi.iptr(bad), _cabi.stream_ptr()), "mlg_attr_eg_interp")
    got = out.cpu()
    assert int(bad.item()) == 0
    assert torch.equal(got.view(torch.int32), _interp_host(alpha, x, bank, j).view(torch.int32))
    assert torch.equal(got[B - 2], bank[j[B - 2].long()]) and torch.equal(got[B - 1], x[B - 1])     # alpha = 0 / alpha = 1
    # a row index outside [0, M) is not read: that row is NaN, the others are untouched, and the flag is raised
    dj[3] = M
    dj[7] = -1
    _cabi.check(L.mlg_attr_eg_interp(_cabi.fptr(dx), _cabi.fptr(db), M, _cabi.iptr(dj), _cabi.fptr(da), B, N, _cabi.fptr(out),
                                     _cabi.iptr(bad), _cabi.stream_ptr()), "mlg_attr_eg_interp")
    got2 = out.cpu()
    assert int(bad.item()) == 1
    assert bool(got2[3].isnan().all()) and bool(got2[7].isnan().all())
    keep = [s for s in range(B) if s not in (3, 7)]
    assert torch.equal(got2[keep], got[keep])
    assert L.mlg_attr_eg_interp(None, _cabi.fptr(db), M, None, None, B, N, None, None, None) < 0
    assert L.mlg_attr_eg_interp(_cabi.fptr(dx), _cabi.fptr(db), 0, _cabi.iptr(dj), _cabi.fptr(da), B, N, _cabi.fptr(out),
                                _cabi.iptr(bad), _cabi.stream_ptr()) < 0


def test_accumulate_kernel_vs_float64(mlg):
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()
    g = torch.Generator().manual_seed(2)
    slots, N, M = 30, 15405, 7
    counts = [5, 1, 9, 15]
    ptr = torch.tensor([0] + list(torch.tensor(counts).cumsum(0)), dtype=torch.int32)
    gr = torch.randn(slots, N, generator=g)
    x = torch.randn(slots, N, generator=g)
    bank = torch.randn(M, N, generator=g)
    j = torch.randint(0, M, (slots,), generator=g, dtype=torch.int32)
    w = torch.rand(slots, generator=g)
    acc = torch.randn(len(counts), N, generator=g)
    d = [t.to(DEV) for t in (gr, x, bank, j, w, ptr, acc)]
    bad = torch.zeros(1, dtype=torch.int32, device=DEV)
    terms = (w.double().view(-1, 1) * (x.double() - bank.double()[j.long()]) * gr.double())
    for accumulate in (0, 1):
        out = d[6].clone()
        _cabi.check(L.mlg_attr_eg_accumulate(_cabi.fptr(d[0]), _cabi.fptr(d[1]), _cabi.fptr(d[2]), M, _cabi.iptr(d[3]),
                                             _cabi.fptr(d[4]), _cabi.iptr(d[5]), len(counts), N, accumulate, _cabi.fptr(out),
                                             _cabi.iptr(bad), _cabi.stream_ptr()), "mlg_attr_eg_accumulate")
        ref = acc.double() if accumulate else torch.zeros(len(counts), N, dtype=torch.float64)
        mag = ref.abs().clone()
        for p in range(len(counts)):
            seg = terms[int(ptr[p]):int(ptr[p + 1])]
            ref[p] += seg.sum(0)
            mag[p] += seg.abs().sum(0)
        err = (out.cpu().double() - ref).abs()
        assert bool((err <= 1e-6 * mag).all()), float((err / mag.clamp_min(1e-30)).max())
    assert int(bad.item()) == 0


def test_background_of_the_patient_gives_exact_zeros(mlg):
    model, args = _model(mlg, "gbm", seed=61)
    _to_dev(model)
    pts, topo = _split(mlg, 3, seed=61)
    for i in (0, 2):
        at = _attributor(mlg, model, args, [pts[i]], topo, 8, background=_bank([pts[i]]), samples=4, seed=i,
                         completeness=True)
        r = at.attribute([pts[i]], topo)
        assert bool((r.nodes == 0).all()) and float(r.delta[0]) == 0.0, (i, float(r.delta[0]))
        assert bool(r.pred.isfinite().all()) and r.genes.shape == (1, mlg.MultilevelGNN.GENES, 3)


@pytest.mark.parametrize("cfg,B,S", [("gbm", 16, 8), ("kirc", 3, 4)], ids=["gbm_b16_s8", "kirc_b3_s4"])
def test_expected_gradients_vs_oracle(mlg, cfg, B, S):
    """Three patients against a background of M = 5: sum_k (x - x'_k) g_k / S with float64 oracle gradients at the same fp32
    interpolants of the same draws.  kirc at B = 3 spans several replays per patient (accumulated on the device)."""
    from multilevel_gnn_b200 import attribution as A
    model, args = _model(mlg, cfg, seed=62)
    sd = {k: v.detach().clone().double() for k, v in model.state_dict().items()}
    pts, topo = _split(mlg, 8, seed=62)
    pats, bank = pts[:3], _bank(pts[3:])
    M, seed = bank.shape[0], 5
    J, Al = (torch.stack(t) for t in zip(*(A.eg_draws(seed, i, S, M) for i in range(3))))
    x = _bank(pats)                                                              # [3, N]
    xb = bank[J]                                                                 # [3, S, N]
    xin32 = _interp_host(Al.float().reshape(-1), x.repeat_interleave(S, 0), bank, J.reshape(-1))
    xin = xin32.double().clone().requires_grad_()
    cb = mlg.data.collate([pats[p] for p in range(3) for _ in range(S)], topo, pin=False)
    cb = types.SimpleNamespace(**{k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v)
                                  for k, v in vars(cb).items()})
    cb.x = xin.reshape(-1, 1)
    pred_r, _ = R.multilevel_forward(sd, cb, args)
    g_r, = torch.autograd.grad(pred_r[:, 1].sum(), [xin])
    phi_r = ((x.double().unsqueeze(1) - xb.double()) * g_r.view(3, S, -1)).sum(1) / S
    cx = mlg.data.collate(pats, topo, pin=False)
    cx = types.SimpleNamespace(**{k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v)
                                  for k, v in vars(cx).items()})
    with torch.no_grad():
        fx_r, _ = R.multilevel_forward(sd, cx, args)
    _to_dev(model)
    at = _attributor(mlg, model, args, pats, topo, B, background=bank, samples=S, seed=seed, completeness=True)
    res = at.attribute(pats, topo)
    sc = float(phi_r.abs().max())
    # the tolerance of test_integrated_gradients_vs_oracle: a sum over S fp32 gradients, each held to the full-size bounds
    _check(res.nodes.double() / sc, phi_r / sc, "EG nodes", rtol=2e-4, atol=5e-5, l2=2e-3, outliers=8e-3)
    assert torch.allclose(res.pred.double(), fx_r, rtol=1e-4, atol=1e-5)
    assert res.delta.shape == (3,) and bool(res.delta.isfinite().all())
    assert res.pathways.shape == (3, 146, 3) and res.genes.shape == (3, mlg.MultilevelGNN.GENES, 3)


def test_same_bits_in_any_batch_slot_and_company(mlg):
    """11 patients, S = 5 with completeness (10 slots per patient): at B = 8 a patient spans two replays, at B = 32 three
    patients share a replay at slots 0 / 10 / 20; a shorter dataset puts the first patients in other company."""
    model, args = _model(mlg, "gbm", seed=63)
    _to_dev(model)
    pts, topo = _split(mlg, 17, seed=63)
    data, bank = pts[:11], _bank(pts[11:])
    res = {}
    for B in (8, 32):
        at = _attributor(mlg, model, args, data, topo, B, background=bank, samples=5, seed=9, completeness=True)
        r1 = at.attribute(data, topo)
        r2 = at.attribute(data, topo)
        for f in ("nodes", "pathways", "pred", "delta"):
            assert torch.equal(getattr(r1, f), getattr(r2, f)), (B, f)
        short = at.attribute(data[:4], topo)
        for f in ("nodes", "pathways", "pred", "delta"):
            assert torch.equal(getattr(short, f), getattr(r1, f)[:4]), (B, f)
        res[B] = r1
    for f in ("nodes", "pathways", "pred", "delta"):
        assert torch.equal(res[8].__getattribute__(f), res[32].__getattribute__(f)), f
    assert float(res[8].nodes.abs().max()) > 0
    # a replay is the eager pass, bit for bit (the static buffers hold the last replay's patients)
    at.j.copy_(torch.arange(32, device=DEV, dtype=torch.int32) % bank.shape[0])
    at.alpha.copy_(torch.linspace(0.05, 0.95, 32, device=DEV))
    at.graph.replay()
    g_graph, p_graph = at.out_g.clone(), at.out_pred.clone()
    at.eager()
    assert torch.equal(at.out_g, g_graph) and torch.equal(at.out_pred, p_graph)


def test_completeness_gap_shrinks_with_samples(mlg):
    model, args = _model(mlg, "gbm", seed=64)
    _to_dev(model)
    pts, topo = _split(mlg, 24, seed=64)
    data, bank = pts[:16], _bank(pts[16:])
    gap = {}
    for S in (4, 64):
        at = _attributor(mlg, model, args, data, topo, 32, background=bank, samples=S, seed=1, completeness=True)
        gap[S] = float(at.attribute(data, topo).delta.double().abs().mean())
    assert gap[64] < gap[4], gap


def test_trainer_state_untouched(mlg):
    """Trainer step -> attribute -> Trainer step leaves the flat parameters and Adam moments bitwise equal to two plain steps;
    the Attributor captured before the Trainer re-homed the parameters re-captures."""
    B = 8
    pts, topo = _split(mlg, 19, seed=65)
    data, bank = pts[:16], _bank(pts[16:])
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(DEV)

    def batch(p):
        return mlg.data.to_device(mlg.data.collate(p, topo, pin=False), topo, DEV)

    states = []
    for with_attr in (False, True):
        model, args = _model(mlg, "gbm", seed=65)
        _to_dev(model)
        at = _attributor(mlg, model, args, data, topo, B, background=bank, samples=3, completeness=True) if with_attr else None
        tr = mlg.train.Trainer(model, args, weight)
        tr.capture(batch(data[:B]))
        torch.manual_seed(1)
        tr.step(batch(data[:B]))
        if with_attr:
            old = at.graph
            at.attribute(data[:5], topo)
            assert at.graph is not old
        tr.step(batch(data[B:]))
        torch.cuda.synchronize()
        states.append([t.clone() for t in (tr.opt.flat_p, tr.opt.exp_avg, tr.opt.exp_avg_sq)])
    for a, c in zip(*states):
        assert torch.equal(a, c)


class _Recorder:
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


def test_zz_expected_gradients_structure(mlg, monkeypatch):
    """The replay body: no weight-gradient kernel (xty / fold backward / wcolsum / pool weight gradient / rank-1 rows h /
    head weight gradients), no library GEMM; an attribute call adds only the accumulations and writes no .grad; a training
    step launches the same native calls before and after, none of them the new ones."""
    from multilevel_gnn_b200 import _cabi
    model, args = _model(mlg, "kirc", seed=66)
    _to_dev(model)
    pts, topo = _split(mlg, 6, seed=66)
    data, bank = pts[:4], _bank(pts[4:])
    batch = mlg.data.to_device(mlg.data.collate(data, topo, pin=False), topo, DEV)
    before = _step_calls(mlg, model, args, batch, monkeypatch)
    assert not [n for n in before if n.startswith("mlg_attr")]
    for p in model.parameters():
        p.grad = None
    at = _attributor(mlg, model, args, data, topo, 4, background=bank, samples=3, completeness=True)
    rec = _Recorder(_cabi.lib())
    monkeypatch.setattr(_cabi, "_lib", rec)
    gemms = ("aten::mm", "aten::addmm", "aten::bmm", "aten::matmul", "aten::linear")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        at.eager()
        torch.cuda.synchronize()
    names = [c[0] for c in rec.calls]
    banned = ("mlg_xty", "mlg_sage_fold_stacked_bwd", "mlg_sage_fold_bwd", "mlg_wcolsum", "mlg_pool_bwd_w",
              "mlg_pool_bwd_layout", "mlg_sage_rank1_bwd_rows", "mlg_adam", "mlg_peer")
    assert not [n for n in names if n.startswith(banned) and not n.endswith("_supported")], names
    assert names.count("mlg_attr_eg_interp") == 1 and "mlg_sage_rank1_bwd_xs" in names and "mlg_pool_bwd_vm" in names
    for n, a in rec.calls:
        if n == "mlg_head_mlp_bwd":
            assert all(v is None for v in a[16:20])
        if n == "mlg_head_conv_pool_bwd":
            assert all(v is None for v in a[15:20])
    assert not {e.key for e in prof.key_averages()} & set(gemms + ("aten::cat", "aten::leaky_relu_backward"))
    rec.calls.clear()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        at.attribute(data, topo)           # (host-side torch.stack of the plan and of collate runs aten::cat on CPU tensors)
    assert {c[0] for c in rec.calls} == {"mlg_attr_eg_accumulate", "mlg_attr_accumulate"}, {c[0] for c in rec.calls}
    assert not {e.key for e in prof.key_averages()} & set(gemms)
    monkeypatch.setattr(_cabi, "_lib", rec._lib)
    assert all(p.grad is None for p in model.parameters())
    for p in model.parameters():
        p.grad = None
    assert _step_calls(mlg, model, args, batch, monkeypatch) == before
