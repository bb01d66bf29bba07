"""Full-size parity of the DEFAULT CUDA path against the CPU oracle (oracle/restated.py) -- not against another CUDA
formulation of itself.  Sizes are the benchmarked ones (N = 15 405 nodes and G = 25 015 gene slots per graph, hub rows,
factored first layer + transform-first second layer, more than 32 replicas; GENConv at N = 100 k, k = 16, H = 128; DiffPool on
the tensor-core path at N = 4096); batches are small enough that the oracle finishes in seconds on the box's host cores.

Reference lines the oracle follows: models/multilevel_gnn.py:132-292,329-348, gcn_lib/sparse/torch_vertex.py:72-101,269-294,
gcn_lib/sparse/torch_message.py:44-85,175-179, models/diff_pooling.py:24-65,116-133, train.py:60,118.
Tolerance: fp32 rtol 1e-4 on activations / loss (BASELINE.json north_star) with a norm-wise bound of 2e-5 so that small entries
are not hidden behind the largest one; gradients: rtol 2e-4 element-wise with at most 0.1 % of the entries outside it (activation
branch flips at |z| ~ fp32 rounding, see _check) and a norm-wise bound of 1e-3 (2e-3 for the 100k-node GENConv, where one flipped
LayerNorm-ReLU unit moves ~2000 gradient entries); bf16 tensor-core DiffPool: 3e-2 (fp32 accumulate).
"""
import types

import pytest
import torch

from conftest import assert_close
from oracle import restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def mlg():
    import multilevel_gnn_b200 as m
    m._cabi.lib()
    return m


from conftest import assert_close_flips as _check, rel_l2 as _rel_l2  # noqa: E402


def _cpu_batch(b):
    return types.SimpleNamespace(**{k: v for k, v in vars(b).items()})


def _multilevel_case(mlg, cfg, bsz, seed, **overrides):
    from multilevel_gnn_b200 import configs, synth
    args = configs.make_args(cfg, **overrides)
    torch.manual_seed(seed)
    model = mlg.MultilevelGNN(args)
    synth.multilevel_params(model, seed=seed)
    model.eval()                       # dropout = identity (the oracle has none); gradients still flow
    batch = synth.multilevel_batch(batch_size=bsz, seed=seed)
    weight = (torch.rand(bsz, 2, generator=torch.Generator().manual_seed(seed)) + 0.5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return model, args, batch, weight, sd


FULL = [("gbm", 3, {}), ("kirc", 3, {}), ("lgg", 3, {"gnn_name": "rsage"}), ("lgg", 3, {}), ("gbm", 40, {}),
        ("gbm", 32, {}), ("kirc", 64, {}), ("lgg", 64, {}), ("gbm", 256, {})]
# the benchmarked widths (gbm 32, kirc / lgg 64, the strong-scaling leg's 256 graphs on one GPU) take the float64 oracle over
# chunks of graphs (test_gpu_batch_widths.py); the small batches keep the one fp32 pass they always had
CHUNKED = 32


@pytest.mark.parametrize("cfg,bsz,over", FULL, ids=["gbm_b3", "kirc_b3", "lgg_rsage_b3", "lgg_b3", "gbm_b40", "gbm_b32", "kirc_b64",
                                                     "lgg_b64", "gbm_b256"])
def test_multilevel_full_size_vs_oracle(mlg, cfg, bsz, over):
    """pred, pooled features, per-layer activations, feature loss, BCE loss and EVERY parameter gradient of the default
    CUDA path at N = 15 405 / G = 25 015 against oracle.multilevel_forward + feature_loss + bce_loss on the CPU."""
    from test_gpu_batch_widths import ORACLE_CHUNK, oracle_params, train_oracle
    model, args, batch, weight, sd = _multilevel_case(mlg, cfg, bsz, seed=21 + bsz, **over)
    names = [k for k, p in model.named_parameters() if p.requires_grad and not k.endswith("lin_l.weight")]
    n = 3 * mlg.MultilevelGNN.GENES
    # --- CUDA path, shipped defaults ---
    pathway_indexs = model.pathway_indexs.clone()
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    acts = {}
    hooks = [layer.register_forward_hook(lambda m, a, o, j=j: acts.__setitem__("gnn%d" % j, o.detach()))
             for j, layer in enumerate(model.gnn_model)]
    gb = batch.to(DEV)
    pred, feat = model(gb)
    for h in hooks:
        h.remove()
    fl = model.get_feature_loss(feat)
    crit = torch.nn.BCELoss(weight=weight.to(DEV)) if args.weight_balance else torch.nn.BCELoss()
    loss = crit(pred.float(), gb.y.reshape(-1, 2)) + fl
    params = dict(model.named_parameters())
    g = torch.autograd.grad(loss, [params[k] for k in names], allow_unused=True)
    tag = "%s B=%d" % (cfg, bsz)

    # --- oracle (CPU, autograd through the reference's op order), compared chunk by chunk ---
    def visit(g0, g1, pred_r, feat_r, acts_r):
        part = "%s graphs %d..%d" % (tag, g0, g1 - 1)
        _check(pred[g0:g1], pred_r, part + " pred")
        _check(feat[g0:g1], feat_r, part + " pca_feature")
        for k in ("gnn0", "gnn1"):
            _check(acts[k][g0 * n:g1 * n], acts_r[k], part + " " + k)

    chunked = bsz >= CHUNKED
    loss_r, g_r = train_oracle(oracle_params(sd, names, torch.float64 if chunked else torch.float32), names, _cpu_batch(batch),
                               args, n, pathway_indexs, weight if args.weight_balance else None,
                               chunk=ORACLE_CHUNK if chunked else bsz, dtype=torch.float64 if chunked else torch.float32,
                               visit=visit)
    fl_r = R.feature_loss(None, sd["learnable_pca_params"], sd["info_mask"], pathway_indexs, pca_loss=args.pca_loss,
                          pca_indep_loss=args.pca_indep_loss)
    _check(torch.as_tensor(fl).reshape(()), torch.as_tensor(fl_r).reshape(()), tag + " feature_loss")
    _check(loss, loss_r, tag + " loss")
    for k, a, c in zip(names, g, g_r):
        if a is None or c is None:
            assert a is None and c is None, k
            continue
        _check(a, c, tag + " g_" + k, rtol=2e-4, atol=1e-5, l2=1e-3, outliers=1e-3)


def test_genconv_100k_vs_oracle(mlg):
    """GENConv softmax aggregation + MsgNorm + learn_t + per-layer edge encoder at the cfg4 shape (N = 100 k, k = 16,
    H = 128; the ring kernel's shape) against R.genconv_forward: output and gradients w.r.t. x, the edge features and
    every parameter.  The kNN graph comes from the CUDA kNN kernel (checked on its own elsewhere)."""
    from multilevel_gnn_b200 import synth
    n, H, k = 100000, 128, 16
    pts = synth.knn_points(n, 64, seed=2)
    ei = mlg.knn_graph_matrix(pts.to(DEV), k).cpu()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(n, H, generator=g)
    ea = torch.randn(ei.shape[1], H, generator=g) * 0.5
    torch.manual_seed(7)
    conv = mlg.GENConv(H, H, aggr="softmax", learn_t=True, msg_norm=True, learn_msg_scale=True, encode_edge=True,
                       edge_feat_dim=H, norm="layer")
    # the oracle in fp64: the weight gradients are sums over 1.6 M edges / 100 k nodes, where an fp32 CPU reduction is itself only
    # good to ~1e-3 of the result (measured: half of edge_encoder.weight's entries 9e-4 of the scale apart between two fp32 orders)
    sd = {kk: v.detach().clone().double().requires_grad_() for kk, v in conv.state_dict().items()}
    xr, er = x.clone().double().requires_grad_(), ea.clone().double().requires_grad_()
    Rw = torch.randn(n, H, generator=g)
    yr = R.genconv_forward(sd, xr, ei, er, aggr="softmax", learn_t=True, msg_norm_on=True, encode_edge=True, norm="layer")
    names = list(sd)
    g_r = torch.autograd.grad((yr * Rw.double()).sum(), [xr, er] + [sd[kk] for kk in names], allow_unused=True)
    conv.to(DEV).train()
    xg, eg = x.to(DEV).requires_grad_(), ea.to(DEV).requires_grad_()
    y = conv(xg, ei.to(DEV), eg)
    params = dict(conv.named_parameters())
    gs = torch.autograd.grad((y * Rw.to(DEV)).sum(), [xg, eg] + [params[kk] for kk in names], allow_unused=True)
    _check(y, yr, "GENConv 100k y")
    _check(gs[0], g_r[0], "GENConv 100k g_x", rtol=2e-4, l2=2e-3, outliers=1e-3)
    _check(gs[1], g_r[1], "GENConv 100k g_edge_attr", rtol=2e-4, l2=2e-3, outliers=1e-3)
    for kk, a, c in zip(names, gs[2:], g_r[2:]):
        if c is None:
            continue
        # Parameter gradients here are reductions over 1.6 M edges / 100 k nodes with heavy cancellation.  The tensor-core weight
        # gradient (3xTF32, mlg_xty_tc) is accurate to ~4e-6 of sum |a||x| (tests/test_gpu_parity.py::
        # test_xty_tensor_core_matches_fp64), i.e. up to ~1e-3 of the tensor's largest entry for these sums, uniformly over the
        # entries -- so they are held to a norm-wise bound and a max-error bound relative to the tensor's scale, not element-wise
        # relative error; one flipped LayerNorm-ReLU unit additionally moves a whole row of its weight gradient by that node's full
        # contribution (O(1) against sums that only reach ~1e3 by random-sign accumulation: 4.3 of 838 measured).
        ad, cd = a.detach().cpu().double(), c.detach().cpu().double()
        scale = float(cd.abs().max())
        assert ad.shape == cd.shape
        assert float((ad - cd).abs().max()) <= 1e-2 * scale, "GENConv 100k g_%s: max abs err %.3e (scale %.3e)" % (
            kk, float((ad - cd).abs().max()), scale)
        assert _rel_l2(a, c) <= 3e-3, "GENConv 100k g_%s: relative L2 error %.3e" % (kk, _rel_l2(a, c))


def test_diffpool_tensor_core_path_vs_oracle(mlg):
    """DiffPool with every first-layer contraction on the tensor-core bf16 path (N = 4096 nodes -> 1024 clusters,
    C = 1024: M, N and K all >= dense_ops.TENSOR_CORE_MIN) against R.diffpool_forward in fp32 on the CPU: pooled features,
    link and entropy terms.  bf16 operands / fp32 accumulate: tolerance 3e-2 of the tensor's scale (the fp32 rtol 1e-4 bar
    applies to the reference-sized fp32 path, test_gpu_parity.py::test_diffpool_golden)."""
    from multilevel_gnn_b200 import _cabi, configs
    b, n, c = 2, 4096, 1024
    g = torch.Generator().manual_seed(9)
    x = torch.randn(b, n, c, generator=g)
    a = torch.rand(n, n, generator=g)
    adj = (a + a.t()) * 0.5 + torch.eye(n)
    torch.manual_seed(4)
    dp = mlg.DiffPool(c, 2, n, 2, 1024, 1024, configs.make_args("lgg"))
    sd = {k: v.detach().clone() for k, v in dp.state_dict().items()}
    out_r, l_r, e_r = R.diffpool_forward(sd, x, adj)
    dp.to(DEV).eval()
    timer = _cabi.KernelTimer()
    _cabi.TIMER = timer
    try:
        with torch.no_grad():
            out, l, e = dp(x.to(DEV), adj.to(DEV))
        tags = timer.summary()
    finally:
        _cabi.TIMER = None
    assert tags.get("gemm_bf16", {}).get("launches", 0) >= 5, tags      # A.X (x2), S^T.X, S^T.A, (S^T.A).S, S.S^T
    assert out.shape == out_r.shape
    assert_close(out, out_r, rtol=3e-2, atol=3e-2, what="DiffPool tensor-core out")
    assert _rel_l2(out, out_r) <= 3e-2
    assert_close(torch.as_tensor(l).reshape(()), torch.as_tensor(l_r).reshape(()), rtol=3e-2, atol=1e-4, what="DiffPool link")
    assert_close(torch.as_tensor(e).reshape(()), torch.as_tensor(e_r).reshape(()), rtol=3e-2, atol=1e-3, what="DiffPool entropy")
