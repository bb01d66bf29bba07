"""Parity of the sm_100a kernels (through the C ABI and the drop-in modules) against
 (a) the committed golden vectors produced by the reference's own files, and
 (b) the CPU oracle (oracle/restated.py) on seeded inputs, at sizes the oracle finishes in seconds.
Tolerance: fp32 rtol 1e-4 (BASELINE.json north_star); kNN indices exact outside fp32 tie classes.
"""
import pytest
import torch

from conftest import as_batch, assert_close, assert_close_flips, load_golden
from oracle import restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def mlg():
    import multilevel_gnn_b200 as m
    m._cabi.lib()      # fail loudly if the native library is missing
    return m


def _load(module, sd):
    module.load_state_dict(sd, strict=True)
    return module.to(DEV)


# ------------------------------------------------------------------------------------------------
# GENConv (all aggregation modes) vs golden
# ------------------------------------------------------------------------------------------------
GEN = load_golden("genconv")


@pytest.mark.parametrize("name", sorted(GEN))
def test_genconv_golden(mlg, name):
    c = GEN[name]
    H = c["H"]
    conv = _load(mlg.GENConv(H, H, encode_edge=True, edge_feat_dim=H, **c["kw"]), c["state_dict"])
    conv.train()
    x = c["x"].to(DEV).requires_grad_()
    ea = c["edge_attr"].to(DEV).requires_grad_()
    ei = c["edge_index"].to(DEV)
    y = conv(x, ei, ea)
    assert_close(y, c["y"], what=name + ".y")
    names = list(c["g_params"])
    params = dict(conv.named_parameters())
    gs = torch.autograd.grad((y * c["R"].to(DEV)).sum(), [x, ea] + [params[k] for k in names], allow_unused=True)
    assert_close(gs[0], c["g_x"], what=name + ".g_x")
    assert_close(gs[1], c["g_edge_attr"], what=name + ".g_edge_attr")
    for k, g in zip(names, gs[2:]):
        assert_close(g, c["g_params"][k], rtol=2e-4, what=name + ".g_" + k)


@pytest.mark.parametrize("name", sorted(GEN))
def test_gen_aggregate_golden(mlg, name):
    """GenMessagePassing.aggregate(inputs, index, dim_size) on explicit messages."""
    c = GEN[name]
    H = c["H"]
    conv = _load(mlg.GENConv(H, H, encode_edge=True, edge_feat_dim=H, **c["kw"]), c["state_dict"])
    msg = c["msg"].to(DEV).requires_grad_()
    agg = conv.aggregate(msg * 1.0, c["edge_index"][1].to(DEV), dim_size=c["x"].shape[0])
    assert_close(agg, c["agg"], what=name + ".agg")
    g = torch.autograd.grad((agg * c["R"].to(DEV)).sum(), msg)[0]
    assert_close(g, c["g_msg"], what=name + ".g_msg")


PWC = load_golden("pathwayconv")


@pytest.mark.parametrize("name", sorted(PWC))
def test_pathwayconv_golden(mlg, name):
    """PathwayConv (torch_vertex.py:107-178; SURVEY section 8 row f4): transform-first message + the aggregation kernel on
    explicit messages, against the reference's own class."""
    c = PWC[name]
    H = c["H"]
    conv = _load(mlg.PathwayConv(H, H, **c["kw"]), c["state_dict"])
    conv.train()
    x = c["x"].to(DEV).requires_grad_()
    ea = c["edge_attr"].to(DEV).requires_grad_()
    mask = None if c["mask"] is None else c["mask"].to(DEV)
    y = conv(x, c["edge_index"].to(DEV), ea, mask)
    assert_close(y, c["y"], what=name + ".y")
    names = [k for k, g in c["g_params"].items() if g is not None]
    params = dict(conv.named_parameters())
    gs = torch.autograd.grad((y * c["R"].to(DEV)).sum(), [x, ea] + [params[k] for k in names], allow_unused=True)
    assert_close(gs[0], c["g_x"], rtol=2e-4, what=name + ".g_x")
    assert_close(gs[1], c["g_edge_attr"], rtol=2e-4, what=name + ".g_edge_attr")
    for k, g in zip(names, gs[2:]):
        assert_close(g, c["g_params"][k], rtol=2e-4, what=name + ".g_" + k)


def test_pathwayconv_tall_vs_oracle(mlg):
    """PathwayConv with enough nodes for the tensor-core (3xTF32) transform-first GEMM: forward and input gradient against
    the oracle's direct outer-product formulation."""
    from conftest import assert_close_flips
    n, e, H = 70000, 280000, 32
    g = torch.Generator().manual_seed(11)
    x = torch.randn(n, H, generator=g)
    ea = torch.randn(e, 2, generator=g)
    ei = torch.stack([torch.randint(0, n, (e,), generator=g), torch.randint(0, n, (e,), generator=g)])
    torch.manual_seed(12)
    conv = mlg.PathwayConv(H, H, aggr="softmax", t=0.9, learn_t=True, norm="layer")
    sd = {k: v.detach().clone() for k, v in conv.state_dict().items()}
    xr = x.clone().requires_grad_()
    yr = R.pathway_conv_forward(sd, xr, ei, ea, aggr="softmax", learn_t=True, norm="layer")
    Rw = torch.randn(n, H, generator=g)
    gr = torch.autograd.grad((yr * Rw).sum(), xr)[0]
    conv.to(DEV).train()
    xg = x.to(DEV).requires_grad_()
    y = conv(xg, ei.to(DEV), ea.to(DEV))
    assert_close(y, yr, what="pathwayconv tall y")
    gx = torch.autograd.grad((y * Rw.to(DEV)).sum(), xg)[0]
    assert_close_flips(gx, gr, "pathwayconv tall g_x", rtol=2e-4, l2=1e-3, outliers=1e-3)


# ------------------------------------------------------------------------------------------------
# SAGE / RSAGE vs golden
# ------------------------------------------------------------------------------------------------
SAGE = load_golden("sage")


@pytest.mark.parametrize("name", sorted(SAGE))
def test_sage_golden(mlg, name):
    c = SAGE[name]
    conv = _load(mlg.GraphConv(c["cin"], c["cout"], conv=c["conv"], act="leakyrelu", norm=None, mlp_norm="none"),
                 c["state_dict"])
    x = c["x"].to(DEV).requires_grad_()
    y = conv(x, c["edge_index"].to(DEV), c["edge_attr"].to(DEV))
    assert_close(y, c["y"], what=name + ".y")
    names = [k for k, g in c["g_params"].items() if g is not None]
    params = dict(conv.named_parameters())
    gs = torch.autograd.grad((y * c["R"].to(DEV)).sum(), [x] + [params[k] for k in names])
    assert_close(gs[0], c["g_x"], what=name + ".g_x")
    for k, g in zip(names, gs[1:]):
        assert_close(g, c["g_params"][k], what=name + ".g_" + k)
    assert c["g_params"]["gconv.lin_l.weight"] is None and params["gconv.lin_l.weight"].grad is None


# ------------------------------------------------------------------------------------------------
# kNN vs golden: identical indices wherever the fp64 distances separate the ranks
# ------------------------------------------------------------------------------------------------
KNN = load_golden("knn")


def _check_knn(x, batch, k, got, ref, name):
    """got/ref: [2, B*N*k].  Centres must match exactly; neighbour ids must match wherever the
    neighbour's distance is separated from the adjacent ranks by more than the fp32 evaluation error;
    inside a near-tie class any permutation is accepted but the distances must agree."""
    assert torch.equal(got[1].cpu(), ref[1]), name + ": centre ids"
    vals, _, d = R.knn_distance_gap(x, k, batch)          # fp64
    bsz = 1 if batch is None else int(batch[-1]) + 1
    n = x.shape[0] // bsz
    g, r = got[0].cpu().view(bsz, n, k), ref[0].view(bsz, n, k)
    offs = (torch.arange(bsz) * n).view(bsz, 1, 1)
    dg = torch.gather(d, 2, g - offs)
    dr = torch.gather(d, 2, r - offs)
    scale = d.abs().max()
    assert float((dg - dr).abs().max()) <= 1e-5 * float(scale), name + ": neighbour distances differ"
    gap_next = (vals[..., 1:k + 1] - vals[..., :k]) if vals.shape[-1] > k else None
    sep = torch.ones_like(dg, dtype=torch.bool)
    tol = 4e-6 * float(scale)
    sep[..., 1:] &= (vals[..., 1:k] - vals[..., :k - 1]) > tol
    if gap_next is not None:
        sep &= gap_next > tol
    assert torch.equal(g[sep], r[sep]), name + ": ids differ outside tie classes"
    # every row: k distinct neighbours
    assert int((torch.sort(g, -1).values.diff(dim=-1) == 0).sum()) == 0


@pytest.mark.parametrize("name", sorted(KNN))
def test_knn_golden(mlg, name):
    c = KNN[name]
    x, batch = c["x"].to(DEV), c["batch"].to(DEV)
    kk = c["k"] * c["dil"]
    full = mlg.knn_graph_matrix(x, kk, batch if c["b"] > 1 else None)
    _check_knn(c["x"], c["batch"] if c["b"] > 1 else None, kk, full, c["edge_index_full"], name)
    if name == "grid_ties":
        # canonical order inside exact ties: ascending distance, then ascending index
        d = R.pairwise_distance(c["x"].view(1, -1, 2))[0]
        g = full[0].cpu().view(-1, kk)
        dsel = torch.gather(d, 1, g)
        assert bool((dsel.diff(dim=1) >= 0).all())
        same = dsel.diff(dim=1) == 0
        assert bool((g.diff(dim=1)[same] > 0).all())
        return
    dil = mlg.DilatedKnnGraph(c["k"], c["dil"]).eval()(x, batch)
    assert torch.equal(dil.cpu(), full.cpu().view(2, -1, kk)[:, :, ::c["dil"]].reshape(2, -1))
    xd = c["x"].view(c["b"], c["n"], c["d"]).transpose(1, 2).unsqueeze(-1).contiguous().to(DEV)
    dense = mlg.dense_knn_matrix(xd, kk)
    assert dense.shape == c["dense_full"].shape
    offs = (torch.arange(c["b"]) * c["n"]).view(1, c["b"], 1, 1)
    assert torch.equal((dense.cpu() + offs).reshape(2, -1), full.cpu())
    dd = mlg.DenseDilatedKnnGraph(c["k"], c["dil"])(xd)
    assert torch.equal(dd.cpu(), dense.cpu()[:, :, :, ::c["dil"]])


def test_knn_vs_oracle_larger(mlg):
    g = torch.Generator().manual_seed(7)
    x = torch.randn(3 * 700, 24, generator=g)
    batch = torch.arange(3).repeat_interleave(700)
    ref = R.knn_graph_matrix(x, 16, batch)
    got = mlg.knn_graph_matrix(x.to(DEV), 16, batch.to(DEV))
    _check_knn(x, batch, 16, got, ref, "n700")


# ------------------------------------------------------------------------------------------------
# MultilevelGNN (small re-sized instance) vs golden: pred, pooled features, per-layer activations,
# loss, every gradient
# ------------------------------------------------------------------------------------------------
ML = load_golden("multilevel")


def _build_multilevel(mlg, c):
    args = mlg.configs.make_args(c["config"], **c["overrides"])
    model = mlg.MultilevelGNN(args)
    model.node_num = c["genes"]
    sd = c["state_dict"]
    model.node_embedding = torch.nn.Parameter(sd["node_embedding"].clone())
    model.learnable_pca_params = torch.nn.Parameter(sd["learnable_pca_params"].clone())
    model.set_info_mask(sd["info_mask"].clone())
    model.load_state_dict(sd, strict=True)
    model.set_pathway_indexs(c["batch"]["raw_indice"][0].clone())
    return model.to(DEV), args


@pytest.mark.parametrize("name", sorted(ML))
def test_multilevel_golden(mlg, name):
    c = ML[name]
    model, args = _build_multilevel(mlg, c)
    model.eval()
    acts = {}
    hooks = [layer.register_forward_hook(lambda m, a, o, j=j: acts.__setitem__("gnn%d" % j, o.detach()))
             for j, layer in enumerate(model.gnn_model)]
    batch = as_batch(c["batch"], DEV)
    pred, feat = model(batch)
    for h in hooks:
        h.remove()
    assert_close(pred, c["pred"], what=name + ".pred")
    assert_close(feat, c["pca_feature"], what=name + ".pca_feature")
    for k, v in c["acts"].items():
        assert_close(acts[k], v, what=name + "." + k)
    fl = model.get_feature_loss(feat)
    assert_close(torch.as_tensor(fl), c["feature_loss"], what=name + ".feature_loss")
    loss = torch.nn.BCELoss(weight=c["weight"].to(DEV))(pred.float(), batch.y.reshape(-1, 2)) + fl
    assert_close(loss, c["loss"], what=name + ".loss")
    loss.backward()
    for k, p in model.named_parameters():
        if not p.requires_grad:
            continue
        if c["grads"][k] is None:
            assert p.grad is None, k
        else:
            assert_close(p.grad, c["grads"][k], rtol=2e-4, what=name + ".g_" + k)


# ------------------------------------------------------------------------------------------------
# DeeperGCN vs golden
# ------------------------------------------------------------------------------------------------
DG = load_golden("deepergcn")


@pytest.mark.parametrize("affine", [True, False], ids=["affine_edge", "edge_gemm"])
@pytest.mark.parametrize("name", sorted(DG))
def test_deepergcn_golden(mlg, name, affine):
    """Both edge paths against the reference's outputs: the factored scalar-edge term (functional.AffineEdge, no [E, H]
    tensor) and the literal per-layer edge GEMM."""
    c = DG[name]
    args = mlg.configs.make_args(None, **c["overrides"])
    model = _load(mlg.DeeperGCN(args), c["state_dict"])
    model.AFFINE_EDGE = affine
    model.train()
    batch = as_batch(c["batch"], DEV)
    batch.node_size = c["batch"]["node_size"]          # host tensor: no device sync needed
    pred = model(batch)
    assert_close(pred, c["pred"], what=name + ".pred")
    (pred * c["R"].to(DEV)).sum().backward()
    for k, p in model.named_parameters():
        if c["grads"].get(k) is None:
            continue
        assert_close(p.grad, c["grads"][k], rtol=5e-4, atol=2e-5, what=name + ".g_" + k)


@pytest.mark.parametrize("aggr,H,epi", [("softmax", 128, "msgnorm"), ("softmax", 256, "residual"), ("softmax_sg", 64, "msgnorm"),
                                        ("power", 32, "msgnorm"), ("softmax_sum", 96, "residual"), ("power_sum", 128, "msgnorm"),
                                        ("add", 128, "residual"), ("mean", 48, "msgnorm"), ("max", 128, "residual")])
def test_gen_aggregate_affine_vs_materialized(mlg, aggr, H, epi):
    """mlg_gen_aggr_{fwd,bwd}_affine + mlg_wcolsum (edge term a_e * p + q rebuilt in registers) against the [E, H] path on
    the same numbers: output, g_x, g_p, g_q, g_a and the learnable scalars."""
    Fn = mlg.functional
    n, e = 2500, 30000
    ei, g = _rand_graph(n, e, 23)
    topo = mlg.graph.topology(ei.to(DEV), n)
    x0 = torch.randn(n, H, generator=g).to(DEV)
    a0 = torch.rand(e, generator=g).to(DEV)
    p0, q0 = torch.randn(H, generator=g).to(DEV), (0.3 * torch.randn(H, generator=g)).to(DEV)
    Rm = torch.randn(n, H, generator=g).to(DEV)
    learn = True
    outs = []
    for affine in (True, False):
        x, a, p, q = (v.clone().requires_grad_() for v in (x0, a0, p0, q0))
        t = torch.tensor([0.9], device=DEV, requires_grad=True)
        pw = torch.tensor([2.0], device=DEV, requires_grad=True)
        y = torch.tensor([0.1], device=DEV, requires_grad=True) if aggr.endswith("_sum") else None
        sc = torch.tensor([1.3], device=DEV, requires_grad=True) if epi == "msgnorm" else None
        code = Fn.EPI_MSGNORM if epi == "msgnorm" else Fn.EPI_RESIDUAL
        if affine:
            h = Fn.GenAggregateAffine.apply(x, a, p, q, t, pw, y, sc, topo, aggr, 1e-7, code, learn)
        else:
            h = Fn.GenAggregate.apply(x, Fn.AffineEdge(a, p, q).materialize(), t, pw, y, sc, topo, aggr, 1e-7, code, learn)
        leaves = [x, a, p, q] + [v for v in (t, pw, y, sc) if v is not None]
        gs = torch.autograd.grad((h * Rm).sum(), leaves, allow_unused=True)
        outs.append((h, gs))
    (ha, ga), (hm, gm) = outs
    assert_close(ha, hm, what="h")
    for i, (u, v) in enumerate(zip(ga, gm)):
        assert (u is None) == (v is None), i
        if u is not None:
            assert_close(u, v, rtol=2e-4, atol=1e-5 * max(1.0, float(v.abs().max())), what="grad[%d]" % i)


@pytest.mark.parametrize("H,epi,affine,edge_grad", [(128, "msgnorm", False, True), (128, "msgnorm", False, False),
                                                    (256, "residual", False, True), (128, "msgnorm", True, False),
                                                    (256, "residual", True, False), (128, "residual", True, True)])
def test_gen_backward_source_sum_in_kernel(mlg, H, epi, affine, edge_grad):
    """mlg_gen_aggr_bwd_src / _affine_src (the source-side sum as vector reductions inside the backward kernel; default) vs
    the two-pass fixed-order path (mlg_gen_aggr_bwd + mlg_gather_sum) on the same inputs -- hub sources with thousands of
    out-edges, rows without in-edges, edge gradients wanted or not: every gradient within fp32 summation-order noise."""
    Fn = mlg.functional
    n, e = 3000, 48000
    ei, g = _rand_graph(n, e, 31)
    ei[0, :5000] = 7                       # hub: node 7 is the source of 5000 edges
    ei[1, ei[1] == 11] = 12                # node 11 has no in-edges
    topo = mlg.graph.topology(ei.to(DEV), n)
    x0 = torch.randn(n, H, generator=g).to(DEV)
    a0 = torch.rand(e, generator=g).to(DEV)
    p0, q0 = torch.randn(H, generator=g).to(DEV), (0.3 * torch.randn(H, generator=g)).to(DEV)
    e0 = torch.randn(e, H, generator=g).to(DEV)
    Rm = torch.randn(n, H, generator=g).to(DEV)
    code = Fn.EPI_MSGNORM if epi == "msgnorm" else Fn.EPI_RESIDUAL
    outs = []
    old = Fn.GEN_BWD_SRC_ATOMIC
    try:
        for atomic in (True, False):
            Fn.GEN_BWD_SRC_ATOMIC = atomic
            x, a, pp, q, ee = (v.clone().requires_grad_() for v in (x0, a0, p0, q0, e0))
            t = torch.tensor([0.9], device=DEV, requires_grad=True)
            sc = torch.tensor([1.3], device=DEV, requires_grad=True) if epi == "msgnorm" else None
            if affine:
                h = Fn.GenAggregateAffine.apply(x, a, pp, q, t, 1.0, None, sc, topo, "softmax", 1e-7, code, True)
                leaves = [x, pp, q, t] + ([a] if edge_grad else [])
            else:
                h = Fn.GenAggregate.apply(x, ee, t, 1.0, None, sc, topo, "softmax", 1e-7, code, True)
                leaves = [x, t] + ([ee] if edge_grad else [])
            if sc is not None:
                leaves.append(sc)
            outs.append(torch.autograd.grad((h * Rm).sum(), leaves))
    finally:
        Fn.GEN_BWD_SRC_ATOMIC = old
    for i, (u, v) in enumerate(zip(*outs)):
        assert_close(u, v, rtol=1e-4, atol=2e-6 * max(1.0, float(v.abs().max())), what="grad[%d]" % i)


@pytest.mark.parametrize("C", [128, 64, 32, 20, 256])
def test_gather_sum_hub_rows(mlg, C):
    """Rows far longer than the mean (hubs of a by-source kNN CSR) are walked by the whole block: same sums as a
    float64 index_add, with weights / mean post-scale / addend, for every lane-group width."""
    Fn = mlg.functional
    g = torch.Generator().manual_seed(5 + C)
    n, n_src = 700, 5000
    deg = torch.randint(0, 12, (n,), generator=g)
    deg[[3, 77, 78, 300, 699]] = torch.tensor([1502, 97, 96, 640, 2049])
    rowptr = torch.zeros(n + 1, dtype=torch.int64)
    rowptr[1:] = deg.cumsum(0)
    nnz = int(rowptr[-1])
    idx = torch.randint(0, n_src, (nnz,), generator=g)
    val = torch.rand(nnz, generator=g)
    src = torch.randn(n_src, C, generator=g)
    add = torch.randn(n, C, generator=g)
    rows = torch.arange(n).repeat_interleave(deg)
    ref = torch.zeros(n, C, dtype=torch.float64).index_add_(0, rows, src[idx].double() * val.double()[:, None])
    ref = ref / deg.clamp(min=1).double()[:, None] + add.double()
    out = Fn.gather_sum(src.to(DEV), rowptr.to(torch.int32).to(DEV), idx.to(torch.int32).to(DEV), n, val=val.to(DEV),
                        post_mode=1, addend=add.to(DEV))
    assert_close(out, ref.float(), rtol=1e-4, atol=1e-5, what="hub gather_sum C=%d" % C)
    out2 = Fn.gather_sum(src.to(DEV), rowptr.to(torch.int32).to(DEV), idx.to(torch.int32).to(DEV), n, val=val.to(DEV),
                         post_mode=1, addend=add.to(DEV))
    assert torch.equal(out, out2), "hub rows must be summed in a fixed order"


def test_wcolsum(mlg):
    L, cabi = mlg._cabi.lib(), mlg._cabi
    for rows, C in ((1, 4), (777, 128), (50001, 64), (4099, 1024)):
        g = torch.Generator().manual_seed(rows)
        G = torch.randn(rows, C, generator=g).to(DEV)
        a = torch.rand(rows, generator=g).to(DEV)
        u, v = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
        nb = L.mlg_wcolsum_workspace_bytes(rows, C)
        ws = torch.empty(nb // 4, device=DEV)
        cabi.check(L.mlg_wcolsum(cabi.fptr(G), C, cabi.fptr(a), rows, C, cabi.fptr(u), cabi.fptr(v), cabi.fptr(ws), nb,
                                 cabi.stream_ptr()), "mlg_wcolsum")
        Gd = G.double()
        assert_close(u, (a.double() @ Gd).float(), rtol=1e-4, atol=1e-4, what="u")
        assert_close(v, Gd.sum(0).float(), rtol=1e-4, atol=1e-4, what="v")


# ------------------------------------------------------------------------------------------------
# seeded larger cases vs the CPU oracle + size-independent properties
# ------------------------------------------------------------------------------------------------
def _rand_graph(n, e, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randint(0, n, (e,), generator=g), torch.randint(0, n - 5, (e,), generator=g)]), g


@pytest.mark.parametrize("aggr,H", [("softmax", 128), ("softmax", 64), ("softmax", 256), ("power", 32), ("softmax_sum", 96)])
def test_gen_aggr_vs_oracle(mlg, aggr, H):
    n, e = 3000, 40000
    ei, g = _rand_graph(n, e, 11)
    x = torch.randn(n, H, generator=g)
    ea = torch.randn(e, H, generator=g)
    kw = dict(aggr=aggr, t=0.9, learn_t=True, p=2.0, learn_p=True, y=0.1, learn_y=True, msg_norm=True, norm="layer",
              mlp_layers=1)
    torch.manual_seed(1)
    conv = mlg.GENConv(H, H, encode_edge=False, **kw).to(DEV).train()
    sd = {k: v.detach().cpu().clone().requires_grad_() for k, v in conv.state_dict().items()}
    xr, er = x.clone().requires_grad_(), ea.clone().requires_grad_()
    yr = R.genconv_forward(sd, xr, ei, er, aggr=aggr, t=0.9, learn_t=True, p=2.0, learn_p=True, msg_norm_on=True,
                           encode_edge=False, norm="layer")
    Rm = torch.randn(n, H, generator=g)
    gr = torch.autograd.grad((yr * Rm).sum(), [xr, er])
    xg, eg = x.to(DEV).requires_grad_(), ea.to(DEV).requires_grad_()
    yg = conv(xg, ei.to(DEV), eg)
    assert_close(yg, yr, what="y")
    gg = torch.autograd.grad((yg * Rm.to(DEV)).sum(), [xg, eg])
    assert_close(gg[0], gr[0], rtol=2e-4, what="g_x")
    assert_close(gg[1], gr[1], rtol=2e-4, what="g_e")


def test_gen_aggr_properties(mlg):
    """zero in-degree rows -> 0 (softmax) ; permutation of the edge list leaves the result unchanged
    up to fp32 summation order; softmax weights sum to one (aggregating a constant returns it)."""
    n, e, H = 500, 6000, 128
    ei, g = _rand_graph(n, e, 5)
    conv = mlg.GenMessagePassing(aggr="softmax", t=1.0).to(DEV)
    msg = torch.rand(e, H, generator=g).to(DEV)
    out = conv.aggregate(msg, ei[1].to(DEV), dim_size=n)
    assert float(out[n - 5:].abs().max()) == 0.0
    perm = torch.randperm(e, generator=g)
    out_p = conv.aggregate(msg[perm.to(DEV)], ei[1][perm].to(DEV), dim_size=n)
    assert_close(out_p, out.cpu(), what="permutation invariance")
    const = torch.full((e, H), 0.37, device=DEV)
    outc = conv.aggregate(const, ei[1].to(DEV), dim_size=n)
    deg = torch.bincount(ei[1], minlength=n)
    assert_close(outc[deg > 0], torch.full((int((deg > 0).sum()), H), 0.37), what="weights sum to one")
    pw = mlg.GenMessagePassing(aggr="power", p=2.0).to(DEV)
    outp = pw.aggregate(msg, ei[1].to(DEV), dim_size=n)
    assert_close(outp[n - 5:], torch.full((5, H), (1e-7) ** 0.5), what="power-mean of empty rows (SURVEY B.2)")


def test_sage_vs_oracle_gbm_like(mlg):
    from multilevel_gnn_b200 import synth
    genes, bsz = 400, 3
    b = synth.multilevel_batch(batch_size=bsz, genes=genes, slots=900, intra_edges=6000, seed=2)
    n = 3 * genes * bsz
    g = torch.Generator().manual_seed(3)
    x = torch.randn(n, 64, generator=g)
    torch.manual_seed(2)
    conv = mlg.GraphConv(64, 32, conv="sage", act="leakyrelu", mlp_norm="none").to(DEV)
    sd = {k: v.detach().cpu().clone().requires_grad_() for k, v in conv.state_dict().items()}
    xr = x.clone().requires_grad_()
    yr = R.sage_forward(sd, xr, b.edge_index, b.edge_attr)
    Rm = torch.randn(n, 32, generator=g)
    gr = torch.autograd.grad((yr * Rm).sum(), [xr, sd["gconv.lin_r.weight"], sd["gconv.nn.0.weight"]])
    xg = x.to(DEV).requires_grad_()
    yg = conv(xg, b.edge_index.to(DEV), b.edge_attr.to(DEV))
    assert_close(yg, yr, what="y")
    (yg * Rm.to(DEV)).sum().backward()
    assert_close(xg.grad, gr[0], rtol=2e-4, what="g_x")
    assert_close(conv.gconv.lin_r.weight.grad, gr[1], rtol=2e-4, what="g_lin_r")
    assert_close(conv.gconv.nn[0].weight.grad, gr[2], rtol=2e-4, what="g_nn")


def test_pool_linearity_and_oracle(mlg):
    """pool(a*x1 + b*x2) == a*pool(x1) + b*pool(x2); and equality with the oracle incl. -1 slots."""
    from multilevel_gnn_b200 import functional as Fn, graph, synth
    genes, bsz, slots, C, P = 300, 4, 2000, 32, 3
    b = synth.multilevel_batch(batch_size=bsz, genes=genes, slots=slots, intra_edges=100, seed=9)
    n = 3 * genes
    g = torch.Generator().manual_seed(4)
    x1, x2 = torch.randn(bsz * n, C, generator=g), torch.randn(bsz * n, C, generator=g)
    w = torch.randn(slots, P, generator=g)
    mask = (torch.rand(slots, 1, generator=g) < 0.5).float()
    lay = graph.pool_layout(b.gene_pca_match.to(DEV), b.raw_indice.to(DEV), n, 438)
    wm = (w * mask).to(DEV)
    f = lambda t: Fn.PathwayPool.apply(t.to(DEV), wm, None, lay)
    assert_close(f(2.0 * x1 - 0.5 * x2), (2.0 * f(x1) - 0.5 * f(x2)).cpu(), what="linearity")
    ref = R.multilevel_pool(x1, b.gene_pca_match, b.raw_indice, w, mask, n, 438)
    assert_close(f(x1).reshape(ref.shape), ref, what="pool vs oracle")
    # wrap_negative (pca_match_mask False): python negative indexing of the reference
    lay_w = graph.pool_layout(b.gene_pca_match.to(DEV).clone(), b.raw_indice.to(DEV), n, 438, wrap_negative=True)
    ref_w = R.multilevel_pool(x1, b.gene_pca_match, b.raw_indice, w, mask, n, 438, match_mask=False)
    got_w = Fn.PathwayPool.apply(x1.to(DEV), wm, None, lay_w)
    assert_close(got_w.reshape(ref_w.shape), ref_w, what="pool wrap_negative")


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("bsz", [3, 8, 13, 32, 64, 256])
def test_pool_c32_lane_group_kernels(mlg, P, bsz):
    """C == 32 pool kernels (8-lane groups on 128-bit lanes, mlg_pool_fwd / mlg_pool_bwd): forward and both gradients
    against autograd of the oracle's gather / scatter formula (models/multilevel_gnn.py:212-239), with the value mask, for
    every packed-butterfly width (P -> 1, 2, 4, 8 values per group) and replica counts that leave idle lane groups (3),
    fill one warp exactly (8), end in a partial chunk (13), and the benchmarked widths (32, 64, 256: 4, 8 and 32 warps of
    8 replicas, workspace [ceil(B / 8), G, P], pool.cu:675-681)."""
    from multilevel_gnn_b200 import functional as Fn, graph, synth
    genes, slots, C = 200, 1500, 32
    b = synth.multilevel_batch(batch_size=bsz, genes=genes, slots=slots, intra_edges=100, seed=21)
    n = 3 * genes
    g = torch.Generator().manual_seed(5 + P)
    x = torch.randn(bsz * n, C, generator=g)
    vm = torch.randn(bsz * n, generator=g)
    w = torch.randn(slots, P, generator=g)
    mask = (torch.rand(slots, 1, generator=g) < 0.5).float()
    gout = torch.randn(bsz, C, 438, P, generator=g)
    lay = graph.pool_layout(b.gene_pca_match.to(DEV), b.raw_indice.to(DEV), n, 438)
    assert lay.replicas == bsz      # one match / segment table for all graphs: the replicated kernels run
    xd, wd = x.to(DEV).requires_grad_(True), w.to(DEV).requires_grad_(True)
    out = Fn.PathwayPool.apply(xd, wd, vm.to(DEV), lay, None, mask.to(DEV))
    out.backward(gout.to(DEV))
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ref = R.multilevel_pool(xr * vm[:, None], b.gene_pca_match, b.raw_indice, wr, mask, n, 438)
    ref.backward(gout.reshape(ref.shape))
    assert_close(out.reshape(ref.shape), ref, what="pool C=32 forward P=%d B=%d" % (P, bsz))
    assert_close(xd.grad, xr.grad, what="pool C=32 dX P=%d B=%d" % (P, bsz))
    assert_close(wd.grad, wr.grad, what="pool C=32 dW P=%d B=%d" % (P, bsz))


@pytest.mark.gpu
@pytest.mark.parametrize("cout,cin,r,bias", [(64, 64, 64, True), (32, 64, 64, True), (32, 64, 48, False)])
def test_sage_fold_stacked(mlg, cout, cin, r, bias):
    """mlg_sage_fold_stacked_fwd / _bwd (torch_vertex.py:279-291 with lin_r commuted past the mean): Wst = [W1 ; W2 W_r], the
    3xTF32 splits (hi keeps the top 19 bits, hi + lo == w exactly), the split of Wst^T, the bias [b | 0]; backward against
    autograd of the same expression, with the gradient given as one tensor and as the sum of two strided blocks."""
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()
    g = torch.Generator().manual_seed(cout + r)
    nn_w = torch.randn(cout, cin + r, generator=g).to(DEV)
    w_r = torch.randn(r, cin, generator=g).to(DEV)
    nn_b = torch.randn(cout, generator=g).to(DEV) if bias else None
    bufs = [torch.empty(2 * cout, cin, device=DEV) for _ in range(3)] + [torch.empty(cin, 2 * cout, device=DEV) for _ in range(2)]
    bias2 = torch.full((2 * cout,), 7.0, device=DEV)
    with torch.cuda.device(DEV):
        _cabi.check(L.mlg_sage_fold_stacked_fwd(_cabi.fptr(nn_w), _cabi.fptr(w_r), None if nn_b is None else _cabi.fptr(nn_b),
                                                cout, cin, r, *[_cabi.fptr(t) for t in bufs], _cabi.fptr(bias2),
                                                _cabi.stream_ptr()), "fold_stacked_fwd")
    wst, hi, lo, t_hi, t_lo = bufs
    nn_ref, wr_ref = nn_w.double().cpu().requires_grad_(True), w_r.double().cpu().requires_grad_(True)
    ref = torch.cat([nn_ref[:, :cin], nn_ref[:, cin:] @ wr_ref], 0)
    assert_close(wst, ref.detach().float(), rtol=1e-5, atol=1e-6, what="Wst")
    assert torch.equal(hi + lo, wst) and torch.equal(hi.view(torch.int32) & 0x1FFF, torch.zeros_like(hi, dtype=torch.int32))
    assert torch.equal(t_hi, hi.t().contiguous()) and torch.equal(t_lo, lo.t().contiguous())
    want_b = torch.cat([nn_b if bias else torch.zeros(cout, device=DEV), torch.zeros(cout, device=DEV)])
    assert torch.equal(bias2, want_b)
    gw = torch.randn(2 * cout, cin, generator=g)
    ref.backward(gw.double())
    for split in (False, True):
        g_nn, g_wr = torch.empty_like(nn_w), torch.empty_like(w_r)
        if split:     # the gradient as the sum of two blocks of a wider buffer (leading dimension 2 * cin)
            wide = torch.randn(4 * cout, 2 * cin, generator=g).to(DEV)
            part = torch.randn(2 * cout, cin, generator=g).to(DEV)
            wide[:2 * cout, :cin] = part
            wide[2 * cout:, cin:] = gw.to(DEV) - part
            a, bptr, ld = _cabi.fptr(wide), ctypes_ptr(wide[2 * cout:, cin:]), 2 * cin
        else:
            gd = gw.to(DEV)
            a, bptr, ld = _cabi.fptr(gd), None, cin
        with torch.cuda.device(DEV):
            _cabi.check(L.mlg_sage_fold_stacked_bwd(a, bptr, ld, _cabi.fptr(nn_w), _cabi.fptr(w_r), cout, cin, r,
                                                    _cabi.fptr(g_nn), _cabi.fptr(g_wr), _cabi.stream_ptr()), "fold_stacked_bwd")
        assert_close(g_nn, nn_ref.grad.float(), rtol=2e-5, atol=2e-6, what="g_nn_w split=%s" % split)
        assert_close(g_wr, wr_ref.grad.float(), rtol=2e-5, atol=2e-6, what="g_lin_r_w split=%s" % split)


def ctypes_ptr(t):
    import ctypes
    return ctypes.c_void_p(t.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("bsz", [3, 16, 17, 40, 64, 256])
def test_node_major_gradient_between_pool_and_aggregation(mlg, bsz):
    """mlg_pool_bwd_layout(gx_node_major=1) writes the same gradient as mlg_pool_bwd, at row i * B + b instead of b * N + i,
    and mlg_gather_sum_nm on it equals mlg_gather_sum on the graph-major tensor (backward aggregation of the transform-first
    layer, torch_vertex.py:279-286 on the by-source CSR; self rows copied alongside): bit-identical, the FMA order is the same."""
    from multilevel_gnn_b200 import _cabi, functional as Fn, graph, synth
    L = _cabi.lib()
    genes, slots, C, P = 150, 1200, 32, 2
    b = synth.multilevel_batch(batch_size=bsz, genes=genes, slots=slots, intra_edges=900, seed=31)
    n = 3 * genes
    g = torch.Generator().manual_seed(7)
    x = torch.randn(bsz * n, C, generator=g).to(DEV)
    w = torch.randn(slots, P, generator=g).to(DEV)
    gout = torch.randn(bsz, 438, P, C, generator=g).to(DEV)
    lay = graph.pool_layout(b.gene_pca_match.to(DEV), b.raw_indice.to(DEV), n, 438)
    node = lay.node_csr
    outs = []
    for nm in (0, 1):
        gx, gw = torch.empty_like(x), torch.empty_like(w)
        ws = torch.empty(bsz * slots * P, device=DEV)
        with torch.cuda.device(DEV):
            _cabi.check(L.mlg_pool_bwd_layout(_cabi.fptr(gout), _cabi.fptr(x), None, _cabi.fptr(w), _cabi.iptr(node.rowptr),
                                              _cabi.iptr(node.col), _cabi.iptr(lay.seg_of_slot), bsz, n, C, slots, 438, P,
                                              lay.replicas, _cabi.fptr(gx), _cabi.fptr(gw), _cabi.fptr(ws), 1, 0.2, None, nm,
                                              _cabi.stream_ptr()), "mlg_pool_bwd_layout")
        outs.append((gx, gw))
    gx_gm, gx_nm = outs[0][0], outs[1][0]
    assert torch.equal(gx_nm.view(n, bsz, C).transpose(0, 1).reshape(bsz * n, C), gx_gm)
    assert torch.equal(outs[0][1], outs[1][1])
    topo = graph.topology(b.edge_index.to(DEV), bsz * n, self_loops=True, edge_weight=b.edge_attr.to(DEV), period=n)
    assert topo.replicas == bsz
    bw = topo.bwd
    ref = torch.empty(bsz * n, 2 * C, device=DEV)
    Fn.gather_sum(gx_gm, bw.rowptr, bw.col, topo.n_single, val=topo.bwd_val, pre=topo.inv_cnt, out=ref[:, C:],
                  self_out=ref[:, :C], replicas=topo.replicas, order=topo.bwd_order)
    got = torch.empty(bsz * n, 2 * C, device=DEV)
    with torch.cuda.device(DEV):
        _cabi.check(L.mlg_gather_sum_nm(_cabi.fptr(gx_nm), _cabi.iptr(bw.rowptr), _cabi.iptr(bw.col), _cabi.fptr(topo.bwd_val, True),
                                        _cabi.fptr(topo.inv_cnt, True), _cabi.iptr(topo.bwd_order, True), topo.n_single, bsz,
                                        ctypes_ptr(got[:, C:]), 2 * C, _cabi.fptr(got), 2 * C, _cabi.stream_ptr()),
                    "mlg_gather_sum_nm")
    assert torch.equal(got, ref)


def test_csr_build_matches_sort(mlg):
    from multilevel_gnn_b200 import graph
    n, e = 1000, 20000
    ei, g = _rand_graph(n, e, 21)
    ei[:, :50] = ei[0, :50]
    csr = graph.build_csr(ei.to(DEV), n, drop_self=True, add_self=True)
    rp, col, eid = csr.rowptr.cpu().long(), csr.col.cpu().long(), csr.eid.cpu().long()
    keep = ei[0] != ei[1]
    src = torch.cat([ei[0][keep], torch.arange(n)])
    dst = torch.cat([ei[1][keep], torch.arange(n)])
    ids = torch.cat([torch.arange(e)[keep], torch.full((n,), -1)])
    order = torch.sort(dst, stable=True).indices
    nnz = int(rp[-1])
    assert nnz == src.numel()
    assert torch.equal(rp, torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(torch.bincount(dst, minlength=n), 0)]))
    assert torch.equal(col[:nnz], src[order])
    assert torch.equal(eid[:nnz], ids[order])
    empty = graph.build_csr(torch.zeros(2, 0, dtype=torch.long, device=DEV), 7)
    assert torch.equal(empty.rowptr.cpu(), torch.zeros(8, dtype=torch.int32))


def test_errors_are_loud(mlg):
    from multilevel_gnn_b200 import _cabi
    conv = mlg.GraphConv(8, 8, conv="sage", act="leakyrelu", mlp_norm="none")
    with pytest.raises(_cabi.NativeLibraryError):
        conv(torch.randn(4, 8), torch.zeros(2, 3, dtype=torch.long), torch.ones(3, 1))     # CPU tensors: no fallback
    L = _cabi.lib()
    assert L.mlg_gather_sum(None, 8, None, None, None, None, None, None, 4, 8, 1, 4, 0, 0, 0, None, 0, None, 8, None, 0, None, 0,
                            0.0, None, None) < 0
    assert "null" in _cabi.last_error()


def test_xty_matches_matmul(mlg):
    from multilevel_gnn_b200 import functional as Fn
    g = torch.Generator().manual_seed(31)
    for rows, M, K in [(5000, 64, 128), (777, 32, 128), (12345, 64, 64), (33, 8, 4), (1000, 100, 260)]:
        a = torch.randn(rows, M, generator=g).to(DEV)
        x = torch.randn(rows, K, generator=g).to(DEV)
        out, cs = Fn.xty(a, x, want_colsum=True)
        ref = (a.double().t() @ x.double()).float()
        assert_close(out, ref, rtol=1e-5, atol=2e-6, what="xty %s" % ((rows, M, K),))
        assert_close(cs, a.double().sum(0).float(), rtol=1e-5, atol=2e-6, what="colsum")
    # strided operands (halves of a wider buffer)
    big = torch.randn(4000, 96, generator=g).to(DEV)
    out, _ = Fn.xty(big[:, :32], big[:, 32:])
    assert_close(out, (big[:, :32].double().t() @ big[:, 32:].double()).float(), rtol=1e-5, atol=2e-6, what="xty strided")


def test_xty_tensor_core_matches_fp64(mlg):
    """mlg_xty_tc (transpose + 3xTF32 split in shared memory, tcgen05): fp32-accurate, deterministic, ragged row
    counts (zero-filled tail chunk), strided operands, every supported M."""
    from multilevel_gnn_b200 import functional as Fn
    g = torch.Generator().manual_seed(32)
    L = mlg._cabi.lib()
    for rows, M in [(64000, 64), (8192, 16), (100003, 32), (20001, 128), (9000, 48), (300000, 64)]:
        assert L.mlg_xty_tc_supported(rows, M, 128)
        a = torch.randn(rows, M, generator=g).to(DEV)
        x = (torch.randn(rows, 128, generator=g) * 3 + 0.5).to(DEV)
        out, cs = Fn.xty(a, x, want_colsum=True)
        ref = (a.double().t() @ x.double())
        scale = (a.double().abs().t() @ x.double().abs())
        err = ((out.double() - ref).abs() / scale).max().item()
        assert err < 4e-6, ("xty_tc rel-to-abs-product error", rows, M, err)
        assert_close(cs, a.double().sum(0).float(), rtol=1e-5, atol=1e-3, what="colsum_tc")
        out2, cs2 = Fn.xty(a, x, want_colsum=True)
        assert torch.equal(out, out2) and torch.equal(cs, cs2), "xty_tc must be deterministic"
        Fn.USE_TF32X3 = False
        try:
            simt, _ = Fn.xty(a, x)
        finally:
            Fn.USE_TF32X3 = True
        assert ((simt.double() - out.double()).abs() / scale).max().item() < 4e-6
    big = torch.randn(50000, 256, generator=g).to(DEV)      # strided: halves of a wider buffer
    out, _ = Fn.xty(big[:, :64], big[:, 128:])
    ref = big[:, :64].double().t() @ big[:, 128:].double()
    assert ((out.double() - ref).abs().max() / ref.abs().max()).item() < 1e-5
    assert not L.mlg_xty_tc_supported(1000, 64, 64) and not L.mlg_xty_tc_supported(1000, 20, 128)
    # wider problems through the same kernel: M in 128-column chunks, and K > 128 with the roles swapped (the bias
    # gradient then comes from the kernel's X-column sums) -- the node-side MLP Linears 128 -> 256 and 256 -> 128
    for rows, M, K in [(100146, 256, 128), (100146, 128, 256), (9000, 128, 384)]:
        a = torch.randn(rows, M, generator=g).to(DEV)
        x = torch.randn(rows, K, generator=g).to(DEV)
        Fn._cabi.TIMER = Fn._cabi.KernelTimer()
        out, cs = Fn.xty(a, x, want_colsum=True)
        tags = set(Fn._cabi.TIMER.summary())
        Fn._cabi.TIMER = None
        assert all(t.endswith("_tc") for t in tags), tags
        ref = a.double().t() @ x.double()
        scale = a.double().abs().t() @ x.double().abs()
        assert out.shape == (M, K) and out.is_contiguous()
        assert ((out.double() - ref).abs() / scale).max().item() < 4e-6, (rows, M, K)
        assert_close(cs, a.double().sum(0).float(), rtol=1e-5, atol=2e-3, what="colsum wide")


def test_skinny_linear_and_head_wgrad(mlg):
    """Head Linear(6913 -> 256) on <= 32 rows: mlg_skinny_linear forward (bias + act fused) and the single-part
    mlg_xty weight gradient (direct write, no reduce pass) against fp64."""
    from multilevel_gnn_b200 import functional as Fn
    g = torch.Generator().manual_seed(33)
    for rows, N, K in [(32, 256, 6913), (4, 256, 6913), (17, 100, 1025), (1, 8, 5000), (32, 2, 84096)]:
        x = torch.randn(rows, K, generator=g).to(DEV)
        w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV)
        b = torch.randn(N, generator=g).to(DEV)
        for act, slope in [(0, 0.0), (1, 0.0), (1, 0.2)]:
            out = Fn.tall_matmul(x, w, b, act=act, slope=slope)
            ref = x.double() @ w.double().t() + b.double()
            if act:
                ref = torch.where(ref > 0, ref, ref * slope)
            assert_close(out, ref.float(), rtol=1e-5, atol=1e-5, what="skinny %s act=%d" % ((rows, N, K), act))
        assert torch.equal(Fn.tall_matmul(x, w, b), Fn.tall_matmul(x, w, b))
        gy = torch.randn(rows, N, generator=g).to(DEV)
        gw, gb = Fn.xty(gy, x, want_colsum=True)
        assert_close(gw, (gy.double().t() @ x.double()).float(), rtol=1e-5, atol=1e-5, what="head wgrad")
        assert_close(gb, gy.double().sum(0).float(), rtol=1e-5, atol=1e-5, what="head bgrad")
    lin = torch.nn.Linear(6913, 256).to(DEV)
    x = torch.randn(32, 6913, device=DEV, requires_grad=True)
    y = Fn.tall_linear(x, lin, min_rows=1)
    y.square().sum().backward()
    gx, gw = x.grad.clone(), lin.weight.grad.clone()
    x.grad = None; lin.weight.grad = None
    torch.nn.functional.linear(x, lin.weight, lin.bias).square().sum().backward()
    assert_close(gx, x.grad, rtol=1e-4, atol=1e-5, what="head dgrad")
    assert_close(gw, lin.weight.grad, rtol=1e-4, atol=1e-5, what="head wgrad (autograd)")


def test_activation_backward_fusion_is_equivalent(mlg):
    """The cross-layer fusion (consumer kernels apply LeakyReLU' of their input; producers take dL/dz) must give the
    gradients of the unfused chain (numerics only; which kernels ran is asserted in tests/test_gpu_zz_structure.py,
    which sorts last so that a structural regression can never hide numerical tests behind ``-x``)."""
    from multilevel_gnn_b200 import configs, synth
    args = configs.make_args("gbm")
    torch.manual_seed(3)
    model = mlg.MultilevelGNN(args)
    synth.multilevel_params(model)
    model.to(DEV).train()
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    b = synth.multilevel_batch(batch_size=3, seed=5).to(DEV)
    params = [p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]

    def grads(fuse):
        type(model).FUSE_ACT_BACKWARD = fuse
        torch.manual_seed(11)                     # same dropout masks
        try:
            pred, feat = model(b)
            loss = (pred * torch.arange(pred.numel(), device=DEV).reshape(pred.shape)).sum() + feat.square().mean()
            g = torch.autograd.grad(loss, params, allow_unused=True)
        finally:
            type(model).FUSE_ACT_BACKWARD = True
        return g

    g1 = grads(True)
    g0 = grads(False)
    for a, c in zip(g1, g0):
        if a is None or c is None:
            assert a is None and c is None
            continue
        assert_close(a, c, rtol=1e-5, atol=1e-7, what="fused vs unfused grad")


def test_factored_first_layer_is_equivalent(mlg):
    """mlg_sage_rank1_fwd_rows / _bwd_rows (first SAGE layer factored through the per-gene tables E_self / E_nbr) against
    the [x0 | agg] buffer + GEMM path it replaces: prediction, pooled features and every parameter gradient, on the plain
    and on the activation-unfused chain; and the factored path must be the one that ran.  The 32-wide first layer with
    activation fusion off is the one route that applies LeakyReLU' in a library pass (no sign words at width 32)."""
    from multilevel_gnn_b200 import _cabi, configs, functional as Fn, synth
    for cfg, over, fuse in (("gbm", {}, True), ("gbm", {}, False), ("kirc", {}, True), ("gbm", dict(hidden_channels=32), False)):
        args = configs.make_args(cfg, **over)
        torch.manual_seed(3)
        model = mlg.MultilevelGNN(args)
        synth.multilevel_params(model)
        model.to(DEV).train()
        model.pathway_indexs = model.pathway_indexs.to(DEV)
        b = synth.multilevel_batch(batch_size=5, seed=6).to(DEV)
        params = [p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]

        defaults = (Fn.FACTORED_RANK1, Fn.TRANSFORM_FIRST)

        def run(factored, tfirst=True):
            Fn.FACTORED_RANK1 = factored
            Fn.TRANSFORM_FIRST = tfirst
            type(model).FUSE_ACT_BACKWARD = fuse
            torch.manual_seed(11)                     # same dropout masks
            timer = _cabi.KernelTimer()
            _cabi.TIMER = timer
            try:
                pred, feat = model(b)
                loss = (pred * torch.arange(pred.numel(), device=DEV).reshape(pred.shape)).sum() + feat.square().mean()
                g = torch.autograd.grad(loss, params, allow_unused=True)
                torch.cuda.synchronize()
            finally:
                _cabi.TIMER = None
                Fn.FACTORED_RANK1, Fn.TRANSFORM_FIRST = defaults
                type(model).FUSE_ACT_BACKWARD = True
            return pred.detach(), feat.detach(), g, set(timer.summary())

        p0, f0, g0, tags0 = run(False, False)      # [x | agg] buffer + GEMM in both layers
        assert not ({"sage_rank1_fwd", "sage_rank1_bwd"} & tags0), tags0
        names = [n for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]
        # first flag: the factored first layer (backward by target row: mlg_sage_rank1_bwd_rows + segment sum).  second:
        # layer 2 (64 -> 32) transform-first (layer 1 then masks its own output gradient)
        for mode, tfirst in ((True, True), (True, False), (False, True)):
            p1, f1, g1, tags1 = run(mode, tfirst)
            if mode:
                assert {"sage_rank1_fwd", "sage_rank1_bwd", "sage_rank1_bwd_seg"} <= tags1, tags1
            assert_close(p1, p0, rtol=1e-5, atol=1e-6, what="factored vs buffered pred")
            assert_close(f1, f0, rtol=1e-4, atol=1e-6, what="factored vs buffered pooled features")
            for n, a, c in zip(names, g1, g0):
                if a is None or c is None:
                    assert a is None and c is None
                    continue
                sc = float(c.abs().max().clamp_min(1e-30))      # compare at unit scale: atol is then relative to the largest entry
                assert_close_flips(a / sc, c / sc, "factored (%s, transform-first %s) vs buffered grad %s" % (mode, tfirst, n),
                                   rtol=1e-4, atol=2e-6, l2=1e-4, outliers=1e-4)


def test_node_major_activation_is_equivalent(mlg):
    """Layer-to-layer layout hand-shake (Fn.H1_NODE_MAJOR): the factored first layer writes its activation node-major
    (mlg_sage_rank1_fwd_rows_nm), the transform-first second layer aggregates contiguous blocks (mlg_gather_sum_nm_ex) and
    hands a node-major gradient back (mlg_sage_rank1_bwd_rows_nm).  Prediction, pooled features and every parameter
    gradient against the graph-major path, at 5 and at 40 graphs (two replica passes in the first-layer kernels); with a
    forward hook on a layer the hand-shake must stay off (the hook sees the reference's row order)."""
    from multilevel_gnn_b200 import _cabi, configs, functional as Fn, synth
    for cfg, bsz in (("gbm", 5), ("kirc", 5), ("gbm", 40)):
        args = configs.make_args(cfg)
        torch.manual_seed(3)
        model = mlg.MultilevelGNN(args)
        synth.multilevel_params(model)
        model.to(DEV).train()
        model.pathway_indexs = model.pathway_indexs.to(DEV)
        b = synth.multilevel_batch(batch_size=bsz, seed=6).to(DEV)
        params = [p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]
        names = [n for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]

        def run(nm):
            default = Fn.H1_NODE_MAJOR
            Fn.H1_NODE_MAJOR = nm
            torch.manual_seed(11)                     # same dropout masks
            try:
                pred, feat = model(b)
                loss = (pred * torch.arange(pred.numel(), device=DEV).reshape(pred.shape)).sum() + feat.square().mean()
                g = torch.autograd.grad(loss, params, allow_unused=True)
                torch.cuda.synchronize()
            finally:
                Fn.H1_NODE_MAJOR = default
            return pred.detach(), feat.detach(), g

        p0, f0, g0 = run(False)
        p1, f1, g1 = run(True)
        assert_close(p1, p0, rtol=1e-5, atol=1e-6, what="node-major vs graph-major pred")
        assert_close(f1, f0, rtol=1e-4, atol=1e-6, what="node-major vs graph-major pooled features")
        for n, a, c in zip(names, g1, g0):
            if a is None or c is None:
                assert a is None and c is None
                continue
            sc = float(c.abs().max().clamp_min(1e-30))
            # atol: the layer-2 weight gradient is a 3xTF32 sum over B*N rows taken in ANOTHER row order (accurate to ~4e-6 of
            # sum |g||x|, DESIGN section 2): 1e-5 of the largest entry at 616 k rows
            assert_close_flips(a / sc, c / sc, "node-major vs graph-major grad %s (%s, B=%d)" % (n, cfg, bsz),
                               rtol=1e-4, atol=2e-5, l2=1e-4, outliers=1e-4)
        # a hooked layer keeps the reference's row order
        rows = []
        h = model.gnn_model[0].register_forward_hook(lambda m, i, o: rows.append(o.detach().clone()))
        try:
            Fn.H1_NODE_MAJOR = True
            torch.manual_seed(11)
            model(b)
            Fn.H1_NODE_MAJOR = False
            torch.manual_seed(11)
            model(b)
        finally:
            Fn.H1_NODE_MAJOR = True
            h.remove()
        assert torch.equal(rows[0], rows[1])


def test_maxpool_channel_last_matches_torch(mlg):
    """mlg_maxpool_cl_fwd/bwd vs nn.MaxPool2d on the head's shape and on ragged ones (floor mode drops the tail rows /
    columns); ties (quantised values) must route the gradient to the first maximum like ATen."""
    from multilevel_gnn_b200 import functional as Fn
    g = torch.Generator().manual_seed(41)
    for (B, C, H, W, kh, kw), quant in [((32, 64, 146, 6, 4, 2), False), ((3, 32, 146, 6, 4, 2), True),
                                        ((2, 5, 7, 9, 3, 2), True), ((1, 64, 8, 8, 1, 1), False), ((2, 16, 5, 4, 5, 4), False)]:
        base = torch.randn(B, H, W, C, generator=g)
        if quant:
            base = (base * 2).round() / 2          # many exact ties inside a window
        x = base.to(DEV).permute(0, 3, 1, 2).requires_grad_(True)          # NCHW view of channel-last memory
        xr = base.permute(0, 3, 1, 2).contiguous().to(DEV).requires_grad_(True)
        y = Fn.MaxPoolCL.apply(x, kh, kw)
        yr = torch.nn.functional.max_pool2d(xr, (kh, kw))
        assert y.is_contiguous() and torch.equal(y, yr)
        go = torch.randn(yr.shape, generator=g).to(DEV)
        (gx,) = torch.autograd.grad(y, x, go)
        (gr,) = torch.autograd.grad(yr, xr, go)
        assert torch.equal(gx, gr), (B, C, H, W, kh, kw)


def test_layernorm_matches_torch(mlg):
    """mlg_layernorm_fwd/bwd (functional.LayerNormFn) vs torch layer_norm in fp64: output, input gradient, gamma / beta
    gradients; ragged row counts; deterministic; module wrapper falls back for unsupported widths."""
    from multilevel_gnn_b200 import functional as Fn
    from multilevel_gnn_b200.gcn_lib.sparse.torch_nn import norm_layer
    g = torch.Generator().manual_seed(51)
    for rows, C in [(100146, 128), (100146, 256), (4097, 384), (5000, 512)]:
        x = (torch.randn(rows, C, generator=g) * 2 + 0.7).to(DEV).requires_grad_(True)
        w = (torch.rand(C, generator=g) + 0.5).to(DEV).requires_grad_(True)
        b = torch.randn(C, generator=g).to(DEV).requires_grad_(True)
        go = torch.randn(rows, C, generator=g).to(DEV)
        y = Fn.LayerNormFn.apply(x, w, b, 1e-5)
        gx, gw, gb = torch.autograd.grad(y, [x, w, b], go)
        xd, wd, bd = x.detach().double().requires_grad_(True), w.detach().double().requires_grad_(True), b.detach().double().requires_grad_(True)
        yr = torch.nn.functional.layer_norm(xd, (C,), wd, bd, 1e-5)
        rx, rw, rb = torch.autograd.grad(yr, [xd, wd, bd], go.double())
        assert_close(y, yr.float(), rtol=1e-5, atol=1e-5, what="ln y")
        assert_close(gx, rx.float(), rtol=1e-4, atol=1e-5, what="ln gx")
        assert_close(gw, rw.float(), rtol=1e-4, atol=2e-3, what="ln dgamma")
        assert_close(gb, rb.float(), rtol=1e-4, atol=2e-3, what="ln dbeta")
        y2 = Fn.LayerNormFn.apply(x, w, b, 1e-5)
        g2 = torch.autograd.grad(y2, [x, w, b], go)
        assert torch.equal(y, y2) and all(torch.equal(a, c) for a, c in zip((gx, gw, gb), g2))
    # norm + ReLU in one pass each way (mlg_layernorm_relu_fwd / _bwd) vs relu(layer_norm) in fp64; entries whose
    # pre-activation is within fp32 rounding of 0 may take the other branch: excluded from the gradient comparison
    for rows, C in [(100146, 128), (5003, 256)]:
        x = (torch.randn(rows, C, generator=g) * 2 + 0.7).to(DEV).requires_grad_(True)
        w = (torch.rand(C, generator=g) + 0.5).to(DEV).requires_grad_(True)
        b = torch.randn(C, generator=g).to(DEV).requires_grad_(True)
        go = torch.randn(rows, C, generator=g).to(DEV)
        y = Fn.LayerNormFn.apply(x, w, b, 1e-5, True)
        xd, wd, bd = x.detach().double().requires_grad_(True), w.detach().double().requires_grad_(True), b.detach().double().requires_grad_(True)
        pre = torch.nn.functional.layer_norm(xd, (C,), wd, bd, 1e-5)
        safe = (pre.detach().abs() > 1e-5)
        gom = go.double() * safe                                   # no gradient through the borderline entries on either side
        yr = torch.relu(pre)
        rx, rw, rb = torch.autograd.grad(yr, [xd, wd, bd], gom)
        gx, gw, gb = torch.autograd.grad(y, [x, w, b], gom.float())
        assert_close(y, yr.float(), rtol=1e-5, atol=1e-5, what="ln+relu y")
        assert float((y < 0).sum()) == 0
        assert_close(gx, rx.float(), rtol=1e-4, atol=1e-5, what="ln+relu gx")
        assert_close(gw, rw.float(), rtol=1e-4, atol=2e-3, what="ln+relu dgamma")
        assert_close(gb, rb.float(), rtol=1e-4, atol=2e-3, what="ln+relu dbeta")
    ln = norm_layer("layer", 256).to(DEV)
    xr = torch.randn(5000, 256, generator=g).to(DEV)
    assert torch.equal(ln.forward_relu(xr), torch.relu(ln(xr)))   # same kernel arithmetic, then max(., 0)
    assert type(ln).__mro__[1] is torch.nn.LayerNorm and set(ln.state_dict()) == {"weight", "bias"}
    xs = torch.randn(10, 256, device=DEV)                     # too few rows: library path
    assert_close(ln(xs), torch.nn.functional.layer_norm(xs, (256,), ln.weight, ln.bias, ln.eps), what="ln small")
    ln96 = norm_layer("layer", 96).to(DEV)                    # unsupported width: library path
    xw = torch.randn(5000, 96, device=DEV)
    assert_close(ln96(xw), torch.nn.functional.layer_norm(xw, (96,), ln96.weight, ln96.bias, ln96.eps), what="ln 96")


def test_replicated_topology_equals_generic(mlg):
    """The B-copies fast path (single-graph CSR streamed over the batch) must agree with the generic CSR."""
    from multilevel_gnn_b200 import functional as Fn, graph, synth
    genes, bsz = 250, 5
    b = synth.multilevel_batch(batch_size=bsz, genes=genes, slots=600, intra_edges=3000, seed=12).to(DEV)
    n = 3 * genes * bsz
    x = torch.randn(n, 64, device=DEV, requires_grad=True)
    rep = graph.Topology(b.edge_index, n, self_loops=True, edge_weight=b.edge_attr, period=3 * genes)
    gen = graph.Topology(b.edge_index, n, self_loops=True, edge_weight=b.edge_attr)
    assert rep.replicas == bsz and gen.replicas == 1
    y1, y2 = Fn.SageAggregate.apply(x, rep, False), Fn.SageAggregate.apply(x, gen, False)
    assert_close(y1, y2.cpu(), rtol=1e-6, what="replicated fwd")
    go = torch.randn_like(y1)
    g1, g2 = torch.autograd.grad(y1, x, go)[0], torch.autograd.grad(y2, x, go)[0]
    assert_close(g1, g2.cpu(), rtol=1e-5, what="replicated bwd")
    # a batch whose graphs differ must NOT be detected as replicated
    ei = b.edge_index.clone()
    ei[0, -1] = ei[0, -1] - 3 if int(ei[0, -1]) % (3 * genes) >= 3 else ei[0, -1] + 3
    assert graph.Topology(ei, n, self_loops=True, edge_weight=b.edge_attr, period=3 * genes).replicas == 1


def test_trainer_steps_match_cpu_port(mlg):
    """Two optimizer steps of the B200 Trainer vs the CPU port of train.py:38-68 (loss + updated weights)."""
    from multilevel_gnn_b200.train import Trainer
    from oracle.train_port import CpuTrainer
    c = load_golden("multilevel")["gbm"]
    model, args = _build_multilevel(mlg, c)
    args.lr = 1e-2
    model.drop1.p = 0.0
    model.head[2].p = 0.0                      # dropout off: the port has none
    batch = as_batch(c["batch"], DEV)
    cpu = CpuTrainer({k: v.clone() for k, v in c["state_dict"].items()}, args, c["weight"], c["batch"]["raw_indice"][0])
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    tr = Trainer(model, args, c["weight"].to(DEV))
    for step in range(2):
        lg = tr.step(batch)
        lc = cpu.step(as_batch(c["batch"]))
        assert_close(lg, lc, rtol=2e-4, what="loss step %d" % step)
    sd = model.state_dict()
    for k in cpu.train_keys:
        assert_close(sd[k], cpu.sd[k], rtol=1e-3, atol=2e-5, what="weights after 2 steps: " + k)


# ------------------------------------------------------------------------------------------------
# DiffPool vs golden (reference-sized problems: fp32 library GEMMs, rtol 1e-4)
# ------------------------------------------------------------------------------------------------
DPG = load_golden("diffpool")


@pytest.mark.parametrize("name", sorted(DPG))
def test_diffpool_golden(mlg, name):
    c = DPG[name]
    args = mlg.configs.make_args("lgg")
    dp = _load(mlg.DiffPool(c["c"], 2, c["n"], 2, c["hid"], c["outd"], args), c["state_dict"])
    dp.train()
    x = c["x"].to(DEV).requires_grad_()
    out, l, e = dp(x, c["adj"].to(DEV))
    assert_close(out, c["out"], what=name + ".out")
    assert_close(l, c["link"], what=name + ".link")
    assert_close(e, c["ent"], what=name + ".ent")
    ((out * c["R"].to(DEV)).sum() + 3.0 * l + 0.5 * e).backward()
    assert_close(x.grad, c["g_x"], rtol=2e-4, what=name + ".g_x")
    for k, p in dp.named_parameters():
        if c["g_params"].get(k) is not None:
            assert_close(p.grad, c["g_params"][k], rtol=2e-4, what=name + ".g_" + k)


def test_cuda_graph_step_equals_eager(mlg):
    """Trainer.capture(): 3 warm-up steps + 2 graph replays must land on the same weights as 5 eager steps."""
    from multilevel_gnn_b200.train import Trainer
    c = load_golden("multilevel")["kirc"]
    results = []
    for graphed in (False, True):
        model, args = _build_multilevel(mlg, c)
        args.lr = 1e-2
        model.drop1.p = 0.0
        model.head[2].p = 0.0
        model.pathway_indexs = model.pathway_indexs.to(DEV)
        batch = as_batch(c["batch"], DEV)
        tr = Trainer(model, args, c["weight"].to(DEV))
        if graphed:
            tr.capture(batch, warmup=3)
            for _ in range(2):
                loss = tr.step()
        else:
            for _ in range(5):
                loss = tr.step(batch)
        torch.cuda.synchronize()
        results.append((float(loss), {k: v.detach().clone() for k, v in model.state_dict().items()}))
    assert abs(results[0][0] - results[1][0]) <= 1e-5 * max(1.0, abs(results[0][0]))
    for k in results[0][1]:
        assert_close(results[1][1][k], results[0][1][k], rtol=1e-5, atol=1e-6, what="graph vs eager: " + k)


def test_captured_trainer_prefetch_keyed_and_keyless_batches(mlg):
    """The end-to-end path bench.py's `e2e` legs use (Trainer.prefetch -> step_prefetched -> loss_to_host):
    * a host batch fed through the staging buffers gives the loss an eager step on the same weights gives;
    * a keyless batch (the reference loader's layout: topology re-sent every step, train.py:42) with the SAME topology is
      accepted, one with ANOTHER edge list raises when its loss is read -- the topology is frozen at capture();
    * a keyed batch with a different key is refused before anything is copied."""
    import copy
    from multilevel_gnn_b200.train import Trainer
    c = load_golden("multilevel")["kirc"]
    model, args = _build_multilevel(mlg, c)
    args.lr = 1e-3
    model.drop1.p = 0.0
    model.head[2].p = 0.0
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    host = as_batch({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in c["batch"].items()})
    twin = copy.deepcopy(model)
    tr = Trainer(model, args, c["weight"].to(DEV))
    tr.capture(as_batch(c["batch"], DEV), warmup=3)
    ref = Trainer(twin, args, c["weight"].to(DEV))
    for _ in range(3):
        ref.step(as_batch(c["batch"], DEV))
    # (1) same data through the staging buffers: step 4 of both trainers
    host2 = as_batch({k: (v.clone().pin_memory() if torch.is_tensor(v) else v) for k, v in c["batch"].items()})
    host2.x = (host2.x * 0.5).pin_memory()
    tr.prefetch(host2)
    got = tr.loss_to_host(tr.step_prefetched()).get()
    b2 = as_batch(c["batch"], DEV)
    b2.x = b2.x * 0.5
    want = float(ref.step(b2))
    assert abs(got - want) <= 1e-5 * max(1.0, abs(want)), (got, want)
    # (2) keyless batch, same topology: fine (and the flag stays clear)
    tr.prefetch(host)
    tr.loss_to_host(tr.step_prefetched()).get()
    tr.check_topology_flag()
    # (3) keyless batch with another edge list: the mismatch surfaces with the loss
    bad = as_batch({k: (v.clone().pin_memory() if torch.is_tensor(v) else v) for k, v in c["batch"].items()})
    ei = bad.edge_index.clone()
    ei[0, 0] = (ei[0, 0] + 1) % int(ei.max())
    bad.edge_index = ei.pin_memory()
    tr.prefetch(bad)
    with pytest.raises(RuntimeError, match="different topology"):
        tr.loss_to_host(tr.step_prefetched()).get()
    # (4) keyed batches: the key the graph was captured with is required
    model3, args3 = _build_multilevel(mlg, c)
    model3.pathway_indexs = model3.pathway_indexs.to(DEV)
    dev_keyed = as_batch(c["batch"], DEV)
    dev_keyed.topology_key = "fold-0"
    tr3 = Trainer(model3, args3, c["weight"].to(DEV))
    tr3.capture(dev_keyed, warmup=3)
    other = as_batch({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in c["batch"].items()})
    other.topology_key = "fold-1"
    with pytest.raises(ValueError, match="frozen at capture"):
        tr3.prefetch(other)
    same = as_batch({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in c["batch"].items()})
    same.topology_key = "fold-0"
    tr3.prefetch(same)
    assert set(tr3._staging) == {k for k in vars(dev_keyed) if torch.is_tensor(getattr(dev_keyed, k))} - set(Trainer.STATIC_TOPOLOGY_FIELDS)
    loss = tr3.loss_to_host(tr3.step_prefetched()).get()
    assert loss == loss


# ------------------------------------------------------------------------------------------------
# edge cases: empty / ragged / non-replicated inputs
# ------------------------------------------------------------------------------------------------
def test_empty_edge_list(mlg):
    """A graph without edges: GENConv softmax aggregate -> 0 (so h = x), SAGE -> every node only sees its self loop."""
    n, H = 70, 32
    g = torch.Generator().manual_seed(2)
    x = torch.randn(n, H, generator=g)
    ei = torch.zeros(2, 0, dtype=torch.long)
    conv = mlg.GENConv(H, H, aggr="softmax", msg_norm=True, encode_edge=False, norm="layer").to(DEV)
    sd = {k: v.detach().cpu() for k, v in conv.state_dict().items()}
    y = conv(x.to(DEV), ei.to(DEV), torch.zeros(0, H, device=DEV))
    assert_close(y, R.genconv_forward(sd, x, ei, torch.zeros(0, H), aggr="softmax", msg_norm_on=True, norm="layer"), what="GENConv E=0")
    sage = mlg.GraphConv(H, 16, conv="sage", act="leakyrelu", mlp_norm="none").to(DEV)
    ssd = {k: v.detach().cpu() for k, v in sage.state_dict().items()}
    ys = sage(x.to(DEV), ei.to(DEV), torch.zeros(0, 1, device=DEV))
    assert_close(ys, R.sage_forward(ssd, x, ei, torch.zeros(0, 1)), what="SAGE E=0")


def test_ragged_batch_is_not_replicated(mlg):
    """Graphs of different sizes / different edge lists in one batch: the generic CSR path must be taken and agree
    with the oracle (the replicated fast path only applies to B offset copies of one edge list)."""
    from multilevel_gnn_b200 import graph
    g = torch.Generator().manual_seed(8)
    sizes = [40, 65, 13]
    eis, off = [], 0
    for s in sizes:
        e = torch.stack([torch.randint(0, s, (5 * s,), generator=g), torch.randint(0, s, (5 * s,), generator=g)]) + off
        eis.append(e)
        off += s
    ei = torch.cat(eis, 1)
    n = sum(sizes)
    w = torch.rand(ei.shape[1], 1, generator=g)
    x = torch.randn(n, 64, generator=g)
    topo = graph.Topology(ei.to(DEV), n, self_loops=True, edge_weight=w.to(DEV), period=40)
    assert topo.replicas == 1
    sage = mlg.GraphConv(64, 32, conv="rsage", act="relu", mlp_norm="none").to(DEV)
    ssd = {k: v.detach().cpu().clone().requires_grad_() for k, v in sage.state_dict().items()}
    xr = x.clone().requires_grad_()
    yr = R.sage_forward(ssd, xr, ei, w, relative=True, act="relu")
    xg = x.to(DEV).requires_grad_()
    yg = sage(xg, ei.to(DEV), w.to(DEV))
    assert_close(yg, yr, what="ragged rsage fwd")
    yr.sum().backward()
    yg.sum().backward()
    assert_close(xg.grad, xr.grad, rtol=2e-4, what="ragged rsage g_x")


def test_multilevel_single_graph_batch(mlg):
    """B = 1: no replication to exploit, rank-1 first layer falls back to the materialised embed-scale."""
    c = load_golden("multilevel")["gbm"]
    model, args = _build_multilevel(mlg, c)
    model.eval()
    n, G = 3 * c["genes"], c["slots"]
    E = c["batch"]["edge_index"].shape[1] // 3
    one = dict(x=c["batch"]["x"][:n], edge_index=c["batch"]["edge_index"][:, :E], edge_attr=c["batch"]["edge_attr"][:E],
               gene_pca_match=c["batch"]["gene_pca_match"][:1], raw_indice=c["batch"]["raw_indice"][:1],
               age=c["batch"]["age"][:1], y=c["batch"]["y"][:2])
    pred, feat = model(as_batch(one, DEV))
    assert_close(pred, c["pred"][:1], what="B=1 pred")
    assert_close(feat, c["pca_feature"][:1], what="B=1 pca_feature")


def test_knn_ragged_sizes_and_full_k(mlg):
    g = torch.Generator().manual_seed(4)
    for n, d, k in [(1, 5, 1), (7, 3, 7), (129, 17, 16), (300, 130, 64)]:
        x = torch.randn(n, d, generator=g)
        got = mlg.knn_graph_matrix(x.to(DEV), k)
        _check_knn(x, None, k, got, R.knn_graph_matrix(x, k), "n%d" % n)
    with pytest.raises(RuntimeError):
        mlg.knn_graph_matrix(torch.randn(5, 3, device=DEV), 6)          # k > N: torch.topk raises in the reference too


def _knn_raw(mlg, xb, k, dil, tensor_path):
    """mlg_knn_graph through the C ABI with either the full workspace (tensor-core candidate search where eligible) or just
    the squared-norm workspace (forces the fp32 kernel)."""
    L = mlg._cabi.lib()
    B, N, D = xb.shape
    nbr = torch.empty(B * N * k, dtype=torch.int64, device=DEV)
    ctr = torch.empty_like(nbr)
    dist = torch.empty(B * N * k, dtype=torch.float32, device=DEV)
    nbytes = int(L.mlg_knn_workspace_bytes(B, N, D, k, dil)) if tensor_path else B * N * 4
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=DEV)
    mlg._cabi.check(L.mlg_knn_graph(mlg._cabi.fptr(xb), B, N, D, k, dil, 1, mlg._cabi.lptr(nbr), mlg._cabi.lptr(ctr),
                                    mlg._cabi.fptr(dist), mlg._cabi.fptr(ws), nbytes, mlg._cabi.stream_ptr()), "mlg_knn_graph")
    torch.cuda.synchronize()
    return nbr, ctr, dist


@pytest.mark.parametrize("case", ["gauss_d64", "batch2_pad_dil", "d100_chunk128", "lattice_ties", "duplicates"])
def test_knn_tensor_core_path_equals_fp32_kernel(mlg, case):
    """Graphs of >= 4096 points: candidates from 3xTF32 distance products on the tensor cores, fp32 re-evaluation,
    certificate, repair pass (csrc/knn.cu) -- neighbours, order and distances must be IDENTICAL to the fp32 kernel's, which the
    tests above hold to the oracle.  The lattice / duplicate cases are dense in exact ties, so no row can be certified and
    the repair pass has to reproduce everything."""
    g = torch.Generator().manual_seed(31)
    if case == "gauss_d64":
        x, k, dil = torch.randn(1, 5000, 64, generator=g), 16, 1
    elif case == "batch2_pad_dil":
        x, k, dil = torch.randn(2, 4500, 20, generator=g) * 3.0, 5, 3
    elif case == "d100_chunk128":
        x, k, dil = torch.randn(1, 4200, 100, generator=g), 9, 1
    elif case == "lattice_ties":
        x, k, dil = torch.randint(0, 6, (1, 4096, 3), generator=g).float(), 16, 1
    else:
        base = torch.randn(1, 1024, 32, generator=g)
        x, k, dil = base.repeat(1, 4, 1), 8, 2
    xb = x.to(DEV).contiguous()
    assert int(mlg._cabi.lib().mlg_knn_workspace_bytes(x.shape[0], x.shape[1], x.shape[2], k, dil)) > x.shape[0] * x.shape[1] * 4 + 256
    n1, c1, d1 = _knn_raw(mlg, xb, k, dil, True)
    n0, c0, d0 = _knn_raw(mlg, xb, k, dil, False)
    assert torch.equal(c1, c0)
    assert torch.equal(n1, n0), "%s: %d of %d neighbours differ" % (case, int((n1 != n0).sum()), n0.numel())
    assert torch.equal(d1, d0)


def test_dynconv_knn_then_conv(mlg):
    """DynConv.forward (gcn_lib/sparse/torch_vertex.py:366-380): rebuild the dilated kNN graph from the features, then run the
    static convolution on it -- the kNN -> conv call site.  In the reference this path raises for every conv its configs could
    select (GraphConv.forward passes edge_attr= to EdgConv / MRConv.forward, which do not take it, and SAGEConv.forward calls
    edge_attr.dim() on None); here the 'sage' / 'rsage' convolutions run with unit edge weights, which is what the oracle's
    sage_forward computes for edge_attr=None.  Checked: the edge list (against the kNN oracle), the output and the input
    gradient, for two graphs in one batch, with dilation."""
    g = torch.Generator().manual_seed(21)
    n, c, k, d = 300, 16, 6, 2
    x = torch.randn(2 * n, c, generator=g)
    batch = torch.arange(2).repeat_interleave(n)
    for conv in ("sage", "rsage"):
        torch.manual_seed(5)
        dyn = mlg.DynConv(c, 24, kernel_size=k, dilation=d, conv=conv, act="leakyrelu", norm=None).to(DEV).eval()
        xg = x.to(DEV).requires_grad_()
        y = dyn(xg, batch.to(DEV))
        ei_ref = R.dilate(R.knn_graph_matrix(x, k * d, batch), d)
        ei = dyn.dilated_knn_graph(x.to(DEV), batch.to(DEV))
        assert torch.equal(ei.cpu(), ei_ref), conv + ": dilated kNN edge list"
        sd = {kk: v.detach().cpu().clone() for kk, v in dyn.state_dict().items()}
        xr = x.clone().requires_grad_()
        yr = R.sage_forward(sd, xr, ei_ref, None, relative=(conv == "rsage"), act="leakyrelu")
        assert_close(y, yr, what="DynConv(%s) output" % conv)
        Rw = torch.randn(yr.shape, generator=g)
        (gx,) = torch.autograd.grad((y * Rw.to(DEV)).sum(), xg)
        (gr,) = torch.autograd.grad((yr * Rw).sum(), xr)
        assert_close(gx, gr, rtol=2e-4, what="DynConv(%s) input gradient" % conv)
    with pytest.raises(NotImplementedError):
        mlg.DynConv(c, 24)            # default conv='edge': a torch_geometric wrapper, out of scope (SURVEY section 2 row 2)
