"""Pins oracle/restated.py (the CPU checker) to outputs of the REFERENCE's own files.

tests/golden/*.pt were produced by oracle/make_golden.py from /root/reference behind
oracle/pyg_stub.py.  The first block runs everywhere (CPU); the second re-runs the live reference
and only exists in the build container."""
import argparse

import pytest
import torch

from conftest import as_batch, assert_close, load_golden
from oracle import ref_import, restated as R


def _leafify(d):
    return {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in d.items()}


GEN = load_golden("genconv")
PWC = load_golden("pathwayconv")


@pytest.mark.parametrize("name", sorted(PWC))
def test_pathwayconv_restatement(name):
    """R.pathway_conv_forward against the reference's own PathwayConv (torch_vertex.py:107-178): output and all gradients."""
    c = PWC[name]
    kw = c["kw"]
    sd = _leafify(c["state_dict"])
    x, ea = c["x"].clone().requires_grad_(), c["edge_attr"].clone().requires_grad_()
    y = R.pathway_conv_forward(sd, x, c["edge_index"], ea, mask=c["mask"], aggr=kw["aggr"], t=kw.get("t", 1.0),
                               learn_t=kw.get("learn_t", False), norm=kw["norm"])
    assert_close(y, c["y"], what=name + ".y")
    names = list(c["g_params"])
    gs = torch.autograd.grad((y * c["R"]).sum(), [x, ea] + [sd[k] for k in names], allow_unused=True)
    assert_close(gs[0], c["g_x"], what=name + ".g_x")
    assert_close(gs[1], c["g_edge_attr"], what=name + ".g_edge_attr")
    for k, g in zip(names, gs[2:]):
        if c["g_params"][k] is None:
            assert g is None, k
        else:
            assert_close(g, c["g_params"][k], what=name + ".g_" + k)



@pytest.mark.parametrize("name", sorted(GEN))
def test_genconv_restatement(name):
    c = GEN[name]
    kw = c["kw"]
    sd = _leafify(c["state_dict"])
    x, ea = c["x"].clone().requires_grad_(), c["edge_attr"].clone().requires_grad_()
    y = R.genconv_forward(sd, x, c["edge_index"], ea, aggr=kw["aggr"], t=kw.get("t", 1.0),
                          learn_t=kw.get("learn_t", False), p=kw.get("p", 1.0), learn_p=kw.get("learn_p", False),
                          msg_norm_on=kw.get("msg_norm", False), encode_edge=True, norm=kw["norm"])
    assert_close(y, c["y"], what=name + ".y")
    names = list(c["g_params"])
    gs = torch.autograd.grad((y * c["R"]).sum(), [x, ea] + [sd[k] for k in names], allow_unused=True)
    assert_close(gs[0], c["g_x"], what=name + ".g_x")
    assert_close(gs[1], c["g_edge_attr"], what=name + ".g_edge_attr")
    for k, g in zip(names, gs[2:]):
        if c["g_params"][k] is None:
            assert g is None, k
        else:
            assert_close(g, c["g_params"][k], what=name + ".g_" + k)
    # aggregate on explicit messages
    msg = c["msg"].clone().requires_grad_()
    agg = R.gen_aggregate(msg * 1.0, c["edge_index"][1], c["x"].shape[0], aggr=kw["aggr"],
                          t=sd["t"] if "t" in sd else kw.get("t", 1.0), learn_t="t" in sd,
                          p=sd["p"] if "p" in sd else kw.get("p", 1.0), y=sd.get("y"))
    assert_close(agg, c["agg"], what=name + ".agg")
    assert_close(torch.autograd.grad((agg * c["R"]).sum(), msg)[0], c["g_msg"], what=name + ".g_msg")


SAGE = load_golden("sage")


@pytest.mark.parametrize("name", sorted(SAGE))
def test_sage_restatement(name):
    c = SAGE[name]
    sd = _leafify(c["state_dict"])
    x = c["x"].clone().requires_grad_()
    y = R.sage_forward(sd, x, c["edge_index"], c["edge_attr"], relative=c["conv"] == "rsage")
    assert_close(y, c["y"], what=name + ".y")
    names = [k for k in c["g_params"] if c["g_params"][k] is not None]
    gs = torch.autograd.grad((y * c["R"]).sum(), [x] + [sd[k] for k in names])
    assert_close(gs[0], c["g_x"], what=name + ".g_x")
    for k, g in zip(names, gs[1:]):
        assert_close(g, c["g_params"][k], what=name + ".g_" + k)
    assert c["g_params"]["gconv.lin_l.weight"] is None    # registered but unused in the reference


KNN = load_golden("knn")


@pytest.mark.parametrize("name", sorted(KNN))
def test_knn_restatement(name):
    c = KNN[name]
    ei = R.knn_graph_matrix(c["x"], c["k"] * c["dil"], c["batch"])
    if name == "grid_ties":   # tie order of torch.topk is unspecified: compare distances, not ids
        d = R.pairwise_distance(c["x"].view(1, -1, 2))[0]
        assert torch.equal(d[ei[1], ei[0]], d[c["edge_index_full"][1], c["edge_index_full"][0]])
        return
    assert torch.equal(ei, c["edge_index_full"])
    assert torch.equal(R.dilate(ei, c["dil"]), c["edge_index_dilated"])
    xd = c["x"].view(c["b"], c["n"], c["d"]).transpose(1, 2).unsqueeze(-1)
    assert torch.equal(R.dense_knn_matrix(xd, c["k"] * c["dil"]), c["dense_full"])
    assert torch.equal(R.dense_knn_matrix(xd, c["k"] * c["dil"])[:, :, :, ::c["dil"]], c["dense_dilated"])


ML = load_golden("multilevel")


def _ml_args(c):
    from multilevel_gnn_b200 import configs
    return configs.make_args(c["config"], **c["overrides"])


@pytest.mark.parametrize("name", sorted(ML))
def test_multilevel_restatement(name):
    c = ML[name]
    args = _ml_args(c)
    sd = _leafify(c["state_dict"])
    sd["info_mask"] = c["state_dict"]["info_mask"]
    batch = as_batch(c["batch"])
    pred, feat, acts = R.multilevel_forward(sd, batch, args, return_acts=True)
    assert_close(pred, c["pred"], what=name + ".pred")
    assert_close(feat, c["pca_feature"], what=name + ".pca_feature")
    for k, v in c["acts"].items():
        assert_close(acts[k], v, what=name + "." + k)
    fl = R.feature_loss(feat, sd["learnable_pca_params"], sd["info_mask"], c["batch"]["raw_indice"][0],
                        pca_loss=args.pca_loss, pca_indep_loss=args.pca_indep_loss)
    assert_close(torch.as_tensor(fl), c["feature_loss"], what=name + ".feature_loss")
    loss = R.bce_loss(pred, c["batch"]["y"].reshape(-1, 2), c["weight"]) + fl
    assert_close(loss, c["loss"], what=name + ".loss")
    names = [k for k, g in c["grads"].items() if g is not None]
    gs = torch.autograd.grad(loss, [sd[k] for k in names])
    for k, g in zip(names, gs):
        assert_close(g, c["grads"][k], what=name + ".g_" + k)
    assert all(c["grads"][k] is None for k in c["grads"] if k.endswith("lin_l.weight"))


DP = load_golden("diffpool")


@pytest.mark.parametrize("name", sorted(DP))
def test_diffpool_restatement(name):
    c = DP[name]
    sd = _leafify(c["state_dict"])
    x = c["x"].clone().requires_grad_()
    out, l, e = R.diffpool_forward(sd, x, c["adj"])
    assert_close(out, c["out"], what=name + ".out")
    assert_close(l, c["link"], what=name + ".link")
    assert_close(e, c["ent"], what=name + ".ent")
    names = [k for k, g in c["g_params"].items() if g is not None]
    gs = torch.autograd.grad((out * c["R"]).sum() + 3.0 * l + 0.5 * e, [x] + [sd[k] for k in names])
    assert_close(gs[0], c["g_x"], what=name + ".g_x")
    for k, g in zip(names, gs[1:]):
        assert_close(g, c["g_params"][k], what=name + ".g_" + k)


DG = load_golden("deepergcn")


@pytest.mark.parametrize("name", sorted(DG))
def test_deepergcn_restatement(name):
    from multilevel_gnn_b200 import configs
    c = DG[name]
    args = configs.make_args(None, **c["overrides"])
    sd = _leafify(c["state_dict"])
    pred = R.deepergcn_forward(sd, as_batch(c["batch"]), args)
    assert_close(pred, c["pred"], what=name + ".pred")
    names = [k for k, g in c["grads"].items() if g is not None]
    gs = torch.autograd.grad((pred * c["R"]).sum(), [sd[k] for k in names])
    for k, g in zip(names, gs):
        assert_close(g, c["grads"][k], rtol=2e-4, what=name + ".g_" + k)


# ------------------------------------------------------------------------------------------------
# container-only: the live reference at the gbm.yaml shape (B=2 to keep it in seconds)
# ------------------------------------------------------------------------------------------------
needs_ref = pytest.mark.skipif(not ref_import.available(),
                               reason="needs the original Multilevel-GNN source tree (MLG_REFERENCE_ROOT), which the repository does not ship")


@needs_ref
def test_full_size_multilevel_vs_live_reference():
    from multilevel_gnn_b200 import configs, synth
    ns = ref_import.load()
    torch.manual_seed(0)
    ref_args = ref_import.default_args("gbm.yaml")
    model = ns.multilevel_gnn.MultilevelGNN(ref_args)
    synth.multilevel_params(model)
    model.eval()
    batch = synth.multilevel_batch(batch_size=2, seed=3)
    pred, feat = model(batch)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    pred2, feat2 = R.multilevel_forward(sd, batch, configs.make_args("gbm"))
    assert_close(pred2, pred, what="pred")
    assert_close(feat2, feat, what="pca_feature")
    fl = model.get_feature_loss(feat)
    fl2 = R.feature_loss(feat2, sd["learnable_pca_params"], sd["info_mask"], model.pathway_indexs)
    assert_close(torch.as_tensor(fl2), torch.as_tensor(fl), what="feature_loss")


@needs_ref
def test_configs_match_reference_defaults():
    from multilevel_gnn_b200 import configs
    for cfg in (None, "gbm", "kirc", "lgg"):
        ref = ref_import.default_args(None if cfg is None else cfg + ".yaml")
        mine = configs.make_args(cfg)
        for k, v in vars(mine).items():
            if k == "pathway_edge_num":
                continue
            assert hasattr(ref, k), k
            assert getattr(ref, k) == v, (cfg, k, getattr(ref, k), v)


# ------------------------------------------------------------------------------------------------
# the same two checks against stored values (run everywhere): see "source" in each golden file
# ------------------------------------------------------------------------------------------------
def test_full_size_multilevel_restatement():
    """R.multilevel_forward at the gbm.yaml shape (B=2) on the seeded inputs of the live test above, against
    tests/golden/multilevel_full.pt: pred, pca_feature and the feature loss."""
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import configs, synth
    c = load_golden("multilevel_full")
    torch.manual_seed(0)
    args = configs.make_args("gbm")
    model = m.MultilevelGNN(args)
    synth.multilevel_params(model)
    batch = synth.multilevel_batch(batch_size=2, seed=3)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    pred, feat = R.multilevel_forward(sd, batch, args)
    assert_close(pred, c["pred"], what="pred")
    assert_close(feat, c["pca_feature"], what="pca_feature")
    fl = R.feature_loss(feat, sd["learnable_pca_params"], sd["info_mask"], model.pathway_indexs)
    assert_close(torch.as_tensor(fl), c["feature_loss"], what="feature_loss")


def test_configs_match_stored_reference_defaults():
    """configs.make_args against the original's opt.py defaults and config/{gbm,kirc,lgg}.yaml overlays for every key it
    sets (tests/golden/reference_args.json)."""
    import json
    import os
    from conftest import GOLDEN
    from multilevel_gnn_b200 import configs
    with open(os.path.join(GOLDEN, "reference_args.json")) as f:
        ref = json.load(f)["configs"]
    for cfg in (None, "gbm", "kirc", "lgg"):
        want = ref["default" if cfg is None else cfg]
        mine = {k: v for k, v in vars(configs.make_args(cfg)).items() if k != "pathway_edge_num"}
        assert sorted(mine) == sorted(want), cfg
        for k, v in mine.items():
            assert want[k] == v, (cfg, k, want[k], v)


# ------------------------------------------------------------------------------------------------
# VAE.predict_head (DiffPool's only call site) and the per-pathway decoders vs the reference's own VAE class
# ------------------------------------------------------------------------------------------------
VAEG = load_golden("vae")


@pytest.mark.parametrize("name", sorted(VAEG))
def test_predict_head_restatement(name):
    from multilevel_gnn_b200 import configs
    c = VAEG[name]
    args = configs.make_args("lgg", **c["overrides"])
    sd = _leafify(c["state_dict"])
    x = c["x"].clone().requires_grad_()
    adj = c["sim"] + torch.eye(146)
    pred, feat, l, e = R.predict_head(sd, x, c["age"], args, adj)
    assert_close(pred, c["pred"], what=name + ".pred")
    assert_close(torch.as_tensor(l), c["link"], what=name + ".link")
    assert_close(torch.as_tensor(e), c["ent"], what=name + ".ent")
    names = [k for k, g in c["g_params"].items() if g is not None]
    gs = torch.autograd.grad((pred * c["R"]).sum() + 3.0 * l + 0.5 * e, [x] + [sd[k] for k in names])
    assert_close(gs[0], c["g_x"], rtol=2e-4, what=name + ".g_x")
    for k, g in zip(names, gs[1:]):
        assert_close(g, c["g_params"][k], rtol=2e-4, what=name + ".g_" + k)
    if "dec" in c:
        h = c["h"].clone().requires_grad_()
        dec = R.foreach_decoder(sd, h)
        assert_close(dec, c["dec"], what=name + ".dec")
        dn = list(c["g_dec"])
        gd = torch.autograd.grad((dec * c["Rd"]).sum(), [h] + [sd[k] for k in dn])
        assert_close(gd[0], c["g_h"], rtol=2e-4, what=name + ".g_h")
        for k, g in zip(dn, gd[1:]):
            assert_close(g, c["g_dec"][k], rtol=2e-4, what=name + ".g_" + k)
