"""The fused classification head + loss kernels (csrc/head.cu) against plain torch in fp64:
Conv2d(1x1)+ReLU x2 + MaxPool2d + Dropout + flatten + cat(age)  (models/multilevel_gnn.py:262-288 of the reference) and
Linear+ReLU+Dropout + Linear(->2) + Softmax + BCELoss(weight)   (models/multilevel_gnn.py:104-110,288-290; train.py:60,118).
Outputs and every gradient; tolerance fp32 rtol 1e-4."""
import pytest
import torch
import torch.nn.functional as F

from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def mlg():
    import multilevel_gnn_b200 as m
    m._cabi.lib()
    return m


def _ref_conv_pool(x, W1, b1, W2, b2, age, kh, kw, mask=None, p=0.0):
    h = F.relu(F.conv2d(x, W1, b1))
    h = F.relu(F.conv2d(h, W2, b2))
    h = F.max_pool2d(h, (kh, kw))
    if mask is not None:
        h = h * mask.view(h.shape) / (1.0 - p)
    h = torch.flatten(h, start_dim=1)
    if age is not None:
        h = torch.cat([h, age[:, None]], dim=-1)
    return h


@pytest.mark.parametrize("B,H,W,kh,kw,with_age", [(32, 146, 6, 4, 2, True), (5, 146, 9, 1, 1, False), (3, 7, 5, 2, 2, True),
                                                   (2, 9, 4, 3, 4, False), (2, 30, 20, 4, 2, True), (3, 40, 16, 4, 4, False)])
def test_head_conv_pool_matches_torch(mlg, B, H, W, kh, kw, with_age):
    from multilevel_gnn_b200 import functional as Fn
    g = torch.Generator().manual_seed(100 + B)
    x_cl = torch.randn(B, H, W, 32, generator=g)
    W1 = torch.randn(32, 32, 1, 1, generator=g) * 0.3
    b1 = torch.randn(32, generator=g) * 0.2
    W2 = torch.randn(64, 32, 1, 1, generator=g) * 0.3
    b2 = torch.randn(64, generator=g) * 0.2
    age = torch.rand(B, generator=g) if with_age else None
    dev = [t.to(DEV).requires_grad_() for t in (x_cl, W1, b1, W2, b2)]
    feat = dev[0].permute(0, 3, 1, 2)                       # NCHW view of channel-last memory
    a0 = Fn.HeadConvPool.apply(feat, dev[1], dev[2], dev[3], dev[4], None if age is None else age.to(DEV), kh, kw, 0.25, False)
    ref_in = [t.double().requires_grad_() for t in (x_cl, W1, b1, W2, b2)]
    ref = _ref_conv_pool(ref_in[0].permute(0, 3, 1, 2), ref_in[1], ref_in[2], ref_in[3], ref_in[4],
                         None if age is None else age.double(), kh, kw)
    assert a0.shape == ref.shape
    assert_close(a0, ref.float(), what="a0")
    Rw = torch.randn(ref.shape, generator=g)
    gs = torch.autograd.grad((a0 * Rw.to(DEV)).sum(), dev)
    gr = torch.autograd.grad((ref * Rw.double()).sum(), ref_in)
    for name, a, c in zip(("g_x", "g_W1", "g_b1", "g_W2", "g_b2"), gs, gr):
        assert_close(a, c.float(), rtol=1e-4, atol=2e-6, what=name)
    # deterministic
    a0b = Fn.HeadConvPool.apply(feat, dev[1], dev[2], dev[3], dev[4], None if age is None else age.to(DEV), kh, kw, 0.25, False)
    gs2 = torch.autograd.grad((a0b * Rw.to(DEV)).sum(), dev)
    assert torch.equal(a0, a0b) and all(torch.equal(a, c) for a, c in zip(gs, gs2))


def test_head_conv_pool_dropout_uses_torch_generator(mlg):
    """Training mode: the mask is (bits >= p * 2^31) of int32 words drawn from torch's CUDA generator, so torch.manual_seed
    reproduces it; kept elements are scaled by 1/(1-p), the backward pass applies the same mask."""
    from multilevel_gnn_b200 import functional as Fn
    B, H, W, kh, kw, p = 8, 146, 6, 4, 2, 0.25
    g = torch.Generator().manual_seed(5)
    x_cl = torch.randn(B, H, W, 32, generator=g).to(DEV).requires_grad_()
    W1 = (torch.randn(32, 32, 1, 1, generator=g) * 0.3).to(DEV)
    b1 = torch.zeros(32, device=DEV)
    W2 = (torch.randn(64, 32, 1, 1, generator=g) * 0.3).to(DEV)
    b2 = (torch.rand(64, generator=g) + 0.5).to(DEV)
    feat = x_cl.permute(0, 3, 1, 2)
    torch.manual_seed(77)
    a0 = Fn.HeadConvPool.apply(feat, W1, b1, W2, b2, None, kh, kw, p, True)
    torch.manual_seed(77)
    bits = torch.empty(a0.numel(), dtype=torch.int32, device=DEV).random_()
    mask = (bits >= int(p * 2 ** 31)).double().cpu()
    assert 0.70 < float(mask.mean()) < 0.80
    # fp64 reference on the CPU (a GPU conv2d reference would run in TF32)
    xr = x_cl.detach().cpu().double().requires_grad_()
    wr = [t.detach().cpu().double() for t in (W1, b1, W2, b2)]
    ref = _ref_conv_pool(xr.permute(0, 3, 1, 2), wr[0], wr[1], wr[2], wr[3], None, kh, kw, mask=mask, p=p)
    assert_close(a0, ref.float(), what="dropout fwd")
    Rw = torch.randn(a0.shape, generator=g)
    g1 = torch.autograd.grad((a0 * Rw.to(DEV)).sum(), x_cl)[0]
    g2 = torch.autograd.grad((ref * Rw.double()).sum(), xr)[0]
    assert_close(g1, g2.float(), rtol=1e-4, atol=2e-6, what="dropout bwd")
    a_eval = Fn.HeadConvPool.apply(feat, W1, b1, W2, b2, None, kh, kw, p, False)
    ref_eval = _ref_conv_pool(xr.permute(0, 3, 1, 2), wr[0], wr[1], wr[2], wr[3], None, kh, kw)
    assert_close(a_eval, ref_eval.float(), what="eval: no dropout")


# every hidden width the kernels accept (a multiple of 32 up to 512) on both sides of the 32-row tile and at a full 64-row
# tile: the input-gradient pass's row groups (mlp_bwd_rows_per_group) depend on D through the block size; K = 300 leaves a
# partial K slice.  Then kirc's and lgg's classifier heads at their batch width.
MLP_SHAPES = ([(32, 6913, 256), (64, 1000, 512), (3, 77, 32), (17, 300, 64)]
              + [(r, 300, d) for d in range(32, 513, 32) for r in (31, 32, 33, 64)]
              + [(64, 84096, 512), (64, 9217, 512)])


def _clear_of_relu_kink(a0, W0, b0, margin=1e-4):
    """b0 moved (by a few margins) so that no hidden pre-activation a0 W0^T + b0 lies within ``margin`` of its sum|terms| of 0.
    There the ReLU derivative depends on the fp32 rounding of the sum: the kernel and the float64 reference can take different
    branches, and the whole row of g_a0 follows (R = 64, K = 300, D = 256 has a unit at 5e-9 of its sum|terms|).  a0 >= 0.
    This applies to every shape, so the four shapes this test had before the sweep over D also run on moved biases."""
    pre = a0.double() @ W0.double().t()
    mag = a0.double() @ W0.double().abs().t()
    b = b0.double().clone()
    for _ in range(32):
        near = ((pre + b).abs() < margin * (mag + b.abs())).any(0)
        if not bool(near.any()):
            return b.float()
        b[near] += 3 * margin * (mag[:, near].max(0).values + b[near].abs())
    raise AssertionError("no bias clear of the ReLU kink")


@pytest.mark.parametrize("R,K,D", MLP_SHAPES)
def test_head_mlp_and_loss_match_torch(mlg, R, K, D):
    from multilevel_gnn_b200 import functional as Fn
    g = torch.Generator().manual_seed(R + K)
    a0 = torch.randn(R, K, generator=g).abs()
    W0 = torch.randn(D, K, generator=g) / K ** 0.5
    b0 = _clear_of_relu_kink(a0, W0, torch.randn(D, generator=g) * 0.1)
    W3 = torch.randn(2, D, generator=g) / D ** 0.5
    b3 = torch.randn(2, generator=g) * 0.1
    lab = (torch.rand(R, generator=g) < 0.5).long()
    y = F.one_hot(lab, 2).float()
    wt = torch.rand(R, 2, generator=g) + 0.5
    Rw = torch.randn(R, 2, generator=g)
    for use_w in (True, False):
        dev = [t.to(DEV).requires_grad_() for t in (a0, W0, b0, W3, b3)]
        pred, bce = Fn.HeadMLP.apply(*dev, 0.5, False, y.to(DEV), wt.to(DEV) if use_w else None)
        ref_in = [t.double().requires_grad_() for t in (a0, W0, b0, W3, b3)]
        hid = F.relu(F.linear(ref_in[0], ref_in[1], ref_in[2]))
        pr = F.softmax(F.linear(hid, ref_in[3], ref_in[4]), dim=1)
        lr = F.binary_cross_entropy(pr, y.double(), weight=wt.double() if use_w else None)
        assert_close(pred, pr.float(), what="pred")
        assert_close(bce, lr.float(), what="bce")
        gs = torch.autograd.grad((pred * Rw.to(DEV)).sum() + 3.0 * bce, dev)
        gr = torch.autograd.grad((pr * Rw.double()).sum() + 3.0 * lr, ref_in, retain_graph=True)
        for name, a, c in zip(("g_a0", "g_W0", "g_b0", "g_W3", "g_b3"), gs, gr):
            assert_close(a, c.float(), rtol=1e-4, atol=2e-6, what="%s (weight=%s)" % (name, use_w))
        # loss only / pred only
        pred2, bce2 = Fn.HeadMLP.apply(*dev, 0.5, False, y.to(DEV), wt.to(DEV) if use_w else None)
        g_l = torch.autograd.grad(bce2, dev)
        g_lr = torch.autograd.grad(lr, ref_in, retain_graph=True)
        assert_close(g_l[1], g_lr[1].float(), rtol=1e-4, atol=2e-6, what="g_W0 from the loss alone")
        pred3, _ = Fn.HeadMLP.apply(*dev, 0.5, False, None, None)
        g_p = torch.autograd.grad((pred3 * Rw.to(DEV)).sum(), dev)
        g_pr = torch.autograd.grad((pr * Rw.double()).sum(), ref_in)
        assert_close(g_p[0], g_pr[0].float(), rtol=1e-4, atol=2e-6, what="g_a0 from pred alone")


def test_head_mlp_dropout(mlg):
    from multilevel_gnn_b200 import functional as Fn
    R, K, D, p = 16, 500, 128, 0.5
    g = torch.Generator().manual_seed(3)
    a0 = torch.randn(R, K, generator=g).to(DEV).requires_grad_()
    W0 = (torch.randn(D, K, generator=g) / K ** 0.5).to(DEV).requires_grad_()
    b0 = (torch.randn(D, generator=g) * 0.1).to(DEV)
    W3 = (torch.randn(2, D, generator=g) / D ** 0.5).to(DEV)
    b3 = torch.zeros(2, device=DEV)
    torch.manual_seed(9)
    pred, _ = Fn.HeadMLP.apply(a0, W0, b0, W3, b3, p, True, None, None)
    torch.manual_seed(9)
    bits = torch.empty(R * D, dtype=torch.int32, device=DEV).random_()
    mask = (bits >= int(p * 2 ** 31)).double().view(R, D).cpu()
    ar, wr = a0.detach().cpu().double().requires_grad_(), W0.detach().cpu().double().requires_grad_()
    hid = F.relu(F.linear(ar, wr, b0.cpu().double())) * mask / (1 - p)
    ref = F.softmax(F.linear(hid, W3.cpu().double(), b3.cpu().double()), dim=1)
    assert_close(pred, ref.float(), what="mlp dropout pred")
    Rw = torch.randn(pred.shape, generator=g)
    g1 = torch.autograd.grad((pred * Rw.to(DEV)).sum(), [a0, W0])
    g2 = torch.autograd.grad((ref * Rw.double()).sum(), [ar, wr])
    assert_close(g1[0], g2[0].float(), rtol=1e-4, atol=2e-6, what="mlp dropout g_a0")
    assert_close(g1[1], g2[1].float(), rtol=1e-4, atol=2e-6, what="mlp dropout g_W0")


@pytest.mark.parametrize("cfg", ["gbm", "kirc"])
def test_fused_head_equals_module_chain(mlg, cfg):
    """MultilevelGNN with the fused head (default) vs the same model running its conv / pool / Linear modules one by one:
    prediction, BCE loss through forward_with_loss, every parameter gradient (eval mode: dropout off)."""
    from multilevel_gnn_b200 import configs, synth
    args = configs.make_args(cfg)
    torch.manual_seed(3)
    model = mlg.MultilevelGNN(args)
    synth.multilevel_params(model)
    model.to(DEV).eval()
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    b = synth.multilevel_batch(batch_size=4, seed=6).to(DEV)
    params = [p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]
    names = [n for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]
    wt = torch.tensor([[0.8, 1.3]], device=DEV).repeat(4, 1)
    out = []
    for fused in (True, False):
        type(model).FUSED_HEAD = fused
        try:
            pred, feat, bce = model.forward_with_loss(b, b.y.reshape(-1, 2), wt)
            g = torch.autograd.grad(bce + feat.square().mean(), params, allow_unused=True)
        finally:
            type(model).FUSED_HEAD = True
        out.append((pred.detach(), bce.detach(), g))
    assert_close(out[0][0], out[1][0], what="pred")
    assert_close(out[0][1], out[1][1], what="bce")
    for n, a, c in zip(names, out[0][2], out[1][2]):
        if a is None or c is None:
            assert a is None and c is None
            continue
        assert_close(a, c, rtol=2e-4, atol=2e-6, what="grad " + n)
