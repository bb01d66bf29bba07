"""The algebra behind the reformulated SAGE layers, pinned on CPU in fp64 against the oracle restatement of
SAGEConv.forward (oracle/restated.py::sage_forward, torch_vertex.py:269-294) and its autograd gradients:

 * factored first layer (mlg_sage_rank1_fwd_rows / mlg_sage_rank1_bwd_rows): x0[b,n,:] = x[b,n] * emb[n,:] lets the layer run
   through the per-gene tables E_self = emb W1^T, E_nbr = emb (W2 W_r)^T; backward by TARGET row emits per-entry rows h and
   the self / bias reductions, then a segment sum by source;
 * transform-first layer (mlg_gather_sum_act + one dX GEMM): z = U + mean_j(w_ij V_j), [U | V] = x [W1 ; W2 W_r]^T + [b | 0],
   and the ROW-PAIR weight gradient ([G_even | G_odd]^T [x_even | x_odd], diagonal blocks added).

These are plain-torch statements of exactly what the CUDA kernels compute (same index conventions: forward CSR sorted by
target with the added self loop, val = edge weight, 1/cnt_i = PyG's mean divisor); the GPU tests compare the kernels with
the buffered path, this file compares the formulas with the reference order of operations."""
import torch

from oracle import restated as R

torch.manual_seed(0)
DT = torch.float64


def _graph(n, e, g):
    src = torch.randint(0, n, (e,), generator=g)
    dst = torch.randint(0, n, (e,), generator=g)
    w = torch.rand(e, generator=g, dtype=DT) + 0.1
    return torch.stack([src, dst]), w


def _csr_by_target(ei, w, n):
    """Forward CSR as mlg_csr_build(drop_self=1, add_self=1) lays it out: entries sorted by target (stable), the added
    self loop (weight 1) last in its row.  Returns (rowptr, col, val)."""
    keep = ei[0] != ei[1]
    src, dst, ww = ei[0][keep], ei[1][keep], w[keep]
    src = torch.cat([src, torch.arange(n)])
    dst = torch.cat([dst, torch.arange(n)])
    ww = torch.cat([ww, torch.ones(n, dtype=DT)])
    order = torch.sort(dst, stable=True).indices
    col, val, d = src[order], ww[order], dst[order]
    rowptr = torch.searchsorted(d, torch.arange(n + 1))
    return rowptr, col, val, d


def _params(cin, cout, g):
    sd = {"gconv.lin_r.weight": torch.randn(cout, cin, generator=g, dtype=DT) * 0.3,
          "gconv.nn.0.weight": torch.randn(cout, cin + cout, generator=g, dtype=DT) * 0.3,
          "gconv.nn.0.bias": torch.randn(cout, generator=g, dtype=DT) * 0.1}
    return {k: v.requires_grad_() for k, v in sd.items()}


def _stacked(sd, cin):
    """[W1 ; W2 W_r]  [2 cout, cin] -- what mlg_sage_fold_fwd produces (as [W1 | W2 W_r]) re-stacked."""
    w_nn, w_r = sd["gconv.nn.0.weight"], sd["gconv.lin_r.weight"]
    return torch.cat([w_nn[:, :cin], w_nn[:, cin:] @ w_r], 0)


def _replicate(ei, w, n, B):
    eis = torch.cat([ei + b * n for b in range(B)], 1)
    return eis, w.repeat(B)


def test_factored_first_layer_forward_and_backward_by_rows():
    g = torch.Generator().manual_seed(1)
    n, e, B, cin, cout = 37, 160, 5, 6, 4
    ei, w = _graph(n, e, g)
    sd = _params(cin, cout, g)
    emb = torch.randn(n, cin, generator=g, dtype=DT).requires_grad_()
    xs = torch.randn(B, n, generator=g, dtype=DT)
    # reference order on the materialised x0 over the B stacked copies of the graph
    eis, ws = _replicate(ei, w, n, B)
    x0 = (xs.reshape(-1, 1) * emb.repeat(B, 1))
    y_ref = R.sage_forward(sd, x0, eis, ws)
    go = torch.randn(y_ref.shape, generator=g, dtype=DT)
    grads_ref = torch.autograd.grad(y_ref, [emb] + list(sd.values()), go)

    # factored forward
    rowptr, col, val, dst = _csr_by_target(ei, w, n)
    cnt = (rowptr[1:] - rowptr[:-1]).to(DT)
    wst = _stacked({k: v.detach() for k, v in sd.items()}, cin)
    e12 = emb.detach() @ wst.t()
    e_self, e_nbr = e12[:, :cout], e12[:, cout:]
    bias = sd["gconv.nn.0.bias"].detach()
    z = torch.empty(B, n, cout, dtype=DT)
    for b in range(B):
        contrib = val[:, None] * xs[b, col][:, None] * e_nbr[col]                      # per entry
        agg = torch.zeros(n, cout, dtype=DT).index_add_(0, dst, contrib) / cnt[:, None]
        z[b] = xs[b][:, None] * e_self + agg + bias
    y = torch.nn.functional.leaky_relu(z, 0.2).reshape(B * n, cout)
    torch.testing.assert_close(y, y_ref.detach(), rtol=1e-10, atol=1e-12)

    # backward by target row: gz = dL/dz; h[q] = val_q / cnt_i * sum_b xs[b, col_q] gz[b, i, :]; segment sum by source
    gz = (go * torch.where(y_ref.detach() > 0, torch.ones((), dtype=DT), torch.full((), 0.2, dtype=DT))).reshape(B, n, cout)
    g_self = torch.einsum("bn,bnc->nc", xs, gz)
    g_bias = gz.sum((0, 1))
    h = (val / cnt[dst])[:, None] * torch.einsum("bq,bqc->qc", xs[:, col], gz[:, dst])
    g_nbr = torch.zeros(n, cout, dtype=DT).index_add_(0, col, h)
    g12 = torch.cat([g_self, g_nbr], 1)
    g_emb = g12 @ wst
    g_wst = g12.t() @ emb.detach()
    w_nn, w_r = sd["gconv.nn.0.weight"].detach(), sd["gconv.lin_r.weight"].detach()
    g_w1, g_w2p = g_wst[:cout], g_wst[cout:]
    g_wnn = torch.cat([g_w1, g_w2p @ w_r.t()], 1)               # mlg_sage_fold_bwd
    g_wr = w_nn[:, cin:].t() @ g_w2p
    for got, ref, what in zip([g_emb, g_wr, g_wnn, g_bias], grads_ref, ["emb", "lin_r", "nn.0.weight", "nn.0.bias"]):
        torch.testing.assert_close(got, ref, rtol=1e-9, atol=1e-11, msg=lambda m, what=what: what + ": " + m)


def test_transform_first_layer_and_row_pair_weight_gradient():
    g = torch.Generator().manual_seed(2)
    n, e, B, cin, cout = 41, 200, 4, 8, 4
    ei, w = _graph(n, e, g)
    sd = _params(cin, cout, g)
    x = torch.randn(B * n, cin, generator=g, dtype=DT).requires_grad_()
    eis, ws = _replicate(ei, w, n, B)
    y_ref = R.sage_forward(sd, x, eis, ws)
    go = torch.randn(y_ref.shape, generator=g, dtype=DT)
    grads_ref = torch.autograd.grad(y_ref, [x] + list(sd.values()), go)

    rowptr, col, val, dst = _csr_by_target(ei, w, n)
    cnt = (rowptr[1:] - rowptr[:-1]).to(DT)
    sdd = {k: v.detach() for k, v in sd.items()}
    wst = _stacked(sdd, cin)
    bias2 = torch.cat([sdd["gconv.nn.0.bias"], torch.zeros(cout, dtype=DT)])
    uv = (x.detach() @ wst.t() + bias2).reshape(B, n, 2 * cout)
    u, v = uv[..., :cout], uv[..., cout:]
    agg = torch.zeros(B, n, cout, dtype=DT).index_add_(1, dst, val[None, :, None] * v[:, col]) / cnt[None, :, None]
    y = torch.nn.functional.leaky_relu(u + agg, 0.2).reshape(B * n, cout)
    torch.testing.assert_close(y, y_ref.detach(), rtol=1e-10, atol=1e-12)

    # backward: G = [gz | A^T gz] (by-source aggregation of the cout-wide gradient), ONE dX GEMM, row-pair weight gradient
    gz = (go * torch.where(y_ref.detach() > 0, torch.ones((), dtype=DT), torch.full((), 0.2, dtype=DT))).reshape(B, n, cout)
    g_v = torch.zeros(B, n, cout, dtype=DT).index_add_(1, col, (val / cnt[dst])[None, :, None] * gz[:, dst])
    G = torch.cat([gz, g_v], -1).reshape(B * n, 2 * cout)
    g_x = G @ wst
    assert (B * n) % 2 == 0
    o2 = G.reshape(B * n // 2, 4 * cout).t() @ x.detach().reshape(B * n // 2, 2 * cin)       # [4cout, 2cin]
    g_wst = o2[:2 * cout, :cin] + o2[2 * cout:, cin:]
    torch.testing.assert_close(g_wst, G.t() @ x.detach(), rtol=1e-10, atol=1e-12)
    cs2 = G.reshape(B * n // 2, 4 * cout).sum(0)
    g_bias = cs2[:cout] + cs2[2 * cout:3 * cout]
    w_nn, w_r = sdd["gconv.nn.0.weight"], sdd["gconv.lin_r.weight"]
    g_wnn = torch.cat([g_wst[:cout], g_wst[cout:] @ w_r.t()], 1)
    g_wr = w_nn[:, cin:].t() @ g_wst[cout:]
    for got, ref, what in zip([g_x, g_wr, g_wnn, g_bias], grads_ref, ["x", "lin_r", "nn.0.weight", "nn.0.bias"]):
        torch.testing.assert_close(got, ref, rtol=1e-9, atol=1e-11, msg=lambda m, what=what: what + ": " + m)


def test_pca_indep_segment_formula():
    """mlg_pca_indep_loss's per-segment form vs the reference's loop (multilevel_gnn.py:336-346: only the last j of every i
    survives) as restated in MultilevelGNN.get_feature_loss."""
    g = torch.Generator().manual_seed(3)
    G, nseg, P = 300, 17, 3
    idx = torch.sort(torch.randint(0, nseg, (G,), generator=g)).values
    w = torch.randn(G, P, generator=g, dtype=DT)
    a, b = w[:, :P - 1], w[:, P - 1:P]
    seg = torch.zeros(nseg, 2 * (P - 1) + 1, dtype=DT).index_add_(0, idx, torch.cat([a * b, a * a, b * b], 1))
    mul, ln = seg[:, :P - 1], torch.sqrt(seg[:, P - 1:2 * (P - 1)] * seg[:, 2 * (P - 1):])
    ref = torch.abs(mul / (ln + 1e-7)).mean(0).sum() / (P * (P - 1) // 2)
    segptr = torch.searchsorted(idx, torch.arange(nseg + 1))
    tot = torch.zeros((), dtype=DT)
    for s in range(nseg):
        sl = slice(int(segptr[s]), int(segptr[s + 1]))
        bb = (w[sl, P - 1] ** 2).sum()
        for i in range(P - 1):
            tot = tot + torch.abs((w[sl, i] * w[sl, P - 1]).sum() / (torch.sqrt((w[sl, i] ** 2).sum() * bb) + 1e-7))
    torch.testing.assert_close(tot / (nseg * (P * (P - 1) // 2)), ref, rtol=1e-12, atol=1e-14)
