"""The kernels and the training step at the batch widths the benchmark runs (32 graphs for gbm, 64 for kirc / lgg, 256 for the
strong-scaling leg on one GPU) and at the widths next to them, against float64.

The kernels choose their code path from the number of replicas B:

* ``sage_rank1_fwd_rows_kernel`` (sage_rank1.cu:235-246, 296-299) walks blocks of 32 replicas; a full block takes the packed
  replica-pair pass when B % 4 == 0 (scalar FULL pass otherwise), a partial tail block the scalar pass.  B = 31, 33: scalar
  only; 32, 64, 96, 256: packed only; 36: one packed block and a 4-replica tail.
* ``sage_rank1_bwd_rows_kernel<2, true>`` (gather_sum.cu:976) runs only when B % 32 == 0 and the node values come transposed;
  replica blocks after the first ACCUMULATE into g_self, g_bias_rows and h (gather_sum.cu:611-612, 670).  B = 64, 96, 256
  reach those accumulations on the packed path, 33 and 36 on the scalar one.
* ``gather_nm_kernel`` (gather_sum.cu:715-728): 16 replicas per warp, ceil(B / 16) warps per row, the last one clamped: B = 15
  and 17 end in a partial warp, 16, 32, 64 and 256 do not, 40 ends at 8 of 16.
* ``sage_rank1_bwd_xs`` (input_grad.cu:70, 188): blocks of 32 replicas, at most 64: B = 31 (one partial block), 32 (one full),
  33 (a 1-replica second block), 64 (two full).

Every element is held to |got - ref| <= C_TOL * k * 2^-24 * sum|terms|, k the length of that element's sum (plus the few
roundings of the scale factors), sum|terms| computed in float64 from the absolute values of the operands: one wrong replica
row, pair half or tail clamp fails the test whatever the rest of the tensor does.  LeakyReLU takes the branch the kernel took
(its output's sign, or the gradient mask the test gave it), so no element is excused as a branch flip.  Outputs are
pre-filled with NaN, so a row the kernel does not write fails too.

The second half checks the whole model at those widths against the float64 oracle (oracle/restated.py).  The oracle runs over
chunks of at most ORACLE_CHUNK graphs: graphs do not interact in the forward pass, and the shipped loss is the BCE mean over
rows plus an independence term on detached pathway weights (pca_loss off), so the gradient of the whole batch is the sum of
the chunks' gradients weighted by n_chunk / B.  A float64 pass over 256 full-size graphs at once would need more than 60 GB of
host memory; a chunk of 16 needs about 5 GB.  test_chunked_oracle_equals_one_pass (no GPU) shows the chunking is exact.
"""
import ctypes
import types

import pytest
import torch

from conftest import assert_close_flips as _check
from oracle import restated as R

DEV = "cuda:0"
EPS = 2.0 ** -24
C_TOL = 2.0            # c of the element-wise bound c * k * 2^-24 * sum|terms|
SLOPE = 0.2
ORACLE_CHUNK = 16      # graphs per float64 oracle pass


# ---------------------------------------------------------------------------------------------------------------------
# float64 oracle over chunks of graphs
# ---------------------------------------------------------------------------------------------------------------------
def graph_slice(batch, g0, g1, n, dtype=None):
    """Graphs g0 .. g1-1 of a PyG-collated multilevel batch (graph-major nodes, n per graph; edges never leave a graph) as a
    batch of their own, node ids renumbered from 0; floating-point fields cast to ``dtype`` when given."""
    ei = batch.edge_index
    keep = (ei[1] >= g0 * n) & (ei[1] < g1 * n)
    out = types.SimpleNamespace(x=batch.x[g0 * n:g1 * n], edge_index=ei[:, keep] - g0 * n, edge_attr=batch.edge_attr[keep],
                                gene_pca_match=batch.gene_pca_match[g0:g1], raw_indice=batch.raw_indice[g0:g1],
                                age=batch.age[g0:g1])
    if getattr(batch, "y", None) is not None:
        out.y = batch.y[2 * g0:2 * g1]
    if getattr(batch, "batch", None) is not None:
        out.batch = batch.batch[g0 * n:g1 * n] - g0
    if getattr(batch, "reorder_idxs", None) is not None:
        out.reorder_idxs = batch.reorder_idxs
    if dtype is not None:
        for k in ("x", "edge_attr", "age", "y"):
            if hasattr(out, k):
                setattr(out, k, getattr(out, k).to(dtype))
    return out


def oracle_params(sd, names, dtype=torch.float64):
    """The model's state dict as oracle leaves in ``dtype``; the entries named in ``names`` require gradients."""
    out = {}
    for k, v in sd.items():
        v = v.detach().to(dtype).clone() if v.is_floating_point() else v.detach()
        out[k] = v.requires_grad_() if k in names else v
    return out


def forward_chunks(leaf, batch, args, n, chunk=ORACLE_CHUNK, dtype=torch.float64, input_grad=False, pool_arg=None):
    """Yields (g0, g1, chunk batch, pred, pca_feature, acts) of oracle.multilevel_forward over graphs g0 .. g1-1, for
    consecutive chunks of at most ``chunk`` graphs.  input_grad: the chunk's x and age require gradients.  pool_arg: the head
    max-pool's choice per window for the whole batch (oracle.multilevel_forward), sliced per chunk."""
    B = batch.age.shape[0]
    for g0 in range(0, B, chunk):
        g1 = min(B, g0 + chunk)
        cb = graph_slice(batch, g0, g1, n, dtype)
        if input_grad:
            cb.x = cb.x.clone().requires_grad_()
            cb.age = cb.age.clone().requires_grad_()
        pred, feat, acts = R.multilevel_forward(leaf, cb, args, return_acts=True,
                                                pool_arg=None if pool_arg is None else pool_arg[g0:g1])
        yield g0, g1, cb, pred, feat, acts


def train_oracle(leaf, names, batch, args, n, pathway_indexs, weight=None, chunk=ORACLE_CHUNK, dtype=torch.float64,
                 visit=None, pool_arg=None):
    """Loss and gradients (one per name, None when unused) of BCE(weight) + feature loss, the training objective of the shipped
    configs, accumulated over chunks of graphs: the batch's BCE mean is the sum of the chunks' means weighted by n_chunk / B.
    visit(g0, g1, pred, pca_feature, acts) sees each chunk's forward values (detached)."""
    assert not args.pca_loss, "the pca_loss term couples the graphs of a batch: no chunked oracle for it"
    B = batch.age.shape[0]
    params = [leaf[k] for k in names]
    grads = [None] * len(params)

    def add(part):
        for i, g in enumerate(torch.autograd.grad(part, params, allow_unused=True)):
            if g is not None:
                grads[i] = g if grads[i] is None else grads[i] + g

    fl = R.feature_loss(None, leaf["learnable_pca_params"], leaf["info_mask"], pathway_indexs, pca_loss=False,
                        pca_indep_loss=args.pca_indep_loss)
    fl = torch.as_tensor(fl, dtype=dtype)
    if fl.requires_grad:
        add(fl)
    loss = fl.detach()
    for g0, g1, cb, pred, feat, acts in forward_chunks(leaf, batch, args, n, chunk, dtype, pool_arg=pool_arg):
        w = None if weight is None else weight[g0:g1].to(dtype)
        part = R.bce_loss(pred, cb.y.reshape(-1, 2), w) * ((g1 - g0) / B)
        if visit is not None:
            visit(g0, g1, pred.detach(), feat.detach(), {k: v.detach() for k, v in acts.items()})
        add(part)
        loss = loss + part.detach()
    return loss, grads


def test_chunked_oracle_equals_one_pass():
    """The chunked float64 oracle (chunks of 2, 2 and 1 graphs) gives the loss, every parameter gradient, pred, pca_feature
    and the layer activations of one float64 pass over the same 5 graphs."""
    from multilevel_gnn_b200 import configs, synth
    from multilevel_gnn_b200.models.multilevel_gnn import MultilevelGNN
    args = configs.make_args("gbm")
    torch.manual_seed(3)
    model = MultilevelGNN(args)
    synth.multilevel_params(model, seed=3)
    batch = synth.multilevel_batch(batch_size=5, seed=3)
    weight = torch.rand(5, 2, generator=torch.Generator().manual_seed(3)) + 0.5
    n = 3 * MultilevelGNN.GENES
    names = [k for k, p in model.named_parameters() if p.requires_grad and not k.endswith("lin_l.weight")]
    sd = model.state_dict()
    runs = []
    for chunk in (5, 2):
        seen = {}

        def visit(g0, g1, pred, feat, acts):
            seen[g0] = (pred, feat, acts)

        loss, grads = train_oracle(oracle_params(sd, names), names, batch, args, n, model.pathway_indexs, weight, chunk=chunk,
                                   visit=visit)
        keys = sorted(seen)
        assert keys == list(range(0, 5, chunk))
        fwd = [torch.cat([seen[k][0] for k in keys]), torch.cat([seen[k][1] for k in keys])]
        fwd += [torch.cat([seen[k][2][a] for k in keys]) for a in sorted(seen[0][2])]
        runs.append((loss, grads, fwd))
    (l1, g1, f1), (l2, g2, f2) = runs
    assert l1.dtype == torch.float64
    torch.testing.assert_close(l2, l1, rtol=1e-12, atol=0)
    assert any(g is not None for g in g1)
    for k, a, b in zip(names, g2, g1):
        assert (a is None) == (b is None), k
        if a is not None:
            torch.testing.assert_close(a, b, rtol=1e-10, atol=1e-12 * float(b.abs().max()), msg=k)
    for a, b in zip(f2, f1):
        torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-14)


# ---------------------------------------------------------------------------------------------------------------------
# kernel-level checks at the dispatch widths
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L():
    from multilevel_gnn_b200 import _cabi
    return _cabi.lib()


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _sp():
    from multilevel_gnn_b200 import _cabi
    return _cabi.stream_ptr()


def _ok(rc, who):
    from multilevel_gnn_b200 import _cabi
    _cabi.check(rc, who)


def _within(got, ref, k, mag, what):
    """|got - ref| <= C_TOL * k * 2^-24 * mag element-wise (NaN fails)."""
    got = got.detach().cpu().double()
    assert got.shape == ref.shape, "%s: shape %s vs %s" % (what, tuple(got.shape), tuple(ref.shape))
    err = (got - ref).abs()
    tol = C_TOL * EPS * k * mag
    bad = ~(err <= tol)
    if bool(bad.any()):
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError("%s: %d/%d elements outside c*k*2^-24*sum|terms|; first at %s: got %r, ref %r, tol %.3e" % (
            what, int(bad.sum()), got.numel(), i, float(got[i]), float(ref[i]), float(tol[i])))


class _Csr:
    """A hand-built CSR over n rows: row 0 a hub of 100 entries (four 32-entry batches, the last one partial), row 7 empty
    (1 / cnt = 0), the other rows 1..12 entries (every EU = 4 tail length), non-unit edge values of both signs, duplicate
    entries allowed; a shuffled row order; the by-source CSR of entry positions."""

    def __init__(self, n=300, seed=0):
        g = torch.Generator().manual_seed(seed)
        cnt = torch.randint(1, 13, (n,), generator=g)
        cnt[0], cnt[7] = 100, 0
        self.n = n
        self.cnt = cnt
        self.rowptr = torch.cat([torch.zeros(1, dtype=torch.long), cnt.cumsum(0)])
        self.cap = int(self.rowptr[-1])
        self.idx = torch.randint(0, n, (self.cap,), generator=g)
        self.val = (torch.rand(self.cap, generator=g) * 1.6 + 0.2) * torch.where(torch.rand(self.cap, generator=g) < 0.25, -1.0, 1.0)
        self.order = torch.randperm(n, generator=g)
        self.row_of = torch.repeat_interleave(torch.arange(n), cnt)
        self.inv = torch.where(cnt > 0, 1.0 / cnt.clamp(min=1).double(), torch.zeros((), dtype=torch.float64))
        self.A = torch.zeros(n, n, dtype=torch.float64).index_put_((self.row_of, self.idx), self.val.double(), accumulate=True)
        self.Aabs = torch.zeros(n, n, dtype=torch.float64).index_put_((self.row_of, self.idx), self.val.double().abs(), accumulate=True)
        by_src = torch.sort(self.idx, stable=True).indices
        self.rowptr_t = torch.cat([torch.zeros(1, dtype=torch.long), torch.bincount(self.idx, minlength=n).cumsum(0)])
        self.fwd_pos_t = by_src
        d = lambda t: t.to(torch.int32).to(DEV)
        self.d_rowptr, self.d_idx, self.d_order = d(self.rowptr), d(self.idx), d(self.order)
        self.d_rowptr_t, self.d_fwd_pos_t = d(self.rowptr_t), d(self.fwd_pos_t)
        self.d_val = self.val.to(DEV)


def _layout(t, B, n, node_major):
    """[B, n, C] -> rows (b, i) at b * n + i (graph-major) or i * B + b (node-major)."""
    return (t.transpose(0, 1) if node_major else t).reshape(B * n, t.shape[-1]).contiguous()


def _unlayout(t, B, n, node_major):
    C = t.shape[-1]
    return t.view(n, B, C).transpose(0, 1) if node_major else t.view(B, n, C)


def _bit_pos(C):
    c = torch.arange(C)
    return 16 * (c % 4) + c // 4


def _sign_words(y_nbc):
    """[n, B, 64] -> the forward kernel's [n, B] int64 sign words: channel c at bit 16 * (c % 4) + c / 4 (sage_rank1.cu:106-108)."""
    w = torch.zeros(y_nbc.shape[:2], dtype=torch.int64)
    for c, p in enumerate(_bit_pos(64).tolist()):
        w |= (y_nbc[:, :, c] > 0).to(torch.int64) << p
    return w


WIDTHS = [31, 32, 33, 36, 64, 96, 256]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [64, 32])
@pytest.mark.parametrize("B", WIDTHS)
def test_sage_rank1_fwd_rows_at_batch_widths(L, B, C):
    """mlg_sage_rank1_fwd_rows and _nm (graph-major and node-major output) against float64; with C = 64 every sign bit equals
    out > 0 of the kernel's own output in the documented layout."""
    csr = _Csr(seed=B + C)
    n = csr.n
    g = torch.Generator().manual_seed(B * C)
    xs = torch.randn(B, n, generator=g)
    e12 = torch.randn(n, 2 * C, generator=g)           # [E_self | E_nbr], leading dimension 2C as the model passes them
    bias = torch.randn(C, generator=g) * 0.3
    es, en = e12[:, :C].double(), e12[:, C:].double()
    xd = xs.double()
    T = xd[:, :, None] * en[None]                     # [B, n, C]: xs[b, j] E_nbr[j]
    agg = csr.inv[None, :, None] * torch.matmul(csr.A, T)
    agg_mag = csr.inv[None, :, None] * torch.matmul(csr.Aabs, T.abs())
    z = xd[:, :, None] * es[None] + agg + bias.double()
    mag = (xd[:, :, None] * es[None]).abs() + agg_mag + bias.double().abs()
    k = (csr.cnt.double() + 4)[None, :, None]
    xs_t = xs.t().contiguous().to(DEV)
    e12_d, bias_d = e12.to(DEV), bias.to(DEV)
    for nm, fn in ((0, L.mlg_sage_rank1_fwd_rows), (1, L.mlg_sage_rank1_fwd_rows_nm)):
        out = torch.full((B * n, C), float("nan"), device=DEV)
        bits = torch.zeros(n * B, dtype=torch.int64, device=DEV) if C == 64 else None
        with torch.cuda.device(DEV):
            _ok(fn(_vp(xs_t), _vp(e12_d), 2 * C, _vp(e12_d[:, C:]), 2 * C, _vp(csr.d_rowptr), _vp(csr.d_idx), _vp(csr.d_val),
                   _vp(csr.d_order), n, C, B, _vp(bias_d), SLOPE, _vp(out), C, None if bits is None else _vp(bits), _sp()),
                "mlg_sage_rank1_fwd_rows")
        y = _unlayout(out.cpu(), B, n, nm)
        pos = y > 0                                    # the branch the kernel took
        ref = torch.where(pos, z, SLOPE * z)
        _within(y, ref, k, torch.where(pos, mag, SLOPE * mag), "fwd_rows B=%d C=%d nm=%d" % (B, C, nm))
        if bits is not None:
            w = bits.cpu().view(n, B)
            got = (w[:, :, None] >> _bit_pos(64)[None, None, :]) & 1
            assert torch.equal(got.bool(), pos.transpose(0, 1)), "sign bits B=%d nm=%d" % (B, nm)


def _grad_inputs(B, n, C, seed):
    """gz, y (signs ~ half / half) and the LeakyReLU'(y) mask, each [B, n, C]."""
    g = torch.Generator().manual_seed(seed)
    gz = torch.randn(B, n, C, generator=g)
    y = torch.randn(B, n, C, generator=g)
    return gz, y, torch.where(y > 0, 1.0, SLOPE).double()


def _mask_modes(C):
    return ["bits", "y", "none"] if C == 64 else ["y", "none"]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [64, 32])
@pytest.mark.parametrize("B", WIDTHS)
def test_sage_rank1_bwd_rows_at_batch_widths(L, B, C):
    """mlg_sage_rank1_bwd_rows and _nm: h, g_self and g_bias_rows against float64, with the node values transposed and not,
    and gz taken as dL/dz or as dL/dy with LeakyReLU' from sign bits or from y (the reference applies that same mask)."""
    csr = _Csr(seed=3 * B + C)
    n = csr.n
    gz, y, m = _grad_inputs(B, n, C, B + 7 * C)
    xs = torch.randn(B, n, generator=torch.Generator().manual_seed(B))
    xd = xs.double()
    w_q = csr.val.double() * csr.inv[csr.row_of]       # val_q / cnt_i
    xs_d, xs_t_d = xs.contiguous().to(DEV), xs.t().contiguous().to(DEV)
    for mode in _mask_modes(C):
        g = gz.double() * (m if mode != "none" else 1.0)
        M = torch.einsum("bj,bic->jic", xd, g)                      # sum_b xs[b, j] g[b, i, :]
        Mabs = torch.einsum("bj,bic->jic", xd.abs(), g.abs())
        h_ref = w_q[:, None] * M[csr.idx, csr.row_of]
        h_mag = w_q.abs()[:, None] * Mabs[csr.idx, csr.row_of]
        gs_ref = torch.einsum("bi,bic->ic", xd, g)
        gs_mag = torch.einsum("bi,bic->ic", xd.abs(), g.abs())
        gb_ref, gb_mag = g.sum(0), g.abs().sum(0)
        for nm, fn in ((0, L.mlg_sage_rank1_bwd_rows), (1, L.mlg_sage_rank1_bwd_rows_nm)):
            gz_d = _layout(gz, B, n, nm).to(DEV)
            y_d = _layout(y, B, n, nm).to(DEV) if mode == "y" else None
            bits = _sign_words(y.transpose(0, 1)).reshape(-1).to(DEV) if mode == "bits" else None
            for xs_transposed in (1, 0):
                tag = "bwd_rows B=%d C=%d nm=%d xs_t=%d mask=%s" % (B, C, nm, xs_transposed, mode)
                h = torch.full((csr.cap, C), float("nan"), device=DEV)
                g12 = torch.full((n, 2 * C), float("nan"), device=DEV)     # g_self in the left half (ld 2C, as the model)
                gbr = torch.full((n, C), float("nan"), device=DEV)
                with torch.cuda.device(DEV):
                    _ok(fn(_vp(gz_d), C, None if y_d is None else _vp(y_d), None if bits is None else _vp(bits), SLOPE,
                           _vp(xs_t_d if xs_transposed else xs_d), xs_transposed, _vp(csr.d_rowptr), _vp(csr.d_idx),
                           _vp(csr.d_val), _vp(csr.d_order), n, C, B, _vp(h), _vp(g12), 2 * C, _vp(gbr), _sp()),
                        "mlg_sage_rank1_bwd_rows")
                _within(h.cpu(), h_ref, B + 3, h_mag, tag + " h")
                _within(g12[:, :C].cpu(), gs_ref, B, gs_mag, tag + " g_self")
                assert bool(torch.isnan(g12[:, C:]).all()), tag + ": wrote outside g_self's C columns"
                _within(gbr.cpu(), gb_ref, B, gb_mag, tag + " g_bias_rows")


@pytest.mark.gpu
@pytest.mark.parametrize("C", [64, 32])
@pytest.mark.parametrize("B", [31, 32, 33, 64])
def test_sage_rank1_bwd_xs_at_batch_widths(L, B, C):
    """mlg_sage_rank1_bwd_xs: g_xs[b, j] = <g[b, j], E_self[j]> + sum_{(i, q): idx_q = j} (val_q / cnt_i) <g[b, i], E_nbr[j]>
    against float64, gz graph-major and node-major, dL/dz or dL/dy with the mask from sign bits or from y."""
    csr = _Csr(seed=5 * B + C)
    n = csr.n
    gz, y, m = _grad_inputs(B, n, C, 11 * B + C)
    e12 = torch.randn(n, 2 * C, generator=torch.Generator().manual_seed(C + B))
    es, en = e12[:, :C].double(), e12[:, C:].double()
    w_q = csr.val.double() * csr.inv[csr.row_of]
    W = torch.zeros(n, n, dtype=torch.float64).index_put_((csr.row_of, csr.idx), w_q, accumulate=True)
    Wabs = torch.zeros(n, n, dtype=torch.float64).index_put_((csr.row_of, csr.idx), w_q.abs(), accumulate=True)
    indeg = torch.bincount(csr.idx, minlength=n).double()
    e12_d = e12.to(DEV)
    ws_bytes = L.mlg_sage_rank1_bwd_xs_workspace_bytes(csr.cap, n, B)
    for mode in _mask_modes(C):
        g = gz.double() * (m if mode != "none" else 1.0)
        D = torch.einsum("bic,jc->bij", g, en)
        Dabs = torch.einsum("bic,jc->bij", g.abs(), en.abs())
        ref = (g * es[None]).sum(2) + (W[None] * D).sum(1)
        mag = (g * es[None]).abs().sum(2) + (Wabs[None] * Dabs).sum(1)
        for nm in (0, 1):
            gz_d = _layout(gz, B, n, nm).to(DEV)
            y_d = _layout(y, B, n, nm).to(DEV) if mode == "y" else None
            bits = _sign_words(y.transpose(0, 1)).reshape(-1).to(DEV) if mode == "bits" else None
            g_xs = torch.full((B * n,), float("nan"), device=DEV)
            ws = torch.empty(ws_bytes // 4, device=DEV)
            with torch.cuda.device(DEV):
                _ok(L.mlg_sage_rank1_bwd_xs(_vp(gz_d), C, nm, None if y_d is None else _vp(y_d), None if bits is None else _vp(bits),
                                            SLOPE, _vp(e12_d), 2 * C, _vp(e12_d[:, C:]), 2 * C, _vp(csr.d_rowptr), _vp(csr.d_idx),
                                            _vp(csr.d_val), _vp(csr.d_order), _vp(csr.d_rowptr_t), _vp(csr.d_fwd_pos_t), n, csr.cap,
                                            C, B, _vp(g_xs), _vp(ws), ws_bytes, _sp()), "mlg_sage_rank1_bwd_xs")
            _within(g_xs.cpu().view(B, n), ref, (C + indeg + 3)[None], mag,
                    "bwd_xs B=%d C=%d nm=%d mask=%s" % (B, C, nm, mode))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [15, 16, 17, 32, 40, 64, 256])
def test_gather_sum_nm_at_batch_widths(L, B):
    """mlg_gather_sum_nm_ex in both of the model's forms against float64.  Forward (transform-first layer on a node-major
    [U | V]): out = LeakyReLU(U + mean_q val_q V[idx_q]), graph-major output.  Backward: out = sum_q val_q pre[idx_q] gz[idx_q]
    with the row's own gz copied to self_out, output node-major and graph-major."""
    C = 32
    csr = _Csr(seed=B)
    n = csr.n
    g = torch.Generator().manual_seed(100 + B)
    uv = torch.randn(B, n, 2 * C, generator=g)
    U, V = uv[..., :C].double(), uv[..., C:].double()
    z = U + csr.inv[None, :, None] * torch.matmul(csr.A, V)
    mag = U.abs() + csr.inv[None, :, None] * torch.matmul(csr.Aabs, V.abs())
    k = (csr.cnt.double() + 3)[None, :, None]
    uv_d = _layout(uv, B, n, True).to(DEV)
    out = torch.full((B * n, C), float("nan"), device=DEV)
    with torch.cuda.device(DEV):
        _ok(L.mlg_gather_sum_nm_ex(_vp(uv_d[:, C:]), 2 * C, _vp(csr.d_rowptr), _vp(csr.d_idx), _vp(csr.d_val), None,
                                   _vp(csr.d_order), n, B, 1, _vp(uv_d), 2 * C, 1, SLOPE, _vp(out), C, None, 0, 0, _sp()),
            "mlg_gather_sum_nm_ex")
    y = _unlayout(out.cpu(), B, n, False)
    pos = y > 0
    _within(y, torch.where(pos, z, SLOPE * z), k, torch.where(pos, mag, SLOPE * mag), "gather_nm forward B=%d" % B)
    # backward form
    gz = torch.randn(B, n, C, generator=g)
    pre = torch.rand(n, generator=g) + 0.05
    wq = csr.val.double() * pre.double()[csr.idx]
    Wm = torch.zeros(n, n, dtype=torch.float64).index_put_((csr.row_of, csr.idx), wq, accumulate=True)
    Wabs = torch.zeros(n, n, dtype=torch.float64).index_put_((csr.row_of, csr.idx), wq.abs(), accumulate=True)
    ref = torch.matmul(Wm, gz.double())
    mag = torch.matmul(Wabs, gz.double().abs())
    gz_d, pre_d = _layout(gz, B, n, True).to(DEV), pre.to(DEV)
    for out_nm in (1, 0):
        g_uv = torch.full((B * n, 2 * C), float("nan"), device=DEV)
        with torch.cuda.device(DEV):
            _ok(L.mlg_gather_sum_nm_ex(_vp(gz_d), C, _vp(csr.d_rowptr), _vp(csr.d_idx), _vp(csr.d_val), _vp(pre_d),
                                       _vp(csr.d_order), n, B, 0, None, 0, 0, 0.0, _vp(g_uv[:, C:]), 2 * C, _vp(g_uv), 2 * C,
                                       out_nm, _sp()), "mlg_gather_sum_nm_ex")
        got = _unlayout(g_uv.cpu(), B, n, out_nm)
        _within(got[..., C:], ref, (csr.cnt.double() + 2)[None, :, None], mag, "gather_nm backward B=%d out_nm=%d" % (B, out_nm))
        assert torch.equal(got[..., :C], gz), "gather_nm self_out B=%d out_nm=%d" % (B, out_nm)


# ---------------------------------------------------------------------------------------------------------------------
# the benchmark's own path: a captured Trainer step against the float64 oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bsz", [32, 256])
def test_captured_train_step_vs_fp64_oracle(bsz, monkeypatch):
    """gbm's captured Trainer step (bench.py's resident leg: batch from data.collate + FoldTopology, criterion weight, one CUDA
    graph for forward, loss, backward and Adam) with dropout p = 0: the loss of one replay and every p.grad it leaves in the
    gradient bucket (what --dump-outputs writes) against the float64 oracle at the parameters just before that replay.

    Above 64 graphs the head runs as the module chain (MultilevelGNN._fused_head_ok), whose max-pool records the element each
    window took; an eager step at the same parameters must give the replay's gradients bit for bit, and the oracle takes the
    max-pool windows' elements from it.  Without that, a window whose two largest values lie within fp32 rounding of each
    other routes its gradient to another pixel in float64: 3 of 1.77 M windows at B = 256 move dL/dpca_feature of a plain
    fp32 evaluation of the head by 9e-4 of its norm, and every gradient upstream with it."""
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import functional as Fn
    from multilevel_gnn_b200.train import Trainer
    m._cabi.lib()
    args = m.configs.make_args("gbm")
    torch.manual_seed(0)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model)
    for mod in model.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    model.to(DEV)
    model.pathway_indexs = model.pathway_indexs.to(DEV)
    raw = m.synth.multilevel_batch(batch_size=bsz, seed=100)
    n1 = 3 * m.MultilevelGNN.GENES
    e1 = raw.edge_index.shape[1] // bsz
    topo = m.data.FoldTopology(raw.edge_index[:, :e1], raw.edge_attr[:e1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    patients = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(bsz)]
    resident = m.data.to_device(m.data.collate(patients, topo, pin=False), topo, DEV)
    weight = torch.tensor([[0.8, 1.3]]).repeat(bsz, 1)
    tr = Trainer(model, args, weight.to(DEV))
    for _ in range(3):
        tr.step(resident)
    tr.capture(resident)
    tr.step()
    torch.cuda.synchronize()
    names = [k for k, p in model.named_parameters() if p.requires_grad and not k.endswith("lin_l.weight")]
    snap = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    loss = tr.step()
    torch.cuda.synchronize()
    params = dict(model.named_parameters())
    got = {k: params[k].grad.detach().cpu().clone() for k in names}
    assert not torch.equal(params[names[0]].detach().cpu(), snap[names[0]]), "the replay did not update the parameters"
    # the same step eagerly at the snapshot, recording the max-pool's choices (the fused head of <= 64 graphs pools inside
    # its own kernels and records none)
    model.load_state_dict(snap)
    choices, apply = [], Fn.MaxPoolCL.apply

    def recording(x, kh, kw):
        out = apply(x, kh, kw)
        choices.append(out.grad_fn.saved_tensors[0].detach().cpu())
        return out

    monkeypatch.setattr(Fn.MaxPoolCL, "apply", recording)
    loss_e = tr._fwd_bwd(resident)
    monkeypatch.undo()
    torch.cuda.synchronize()
    assert torch.equal(loss_e, loss)
    for k in names:
        assert torch.equal(params[k].grad.detach().cpu(), got[k]), "eager and captured step differ in g_" + k
    assert len(choices) == (1 if bsz > 64 else 0), len(choices)
    loss_r, g_r = train_oracle(oracle_params(snap, names), names, raw, args, n1, model.pathway_indexs.cpu(),
                               weight if args.weight_balance else None, pool_arg=choices[0] if choices else None)
    tag = "captured gbm step B=%d" % bsz
    _check(loss.reshape(()), loss_r.reshape(()), tag + " loss")
    for k, c in zip(names, g_r):
        assert c is not None, k
        _check(got[k], c, tag + " g_" + k, rtol=2e-4, atol=1e-5, l2=1e-3, outliers=1e-3)
