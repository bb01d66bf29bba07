"""torch.autograd Functions over the C ABI (forward AND backward are hand-written kernels).

Each Function cites the reference lines whose autograd graph it replaces.  Tensors are allocated by
torch, the kernels only fill them (include/mlg_b200.h conventions).
"""
import os

import torch

from . import _cabi

AGGR_CODE = {"softmax": 0, "softmax_sg": 0, "softmax_sum": 0, "power": 1, "power_sum": 1,
             "add": 2, "sum": 2, "mean": 3, "max": 4}
EPI_NONE, EPI_RESIDUAL, EPI_MSGNORM = 0, 1, 2


def _f32c(t):
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


def _scalar_args(v):
    """(host float, device pointer or None) for a python float or a 1-element Parameter."""
    if torch.is_tensor(v):
        return 0.0, _cabi.fptr(v.detach().reshape(1))
    return float(v), None


def _ld(t):
    """Leading dimension (floats) of a 2-D fp32 view whose rows are contiguous."""
    if t.dim() != 2 or t.stride(1) != 1 or t.dtype != torch.float32:
        raise ValueError("expected a 2-D fp32 tensor with unit inner stride")
    return t.stride(0)


def _vptr(t):
    import ctypes
    _cabi.require_cuda(t)
    return ctypes.c_void_p(t.data_ptr())


def gather_sum(src, rowptr, idx, n_rows, val=None, pre=None, post=None, post_mode=0, relative=False, out=None,
               addend=None, self_out=None, replicas=1, order=None, rank1=False, tag="gather_sum", mask=None,
               mask_slope=0.0, reduce_scale=None, act_slope=None):
    """Raw (non-differentiable) call of mlg_gather_sum.  src / out / addend / self_out may be column
    slices of wider row-major buffers (leading dimension = stride(0))."""
    L = _cabi.lib()
    C = src.shape[1]
    total_rows = n_rows * replicas
    if reduce_scale is not None:     # per-slice weighted sums over the replicas: [slices * n_rows, C]; caller adds the slices
        slices = L.mlg_gather_sum_slices(n_rows, C, replicas)
        out = torch.empty(slices * n_rows, C, dtype=torch.float32, device=src.device)
    if out is None:
        out = torch.empty(total_rows, C, dtype=torch.float32, device=src.device)
    # algorithmic bytes (SURVEY.md section 8d): rows read once + rows written once + (idx, val) per entry
    nbytes = 4 * C * total_rows * 2 + 8 * idx.numel()
    args = (_vptr(src), _ld(src), _cabi.iptr(rowptr), _cabi.iptr(idx), _cabi.fptr(val, True), _cabi.fptr(pre, True),
            _cabi.fptr(post, True), _cabi.iptr(order, True), n_rows, C, replicas, 0 if rank1 else n_rows,
            n_rows if rank1 else 0, post_mode, int(relative),
            None if addend is None else _vptr(addend), 0 if addend is None else _ld(addend),
            _vptr(out), _ld(out), None if self_out is None else _vptr(self_out),
            0 if self_out is None else _ld(self_out), None if mask is None else _vptr(mask),
            0 if mask is None else _ld(mask), float(mask_slope), _cabi.fptr(reduce_scale, True))
    with torch.cuda.device(src.device), _cabi.span(tag, nbytes):
        if act_slope is None:
            _cabi.check(L.mlg_gather_sum(*args, _cabi.stream_ptr()), "mlg_gather_sum")
        else:     # fused output activation (replicated path)
            _cabi.check(L.mlg_gather_sum_act(*args, 1, float(act_slope), _cabi.stream_ptr()), "mlg_gather_sum_act")
    return out


GRAD_SLOTS_ENABLED = False   # set by train.Trainer around its own autograd.grad call only (loss.backward() would add
                             # the in-place result to .grad a second time)


def _slot_or_empty(param, like):
    """The parameter's bucket slot (functional.grad_slot) or a fresh buffer shaped like ``like``."""
    slot = grad_slot(param, like.shape) if param is not None else None
    return slot if slot is not None else torch.empty_like(like)


def grad_slot(param, shape):
    """A preallocated gradient destination for ``param`` if the trainer registered one (train.GradBucket marks its
    views with ``_mlg_grad_slot``): backward kernels then write the gradient straight into the flat bucket and the
    bucket's multi-tensor copy skips it.  Each slot is handed out once per backward (a parameter used twice falls back
    to a fresh buffer and autograd adds the two)."""
    slot = getattr(param, "_mlg_grad_slot", None) if GRAD_SLOTS_ENABLED else None
    if slot is None or slot["claimed"] or tuple(slot["view"].shape) != tuple(shape) or not slot["view"].is_contiguous():
        return None
    slot["claimed"] = True
    return slot["view"]


# GENConv aggregation backward: the source-side sum g_x[j] += sum over out-edges of g_edge runs inside the backward kernel as
# vector reductions into L2 (mlg_gen_aggr_bwd_src / _affine_src) instead of a second pass over g_edge [E, H]; with the
# affine edge term no [E, H] gradient tensor exists at all.  The order of those additions is not reproducible (neither is
# the reference's scatter-add backward); False / MLG_GEN_BWD_DETERMINISTIC=1 selects the two-pass fixed-order path.
GEN_BWD_SRC_ATOMIC = not bool(int(__import__("os").environ.get("MLG_GEN_BWD_DETERMINISTIC", "0")))
XTY_TC_MIN_ROWS = 8192   # below this the SIMT kernel's single launch wins


def _xty_tc_call(L, a, x, out, cs, cs_x, tag):
    rows, M = a.shape
    ws_bytes = L.mlg_xty_tc_workspace_bytes(M)
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device), _cabi.span(tag + "_tc", 4 * rows * (M + 128)):
        _cabi.check(L.mlg_xty_tc(_vptr(a), _ld(a), _vptr(x), _ld(x), rows, M, 128, _cabi.fptr(out), _cabi.fptr(cs, True),
                                 _cabi.fptr(cs_x, True), _cabi.fptr(ws), ws_bytes, _cabi.stream_ptr()), "mlg_xty_tc")


def xty(a, x, want_colsum=False, tag="xty", out=None):
    """out[M,K] = a[rows,M]^T @ x[rows,K] (+ column sums of a), fp32-accurate and deterministic.  Tensor cores
    (mlg_xty_tc, 3xTF32) when one side is 128 wide: K == 128 directly (M in chunks of <= 128 columns), or M == 128 with
    K a multiple of 128 by computing the transpose (roles swapped, the bias gradient then comes from the kernel's
    X-column sums); else mlg_xty (fp32 FMA)."""
    L = _cabi.lib()
    rows, M = a.shape
    K = x.shape[1]
    aligned = (_ld(a) % 4 == 0 and _ld(x) % 4 == 0 and a.data_ptr() % 16 == 0 and x.data_ptr() % 16 == 0)
    if USE_TF32X3 and rows >= XTY_TC_MIN_ROWS and aligned:
        if K == 128 and M % 16 == 0 and (M <= 128 or M % 128 == 0):
            if out is None:
                out = torch.empty(M, K, dtype=torch.float32, device=a.device)
            cs = torch.empty(M, dtype=torch.float32, device=a.device) if want_colsum else None
            step = min(M, 128)
            for m0 in range(0, M, step):
                _xty_tc_call(L, a[:, m0:m0 + step], x, out[m0:m0 + step], None if cs is None else cs[m0:m0 + step], None, tag)
            return out, cs
        if M == 128 and K % 128 == 0 and K > 128:
            out_t = torch.empty(K, M, dtype=torch.float32, device=a.device)       # (x^T a) = out^T
            cs = torch.empty(M, dtype=torch.float32, device=a.device) if want_colsum else None
            for k0 in range(0, K, 128):
                _xty_tc_call(L, x[:, k0:k0 + 128], a, out_t[k0:k0 + 128], None, cs if k0 == 0 else None, tag)
            res = out_t.t()
            if out is not None:
                out.copy_(res)
                return out, cs
            return res.contiguous(), cs
    if out is None:
        out = torch.empty(M, K, dtype=torch.float32, device=a.device)
    cs = torch.empty(M, dtype=torch.float32, device=a.device) if want_colsum else None
    ws_bytes = L.mlg_xty_workspace_bytes(rows, M, K)
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device), _cabi.span(tag, 4 * rows * (M + K)):
        _cabi.check(L.mlg_xty(_vptr(a), _ld(a), _vptr(x), _ld(x), rows, M, K, _cabi.fptr(out), _cabi.fptr(cs, True),
                              _cabi.fptr(ws), ws_bytes, _cabi.stream_ptr()), "mlg_xty")
    return out, cs


USE_TF32X3 = True      # tall Linears on the tensor cores with the 3xTF32 split (fp32-accurate); False = cuBLAS fp32


def tall_matmul(a, w, bias=None, act=0, slope=0.0, tag="gemm_tf32x3", w_split=None, out=None):
    """act(a @ w^T + bias) for a tall fp32 matrix a [M, K] and a small weight w [N, K]: mlg_gemm_tf32x3 when the shape
    is supported, else cuBLAS fp32 (+ mlg_bias_act).  act: 0 none, 1 LeakyReLU(slope).  ``out`` (contiguous [M, N], e.g. a
    parameter's gradient slot) receives the result on the tensor-core path; the other paths copy into it."""
    if out is not None:
        if not (USE_TF32X3 and a.is_cuda and out.is_contiguous() and w_split is not None
                and _cabi.lib().mlg_gemm_tf32x3_supported(a.shape[0], w.shape[0], a.shape[1])
                and a.stride(1) == 1 and a.stride(0) % 4 == 0 and a.data_ptr() % 16 == 0):
            return out.copy_(tall_matmul(a, w, bias, act, slope, tag, w_split))
    L = _cabi.lib()
    M, K = a.shape
    N = w.shape[0]
    tc_ok = USE_TF32X3 and a.is_cuda and a.stride(1) == 1 and a.stride(0) % 4 == 0 and a.data_ptr() % 16 == 0
    chunk = 0
    if tc_ok and w_split is None and not L.mlg_gemm_tf32x3_supported(M, N, K):
        for c in (128, 64):
            if N > c and N % c == 0 and L.mlg_gemm_tf32x3_supported(M, c, K):
                chunk = c
                break
    if chunk:
        # the split weight of a column slice fits in shared memory, the full width does not (128 -> 256 in two 128-column
        # launches, 256 -> 128 in two 64-column launches): each launch writes its column slice of the output in place
        out = torch.empty(M, N, dtype=torch.float32, device=a.device)
        wd = _f32c(w)
        hi, lo = torch.empty_like(wd), torch.empty_like(wd)
        bd = None if bias is None else _f32c(bias)
        with torch.cuda.device(a.device):
            _cabi.check(L.mlg_split_tf32(_cabi.fptr(wd), wd.numel(), _cabi.fptr(hi), _cabi.fptr(lo), _cabi.stream_ptr()),
                        "mlg_split_tf32")
            for n0 in range(0, N, chunk):
                with _cabi.span(tag, 4 * M * (K + chunk)):
                    _cabi.check(L.mlg_gemm_tf32x3(_vptr(a), a.stride(0), _cabi.fptr(hi[n0:n0 + chunk]),
                                                  _cabi.fptr(lo[n0:n0 + chunk]),
                                                  None if bd is None else _cabi.fptr(bd[n0:n0 + chunk]),
                                                  _vptr(out[:, n0:n0 + chunk]), N, M, chunk, K, int(act), float(slope),
                                                  _cabi.stream_ptr()), "mlg_gemm_tf32x3")
        return out
    if (tc_ok and L.mlg_gemm_tf32x3_supported(M, N, K)):
        if out is None:
            out = torch.empty(M, N, dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            if w_split is not None:
                hi, lo = w_split          # [N, K] hi / lo parts prepared by the caller (mlg_sage_fold_fwd)
            else:
                wd = _f32c(w)
                hi, lo = torch.empty_like(wd), torch.empty_like(wd)
                _cabi.check(L.mlg_split_tf32(_cabi.fptr(wd), wd.numel(), _cabi.fptr(hi), _cabi.fptr(lo),
                                             _cabi.stream_ptr()), "mlg_split_tf32")
            with _cabi.span(tag, 4 * M * (K + N)):
                _cabi.check(L.mlg_gemm_tf32x3(_vptr(a), a.stride(0), _cabi.fptr(hi), _cabi.fptr(lo),
                                              None if bias is None else _cabi.fptr(_f32c(bias)), _cabi.fptr(out), N, M, N, K,
                                              int(act), float(slope), _cabi.stream_ptr()), "mlg_gemm_tf32x3")
        return out
    if a.is_cuda and M <= 32 and K >= 1024 and a.stride(1) == 1 and w.stride(1) == 1:
        # a handful of rows against a wide weight (the head's Linear(6913 -> 256)): one pass over W, bias + act fused
        out = torch.empty(M, N, dtype=torch.float32, device=a.device)
        ws_bytes = L.mlg_skinny_linear_workspace_bytes(N, K)
        ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device), _cabi.span(tag, 4 * (N * K + M * K + M * N)):
            _cabi.check(L.mlg_skinny_linear(_vptr(a), a.stride(0), _vptr(w), w.stride(0),
                                            None if bias is None else _cabi.fptr(_f32c(bias)), M, N, K, int(act),
                                            float(slope), _cabi.fptr(out), N, _cabi.fptr(ws), ws_bytes,
                                            _cabi.stream_ptr()), "mlg_skinny_linear")
        return out
    out = a @ w.t()
    if bias is not None or act:
        with torch.cuda.device(out.device):
            _cabi.check(L.mlg_bias_act(_cabi.fptr(out), None if bias is None else _cabi.fptr(_f32c(bias)), M, N,
                                       float(slope) if act else 1.0, _cabi.stream_ptr()), "mlg_bias_act")
    return out


class TallLinear(torch.autograd.Function):
    """y = x @ W^T + b for a TALL x (rows >> features): forward and dX on the 3xTF32 tcgen05 GEMM (mlg_gemm_tf32x3, bias /
    ReLU in its epilogue; cuBLAS fp32 only for shapes it does not cover), the weight / bias gradient (a [out, rows] x
    [rows, in] product with a tiny output) on mlg_xty_tc / mlg_xty.  Used for GENConv's per-layer edge encoder on [E, H]
    edge embeddings (torch_vertex.py:76-77), its node-side MLP Linears, and 1x1 convolutions outside the fused head."""

    MIN_ROWS = 65536

    @staticmethod
    def forward(ctx, x, weight, bias, relu=False):
        """relu: the ReLU that follows the Linear (nn.Conv2d(1x1) + nn.ReLU in MultilevelGNN's head) applied in the GEMM
        epilogue; backward then starts from the activation's derivative."""
        ctx.has_bias = bias is not None
        ctx.relu = bool(relu)
        y = tall_matmul(_f32c(x.detach()), weight.detach(), None if bias is None else bias.detach(), tag="linear_fwd",
                        act=1 if relu else 0, slope=0.0)
        ctx.save_for_backward(x, weight, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, g):
        x, weight, y = ctx.saved_tensors
        g = _f32c(g)
        if ctx.relu:
            g = torch.ops.aten.threshold_backward(g, y, 0.0)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = tall_matmul(g, weight.t().contiguous(), tag="linear_dgrad")
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            gw, gb = xty(g, _f32c(x), want_colsum=ctx.has_bias, tag="linear_wgrad", out=grad_slot(weight, weight.shape))
        return gx, gw, (gb if ctx.has_bias else None), None


def tall_linear(x, lin, min_rows=None):
    """Apply an nn.Linear through TallLinear (3xTF32 tensor-core forward / dX where the shape allows, mlg_xty weight
    and bias gradient) when x is a CUDA matrix with at least ``min_rows`` rows (default TallLinear.MIN_ROWS)."""
    rows = TallLinear.MIN_ROWS if min_rows is None else min_rows
    if x.is_cuda and x.dim() == 2 and x.shape[0] >= rows and x.dtype == torch.float32:
        return TallLinear.apply(x, lin.weight, lin.bias, False)
    return lin(x)


class GenAggregate(torch.autograd.Function):
    """GENConv.message + GenMessagePassing.aggregate + MsgNorm + residual
    (models/gcn_lib/sparse/torch_vertex.py:82-89,94-101; torch_message.py:44-85,175-179).

    forward(x, e, t, p, y, msg_scale, topo, aggr, eps, epilogue, learn) -> h (or m for EPI_NONE)
      x [N,H] (None = raw messages in e), e [E,H] or None, t/p: float or Parameter[1],
      y / msg_scale: Parameter[1] or None, topo: graph.Topology without self-loop rewrite.
    """

    @staticmethod
    def forward(ctx, x, e, t, p, y, msg_scale, topo, aggr, eps, epilogue, learn):
        L = _cabi.lib()
        _cabi.require_cuda(x, e)
        ref = x if x is not None else e
        n, H = topo.n, ref.shape[1]
        xd = None if x is None else _f32c(x.detach())
        ed = None if e is None else _f32c(e.detach())
        csr = topo.fwd
        mode = AGGR_CODE[aggr]
        t_h, t_d = _scalar_args(t)
        p_h, p_d = _scalar_args(p)
        y_d = None if y is None else _cabi.fptr(y.detach().reshape(1))
        s_d = None if msg_scale is None else _cabi.fptr(msg_scale.detach().reshape(1))
        need_grad = any(ctx.needs_input_grad)      # False under torch.no_grad() as well
        h = torch.empty(n, H, dtype=torch.float32, device=ref.device) if epilogue != EPI_NONE else None
        # inference: only h leaves the kernel (m / aux exist for the backward pass); the kernel re-reads m for
        # the MsgNorm epilogue of rows wider than one chunk on the register-staged path, so keep it there
        m_optional = h is not None and not need_grad and (H <= 128 or (mode == 0 and x is not None and e is not None
                                                                        and H == 256) or epilogue == EPI_RESIDUAL)
        m = None if m_optional else torch.empty(n, H, dtype=torch.float32, device=ref.device)
        aux = torch.empty(n, H, dtype=torch.float32, device=ref.device) if (need_grad and mode in (0, 1)) else None
        n_entries = csr.col.numel()
        ctx_bytes = 4 * H * ((n_entries if e is not None else 0) + 2 * n) + 4 * n_entries + 4 * (n + 1)
        with torch.cuda.device(ref.device), _cabi.span("gen_aggr_fwd", ctx_bytes):
            _cabi.check(L.mlg_gen_aggr_fwd(
                _cabi.fptr(xd, True), _cabi.fptr(ed, True), _cabi.iptr(csr.rowptr), _cabi.iptr(csr.col),
                None if topo.fwd_identity else _cabi.iptr(csr.eid), n, H, mode, t_h, t_d, p_h, p_d, y_d,
                float(eps), epilogue, s_d,
                _cabi.fptr(m, True), _cabi.fptr(aux, True), _cabi.fptr(h, True), _cabi.stream_ptr()),
                "mlg_gen_aggr_fwd")
        if not need_grad:
            return h if h is not None else m
        ctx.topo, ctx.mode, ctx.eps, ctx.epilogue, ctx.learn = topo, mode, float(eps), epilogue, bool(learn)
        ctx.t, ctx.p, ctx.y, ctx.scale = t, p, y, msg_scale
        ctx.has_x, ctx.has_e = x is not None, e is not None
        ctx.e_shape = None if e is None else e.shape
        ctx.save_for_backward(*[v for v in (xd, ed, m, aux) if v is not None])
        ctx.saved_flags = (xd is not None, ed is not None, aux is not None)
        return h if h is not None else m

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        saved = list(ctx.saved_tensors)
        fx, fe, fa = ctx.saved_flags
        xd = saved.pop(0) if fx else None
        ed = saved.pop(0) if fe else None
        m = saved.pop(0)
        aux = saved.pop(0) if fa else None
        topo = ctx.topo
        n, H = m.shape
        g = _f32c(g)
        dev = m.device
        csr = topo.fwd
        n_edges = topo.edge_index.shape[1]
        t_h, t_d = _scalar_args(ctx.t)
        p_h, p_d = _scalar_args(ctx.p)
        y_d = None if ctx.y is None else _cabi.fptr(ctx.y.detach().reshape(1))
        s_d = None if ctx.scale is None else _cabi.fptr(ctx.scale.detach().reshape(1))
        needs = ctx.needs_input_grad
        want_ge = ctx.has_e and needs[1]
        src = (GEN_BWD_SRC_ATOMIC and ctx.has_x and needs[0] and n_edges > 0
               and bool(L.mlg_gen_aggr_bwd_src_supported(H, ctx.mode, int(xd is not None))))
        g_edge = torch.empty(max(n_edges, 1), H, dtype=torch.float32, device=dev) if (want_ge or not src) else None
        g_x = torch.empty(n, H, dtype=torch.float32, device=dev)
        rows = L.mlg_gen_aggr_bwd_partial_rows(n, H)
        partials = torch.empty(rows, 4, dtype=torch.float32, device=dev)
        bwd_bytes = 4 * H * (2 * n_edges + 3 * n) + 8 * n_edges          # SURVEY.md section 8d (no learn_t)
        fn, name = (L.mlg_gen_aggr_bwd_src, "mlg_gen_aggr_bwd_src") if src else (L.mlg_gen_aggr_bwd, "mlg_gen_aggr_bwd")
        with torch.cuda.device(dev), _cabi.span("gen_aggr_bwd", bwd_bytes):
            _cabi.check(fn(
                _cabi.fptr(g), _cabi.fptr(xd, True), _cabi.fptr(ed, True), _cabi.iptr(csr.rowptr),
                _cabi.iptr(csr.col), None if topo.fwd_identity else _cabi.iptr(csr.eid), n, H, ctx.mode, int(ctx.learn), t_h, t_d, p_h, p_d,
                y_d, ctx.eps, ctx.epilogue, s_d, _cabi.fptr(m), _cabi.fptr(aux, True), _cabi.fptr(g_edge, True),
                _cabi.fptr(g_x), _cabi.fptr(partials), _cabi.stream_ptr()), name)
        gx = None
        if src:
            gx = g_x           # direct term + source-side sums, accumulated by the kernel
        elif ctx.has_x and needs[0]:
            bw = topo.bwd      # rows = sources; eid = edge ids whose g_edge rows are summed
            gx = gather_sum(g_edge, bw.rowptr, bw.eid, n, out=g_x, addend=g_x, tag="gen_aggr_bwd_src")
        ge = g_edge[:n_edges].reshape(ctx.e_shape) if want_ge else None
        sums = None

        def part(i):
            nonlocal sums
            if sums is None:
                sums = partials.sum(dim=0)
            return sums[i].reshape(1)

        gt = part(0).reshape(ctx.t.shape) if (torch.is_tensor(ctx.t) and needs[2] and ctx.mode == 0 and ctx.learn) else None
        gp = part(0).reshape(ctx.p.shape) if (torch.is_tensor(ctx.p) and needs[3] and ctx.mode == 1 and ctx.learn) else None
        gy = part(1).reshape(ctx.y.shape) if (ctx.y is not None and needs[4]) else None
        gs = part(2).reshape(ctx.scale.shape) if (ctx.scale is not None and needs[5] and ctx.epilogue == EPI_MSGNORM) else None
        return gx, ge, gt, gp, gy, gs, None, None, None, None, None


class AffineEdge:
    """Edge embedding kept in factored form: e_ij = a_e * p + q with a per-edge scalar ``a`` [E] and H-vectors ``p``, ``q``
    (differentiable tensors).  DeeperGCN builds it from a scalar edge attribute and its Linear(1 -> H) edge encoder; a
    GENConv whose own edge encoder is a Linear composes the two analytically (``compose``) and aggregates through
    GenAggregateAffine, so no [E, H] edge tensor is ever written; ``materialize()`` serves any other consumer."""

    def __init__(self, a, p, q):
        self.a, self.p, self.q = a, p, q

    @property
    def shape(self):
        return (self.a.numel(), self.p.numel())

    def compose(self, lin):
        """The same edge term after an nn.Linear: W (a p + q) + b = a (W p) + (W q + b)."""
        q = lin.weight @ self.q
        return AffineEdge(self.a, lin.weight @ self.p, q if lin.bias is None else q + lin.bias)

    def materialize(self):
        return self.a.reshape(-1, 1) * self.p.reshape(1, -1) + self.q.reshape(1, -1)


class GenAggregateAffine(torch.autograd.Function):
    """GenAggregate with the edge term in AffineEdge form (mlg_gen_aggr_fwd_affine / _bwd_affine + mlg_wcolsum).

    forward(x [N,H], a [E], p [H], q [H], t, pw, y, msg_scale, topo, aggr, eps, epilogue, learn) -> h (or m)."""

    @staticmethod
    def forward(ctx, x, a, p, q, t, pw, y, msg_scale, topo, aggr, eps, epilogue, learn):
        L = _cabi.lib()
        _cabi.require_cuda(x, a, p, q)
        xd, ad, pd, qd = _f32c(x.detach()), _f32c(a.detach().reshape(-1)), _f32c(p.detach()), _f32c(q.detach())
        n, H = xd.shape
        csr = topo.fwd
        mode = AGGR_CODE[aggr]
        t_h, t_d = _scalar_args(t)
        p_h, p_d = _scalar_args(pw)
        y_d = None if y is None else _cabi.fptr(y.detach().reshape(1))
        s_d = None if msg_scale is None else _cabi.fptr(msg_scale.detach().reshape(1))
        need_grad = any(ctx.needs_input_grad)
        h = torch.empty(n, H, dtype=torch.float32, device=xd.device) if epilogue != EPI_NONE else None
        m = torch.empty(n, H, dtype=torch.float32, device=xd.device)
        aux = torch.empty(n, H, dtype=torch.float32, device=xd.device) if (need_grad and mode in (0, 1)) else None
        n_entries = csr.col.numel()
        with torch.cuda.device(xd.device), _cabi.span("gen_aggr_fwd_affine", 4 * H * 3 * n + 8 * n_entries + 4 * (n + 1)):
            _cabi.check(L.mlg_gen_aggr_fwd_affine(
                _cabi.fptr(xd), _cabi.fptr(ad), _cabi.fptr(pd), _cabi.fptr(qd), _cabi.iptr(csr.rowptr), _cabi.iptr(csr.col),
                None if topo.fwd_identity else _cabi.iptr(csr.eid), n, H, mode, t_h, t_d, p_h, p_d, y_d, float(eps),
                epilogue, s_d, _cabi.fptr(m), _cabi.fptr(aux, True), _cabi.fptr(h, True), _cabi.stream_ptr()),
                "mlg_gen_aggr_fwd_affine")
        if not need_grad:
            return h if h is not None else m
        ctx.topo, ctx.mode, ctx.eps, ctx.epilogue, ctx.learn = topo, mode, float(eps), epilogue, bool(learn)
        ctx.t, ctx.p, ctx.y, ctx.scale = t, pw, y, msg_scale
        ctx.has_aux, ctx.a_shape = aux is not None, a.shape
        ctx.save_for_backward(*[v for v in (xd, ad, pd, qd, m, aux) if v is not None])
        return h if h is not None else m

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        saved = list(ctx.saved_tensors)
        xd, ad, pd, qd, m = saved[:5]
        aux = saved[5] if ctx.has_aux else None
        topo = ctx.topo
        n, H = m.shape
        g = _f32c(g)
        dev = m.device
        csr = topo.fwd
        n_edges = topo.edge_index.shape[1]
        t_h, t_d = _scalar_args(ctx.t)
        p_h, p_d = _scalar_args(ctx.p)
        y_d = None if ctx.y is None else _cabi.fptr(ctx.y.detach().reshape(1))
        s_d = None if ctx.scale is None else _cabi.fptr(ctx.scale.detach().reshape(1))
        needs = ctx.needs_input_grad
        want_pq = needs[2] or needs[3]
        src = (GEN_BWD_SRC_ATOMIC and needs[0] and n_edges > 0 and H <= 256
               and bool(L.mlg_gen_aggr_bwd_src_supported(H, ctx.mode, 1)))
        g_edge = torch.empty(max(n_edges, 1), H, dtype=torch.float32, device=dev) if (needs[1] or not src) else None
        g_x = torch.empty(n, H, dtype=torch.float32, device=dev)
        rows = L.mlg_gen_aggr_bwd_partial_rows(n, H)
        partials = torch.empty(rows, 4, dtype=torch.float32, device=dev)
        gp = gq = ws = None
        ws_bytes = 0
        if want_pq:
            gp, gq = torch.empty_like(pd), torch.empty_like(qd)
            ws_bytes = L.mlg_gen_aggr_bwd_affine_workspace_bytes(n, n_edges, H)
            ws = torch.empty((ws_bytes + 3) // 4, dtype=torch.float32, device=dev)
        fn, name = ((L.mlg_gen_aggr_bwd_affine_src, "mlg_gen_aggr_bwd_affine_src") if src
                    else (L.mlg_gen_aggr_bwd_affine, "mlg_gen_aggr_bwd_affine"))
        with torch.cuda.device(dev), _cabi.span("gen_aggr_bwd_affine", 4 * H * (n_edges + 4 * n) + 12 * n_edges):
            _cabi.check(fn(
                _cabi.fptr(g), _cabi.fptr(xd), _cabi.fptr(ad), _cabi.fptr(pd), _cabi.fptr(qd), _cabi.iptr(csr.rowptr),
                _cabi.iptr(csr.col), None if topo.fwd_identity else _cabi.iptr(csr.eid), n, n_edges, H, ctx.mode,
                int(ctx.learn), t_h, t_d, p_h, p_d, y_d, ctx.eps, ctx.epilogue, s_d, _cabi.fptr(m), _cabi.fptr(aux, True),
                _cabi.fptr(g_edge, True), _cabi.fptr(g_x), _cabi.fptr(partials), _cabi.fptr(gp, True), _cabi.fptr(gq, True),
                _cabi.fptr(ws, True), ws_bytes, _cabi.stream_ptr()), name)
        gx = None
        if src:
            gx = g_x
        elif needs[0]:
            bw = topo.bwd
            gx = gather_sum(g_edge, bw.rowptr, bw.eid, n, out=g_x, addend=g_x, tag="gen_aggr_bwd_src")
        ga = None
        if needs[1]:      # gradient w.r.t. the scalar edge attribute itself (not needed by the reference's data path)
            ga = (g_edge[:n_edges] @ pd).reshape(ctx.a_shape)
        sums = None

        def part(i):
            nonlocal sums
            if sums is None:
                sums = partials.sum(dim=0)
            return sums[i].reshape(1)

        gt = part(0).reshape(ctx.t.shape) if (torch.is_tensor(ctx.t) and needs[4] and ctx.mode == 0 and ctx.learn) else None
        gpw = part(0).reshape(ctx.p.shape) if (torch.is_tensor(ctx.p) and needs[5] and ctx.mode == 1 and ctx.learn) else None
        gy = part(1).reshape(ctx.y.shape) if (ctx.y is not None and needs[6]) else None
        gs = part(2).reshape(ctx.scale.shape) if (ctx.scale is not None and needs[7] and ctx.epilogue == EPI_MSGNORM) else None
        return gx, ga, gp, gq, gt, gpw, gy, gs, None, None, None, None, None


class SageAggregate(torch.autograd.Function):
    """Weighted mean over in-neighbours incl. the rewritten self loop, BEFORE the lin_r transform:
    agg_i = (sum_{j->i, j!=i} w_ij x_j + x_i) / (deg_i + 1)   [- x_i for RSAGE]
    (SAGEConv.forward/message + PyG mean aggregation, models/gcn_lib/sparse/torch_vertex.py:269-286)."""

    @staticmethod
    def forward(ctx, x, topo, relative):
        _cabi.require_cuda(x)
        xd = _f32c(x.detach())
        csr = topo.fwd
        out = gather_sum(xd, csr.rowptr, csr.col, topo.n_single, val=topo.fwd_val, post_mode=1, relative=relative,
                         replicas=topo.replicas, order=topo.fwd_order, tag="sage_aggr_fwd")
        ctx.topo, ctx.relative = topo, bool(relative)
        return out

    @staticmethod
    def backward(ctx, g):
        topo = ctx.topo
        g = _f32c(g)
        bw = topo.bwd
        # g_x[j] = sum_{i: j->i} w_ij * g[i] / cnt_i   (entries of the by-source CSR: col = target i)
        gx = gather_sum(g, bw.rowptr, bw.col, topo.n_single, val=topo.bwd_val, pre=topo.inv_cnt,
                        replicas=topo.replicas, order=topo.bwd_order, tag="sage_aggr_bwd")
        if ctx.relative:
            gx = gx - g
        return gx, None, None


def _flag(name, default):
    """Tuning switches that are worth flipping from the shell for an A/B run (tools/): everything else is a module constant."""
    return os.environ.get(name, "1" if default else "0") == "1"


# Evaluation order of a SAGE layer (same algebra, torch_vertex.py:269-294; DESIGN.md section 4).  Module constants -- the parity
# tests flip them to compare each order with the buffered one -- not environment switches.
# first layer of MultilevelGNN through mlg_sage_rank1_fwd_rows / mlg_sage_rank1_bwd_rows; "gather": backward through the
# by-source gather mlg_sage_rank1_bwd (any width); False: [x0 | agg] buffer + GEMMs
FACTORED_RANK1 = True
# SAGE layers with out_channels < in_channels evaluated transform-first (gather on the narrower rows); False: [x | agg] + GEMM
TRANSFORM_FIRST = True
H1_NODE_MAJOR = True     # the factored first layer writes its output node-major for a transform-first consumer (and takes its gradient so)
GZ_NODE_MAJOR = True     # the pool writes the last layer's output gradient node-major for the transform-first backward aggregation
# The factored first layer applies LeakyReLU'(y) to its output gradient INSIDE mlg_sage_rank1_bwd_rows, from 64 sign bits per
# (gene, replica) its forward kernel wrote (B200: 66 us vs 61 us unmasked; re-reading the 126 MB activation instead costs
# 175 us, profiles/r02_rank1_bwd_probe.jsonl).  Widths without sign words (!= 64): one library leaky_relu_backward pass.
RANK1_SIGN_BITS = True
# forward of the factored first layer with one warp per gene for all replicas (mlg_sage_rank1_fwd_rows); False: r01's kernel
RANK1_FWD_ROWS = True

# Independent branches of the backward pass on forked streams (captured by the trainer's CUDA graph as parallel branches):
# a layer's weight gradient does not feed the input-gradient chain, so it runs next to it instead of in front of it.
# Both branches are HBM streams, so the win is the latency / tail overlap, not 2x.  The fork is joined back into the
# launching stream at the END of the backward pass (autograd engine callback); tensors the side branch reads stay
# referenced until then (no cross-stream reuse by the caching allocator).
# measured on B200 (gpurun_out r02_bench_quick: 0.8455 ms forked vs 0.8463 ms serial): no gain today -- the big backward kernels
# (gemm_tf32x3, xty_tc) are persistent one-CTA-per-SM kernels that cannot co-reside, so the branches serialise anyway; off by default
PARALLEL_BACKWARD = _flag("MLG_PARALLEL_BACKWARD", False)     # A/B switch (tools/gpu_quick.sh)
# Set by train.Trainer around its own autograd.grad call only: the gradients a forked branch produces may not be touched
# before the end-of-backward join, which holds for the trainer (it stores them after the pass) but not for an arbitrary
# loss.backward(), whose AccumulateGrad nodes run on the launching stream as soon as a Function returns.
PARALLEL_ACTIVE = False
# set by train.Trainer (data parallel, fused peer update): called at the end of HeadMLP.backward, when the classifier head's
# gradients are final, to start that chunk's reduce-scatter / Adam / all-gather while the rest of backward runs
AFTER_HEAD_BACKWARD = None
_SIDE_STREAMS = {}


def _side_stream(device, idx):
    key = (device.index if device.index is not None else torch.cuda.current_device(), idx)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


class _Forked:
    """with _Forked(device, idx, keep=[tensors the branch reads]) as f: ... enqueue the branch ...
    Inside the block the current stream is a side stream that waits for everything enqueued so far; leaving the block
    registers the join for the end of the backward pass.  Outside a backward pass, or with PARALLEL_BACKWARD off, the
    block simply runs on the current stream."""

    def __init__(self, device, idx, keep=(), force=False):
        self.device, self.idx, self.keep, self.force = device, idx, list(keep), force
        self.active = False

    def __enter__(self):
        if not ((PARALLEL_BACKWARD or self.force) and PARALLEL_ACTIVE and self.device.type == "cuda"):
            return self
        self.main = torch.cuda.current_stream(self.device)
        self.side = _side_stream(self.device, self.idx)
        self.side.wait_stream(self.main)
        self.ctx = torch.cuda.stream(self.side)
        self.ctx.__enter__()
        self.active = True
        return self

    def hold(self, *tensors):
        self.keep.extend(t for t in tensors if t is not None)

    def __exit__(self, *exc):
        if not self.active:
            return False
        self.ctx.__exit__(*exc)
        main, side, keep = self.main, self.side, self.keep

        def join(_keep=keep):
            main.wait_stream(side)

        try:
            torch.autograd.Variable._execution_engine.queue_callback(join)
        except RuntimeError:          # not inside a backward pass: join right away
            join()
        return False


class SageLayer(torch.autograd.Function):
    """One whole SAGEConv layer (torch_vertex.py:269-294 with RSAGEConv's Linear+activation MLP):
        out = act( [x | agg_x] @ [W1 | W2 @ W_r]^T + b ),   nn.0.weight = [W1 | W2], lin_r.weight = W_r
    i.e. the reference's  nn(cat(x, mean_j(w_ij x_j) @ W_r^T))  with the two chained Linears folded into
    one GEMM over the concatenated buffer (fp reassociation only, SURVEY.md App. B.4).
    Three evaluation orders of the same lines, chosen per layer:
    * generic: mlg_gather_sum writes agg_x and the copy of x straight into the two halves of the [N, 2Cin] buffer (no
      torch.cat), one mlg_gemm_tf32x3 update GEMM with bias + activation in its epilogue; backward: mlg_xty_tc / mlg_xty
      weight gradient, mlg_gemm_tf32x3 dX, the backward aggregation reads the right half of d[x|agg_x] in place and adds
      the left half;
    * factored (MultilevelGNN's first layer, rank-1 input): per-gene tables + mlg_sage_rank1_fwd_rows / _bwd_rows;
    * transform-first (out_channels < in_channels): [U | V] GEMM, then the aggregation on the narrower rows.
    The last two take their weights from mlg_sage_fold_stacked_fwd (stacked weight, both 3xTF32 splits, bias: one launch)."""

    @staticmethod
    def forward(ctx, x, xs, lin_r_w, nn_w, nn_b, topo, relative, slope, in_slope=None, out_premasked=False, link=None,
                prod_link=None):
        """x [B*N, Cin] node features -- or, with ``xs`` [B*N] given, x = node_embedding [N, Cin] and the layer
        input is the rank-1 product xs[b,n] * x[n,:] (MultilevelGNN's first layer, never materialised).
        Activation-backward fusion across layers (set by the model, which knows the layer chain):
        ``in_slope`` -- x is the output of a (Leaky)ReLU with that slope whose producer expects dL/dz: the returned
        gradient is multiplied by the activation derivative inside the backward aggregation's epilogue;
        ``out_premasked`` -- the consumer of y does the same for this layer, so backward takes gy as dL/dz."""
        _cabi.require_cuda(x, lin_r_w, nn_w)
        ctx.wparams = (lin_r_w, nn_w, nn_b)      # their gradients are written straight into the trainer's bucket slots
        xd = _f32c(x.detach())
        rank1 = xs is not None
        xs_d = _f32c(xs.detach().reshape(-1)) if rank1 else None
        n = xs_d.numel() if rank1 else xd.shape[0]
        cin = xd.shape[1]
        w_r, w_nn = lin_r_w.detach(), nn_w.detach()
        w_r, w_nn = _f32c(w_r), _f32c(w_nn)
        cout = w_nn.shape[0]
        factored_ok = (FACTORED_RANK1 and rank1 and not relative and topo.replicas > 1 and cout % 4 == 0
                       and xd.shape[0] == topo.n_single and n == topo.n_single * topo.replicas)
        tfirst_ok = (not factored_ok and TRANSFORM_FIRST and not rank1 and not relative and in_slope is None
                     and topo.replicas > 1 and cout < cin and cout % 4 == 0 and cin % 4 == 0
                     and n == topo.n_single * topo.replicas)
        # layout hand-shakes (dicts the model shares between neighbouring Functions; rows node-major = (replica b, node i) at
        # i * B + b): ``prod_link["h1_nm"]`` -- the producer wrote x node-major; ``link["want_h1_nm"]`` -- the consumer of this
        # layer's output can take it node-major (set by the model from the consumer's static configuration)
        x_nm = bool(prod_link is not None and prod_link.get("h1_nm"))
        if x_nm and not (tfirst_ok and cout == 32):
            raise RuntimeError("SageLayer: node-major input rows reached a layer call that does not run transform-first on 32-wide "
                               "rows (model-level layout hand-shake out of sync)")
        if factored_ok or tfirst_ok:
            # Wst = [W1 ; W2 . W_r] [2cout, cin], its tf32 hi / lo split, the split of Wst^T and the bias [b | 0]: one launch
            sb = torch.empty(5 * 2 * cout * cin + 2 * cout, dtype=torch.float32, device=xd.device)
            wparts = [sb[i * 2 * cout * cin:(i + 1) * 2 * cout * cin] for i in range(5)]
            bias2 = sb[5 * 2 * cout * cin:] if (tfirst_ok and nn_b is not None) else None
            with torch.cuda.device(xd.device):
                _cabi.check(_cabi.lib().mlg_sage_fold_stacked_fwd(
                    _cabi.fptr(w_nn), _cabi.fptr(w_r), None if nn_b is None else _cabi.fptr(_f32c(nn_b.detach())), cout, cin,
                    w_r.shape[0], _cabi.fptr(wparts[0]), _cabi.fptr(wparts[1]), _cabi.fptr(wparts[2]), _cabi.fptr(wparts[3]),
                    _cabi.fptr(wparts[4]), None if bias2 is None else _cabi.fptr(bias2), _cabi.stream_ptr()),
                    "mlg_sage_fold_stacked_fwd")
            wst = wparts[0].view(2 * cout, cin)
            wst_split = (wparts[1].view(2 * cout, cin), wparts[2].view(2 * cout, cin))
            ctx.wst_t_split = (wparts[3].view(cin, 2 * cout), wparts[4].view(cin, 2 * cout))    # Wst^T hi / lo: the dX GEMMs
        else:
            wbuf = torch.empty(5, cout * 2 * cin, dtype=torch.float32, device=xd.device)
            with torch.cuda.device(xd.device):   # Wcat = [W1 | W2 . W_r], its tf32 hi/lo split, and the split of Wcat^T
                _cabi.check(_cabi.lib().mlg_sage_fold_fwd(_cabi.fptr(w_nn), _cabi.fptr(w_r), cout, cin, w_r.shape[0],
                                                          _cabi.fptr(wbuf[0]),
                                                          _cabi.fptr(wbuf[1]), _cabi.fptr(wbuf[2]), _cabi.fptr(wbuf[3]),
                                                          _cabi.fptr(wbuf[4]), _cabi.stream_ptr()), "mlg_sage_fold_fwd")
            wcat = wbuf[0].view(cout, 2 * cin)
        ctx.factored = False
        if factored_ok:
            # Fully factored first layer: x0 = xs * emb is rank-1 per node, so z = xs[b,i] E_self[i] + mean_j(w_ij xs[b,j]
            # E_nbr[j]) + b with the per-gene tables [E_self | E_nbr] = emb [W1 ; W2 W_r]^T (an n_single-row GEMM).  Neither
            # x0, the [x0 | agg] buffer nor the B*N-row update / dgrad / weight-gradient GEMMs exist on this path.
            L = _cabi.lib()
            n1 = topo.n_single
            e12 = tall_matmul(xd, wst, tag="sage_rank1_tables", w_split=wst_split)     # [n1, 2cout] = [E_self | E_nbr]
            y = torch.empty(n, cout, dtype=torch.float32, device=xd.device)
            csr = topo.fwd
            bias = None if nn_b is None else _f32c(nn_b.detach())
            nbytes = 4 * cout * n + 4 * n + 8 * csr.col.numel() + 8 * cout * n1
            # the consumer does not pre-mask our output gradient: keep the sign bits of y (8 bytes per row and replica) so that
            # the backward kernel applies LeakyReLU' without re-reading y
            mbits = None
            if RANK1_SIGN_BITS and cout == 64 and not out_premasked and any(ctx.needs_input_grad):
                mbits = torch.empty(n1 * topo.replicas, dtype=torch.int64, device=xd.device)
            rows_ok = RANK1_FWD_ROWS and bool(L.mlg_sage_rank1_fwd_rows_supported(cout))
            xs_t = None
            h1_nm = bool(H1_NODE_MAJOR and rows_ok and link is not None and link.get("want_h1_nm")
                         and bool(L.mlg_sage_rank1_bwd_rows_supported(cout)) and FACTORED_RANK1 != "gather")
            fwd_rows = L.mlg_sage_rank1_fwd_rows_nm if h1_nm else L.mlg_sage_rank1_fwd_rows
            with torch.cuda.device(xd.device):
                if rows_ok:
                    # node values transposed to [n1, B]: one coalesced load per CSR entry in the forward AND the backward kernel
                    xs_t = torch.empty(n1 * topo.replicas, dtype=torch.float32, device=xd.device)
                    _cabi.check(L.mlg_transpose_bn(_cabi.fptr(xs_d), topo.replicas, n1, _cabi.fptr(xs_t), _cabi.stream_ptr()),
                                "mlg_transpose_bn")
                with _cabi.span("sage_rank1_fwd", nbytes):
                    if rows_ok:
                        _cabi.check(fwd_rows(
                            _cabi.fptr(xs_t), _vptr(e12), 2 * cout, _vptr(e12[:, cout:]), 2 * cout, _cabi.iptr(csr.rowptr),
                            _cabi.iptr(csr.col), _cabi.fptr(topo.fwd_val, True),
                            _cabi.iptr(topo.fwd_order, True), n1, cout, topo.replicas,
                            _cabi.fptr(bias, True), float(slope), _cabi.fptr(y), cout, _cabi.lptr(mbits, True),
                            _cabi.stream_ptr()), "mlg_sage_rank1_fwd_rows")
                    else:
                        _cabi.check(L.mlg_sage_rank1_fwd(
                            _cabi.fptr(xs_d), _vptr(e12), 2 * cout, _vptr(e12[:, cout:]), 2 * cout, _cabi.iptr(csr.rowptr),
                            _cabi.iptr(csr.col), _cabi.fptr(topo.fwd_val, True),
                            _cabi.iptr(topo.fwd_order, True), n1, cout, topo.replicas,
                            _cabi.fptr(bias, True), float(slope), _cabi.fptr(y), cout, _cabi.lptr(mbits, True),
                            _cabi.stream_ptr()), "mlg_sage_rank1_fwd")
            ctx.xs_t = xs_t
            ctx.mbits = mbits
            ctx.h1_nm = h1_nm
            # the input gradient w.r.t. xs reads the per-gene tables again (7.9 MB at the gbm shape): kept only when asked for
            ctx.e12 = e12 if ctx.needs_input_grad[1] else None
            ctx.xs_shape = xs.shape
            if h1_nm:
                link["h1_nm"] = True          # y (and the gradient this layer gets back) is node-major
            ctx.save_for_backward(xd, y, wst, w_r, w_nn, xs_d)
            ctx.topo, ctx.relative, ctx.slope, ctx.cin, ctx.has_bias = topo, False, float(slope), cin, nn_b is not None
            ctx.rank1, ctx.factored, ctx.transform_first = True, True, False
            ctx.emb_param = x if isinstance(x, torch.nn.Parameter) else None
            ctx.in_slope = None
            ctx.out_premasked = bool(out_premasked)
            return y
        ctx.transform_first = False
        if tfirst_ok:
            # out_channels < in_channels: transform, THEN aggregate -- z = U + mean_j(w_ij V_j) with
            # [U | V] = x [W1 ; W2 W_r]^T + [b | 0]: the gather (the L2-bandwidth-bound step) runs on cout-wide rows instead of
            # cin-wide ones, forward and backward, and no [x | agg] buffer is written.
            uv = tall_matmul(xd, wst, bias2, tag="sage_update_gemm", w_split=wst_split)     # [n, 2cout] = [U | V]
            csr = topo.fwd
            if x_nm:
                # x came node-major, so [U | V] is: one contiguous block of V rows per CSR entry; y goes out graph-major
                y = torch.empty(n, cout, dtype=torch.float32, device=xd.device)
                with torch.cuda.device(xd.device), _cabi.span("sage_aggr_fwd", 4 * cout * n * 2 + 8 * csr.col.numel()):
                    _cabi.check(_cabi.lib().mlg_gather_sum_nm_ex(
                        _vptr(uv[:, cout:]), 2 * cout, _cabi.iptr(csr.rowptr), _cabi.iptr(csr.col), _cabi.fptr(topo.fwd_val, True),
                        None, _cabi.iptr(topo.fwd_order, True), topo.n_single, topo.replicas, 1, _cabi.fptr(uv), 2 * cout, 1,
                        float(slope), _cabi.fptr(y), cout, None, 0, 0, _cabi.stream_ptr()), "mlg_gather_sum_nm_ex")
            else:
                y = gather_sum(uv[:, cout:], csr.rowptr, csr.col, topo.n_single, val=topo.fwd_val, post_mode=1,
                               addend=uv[:, :cout], replicas=topo.replicas, order=topo.fwd_order,
                               tag="sage_aggr_fwd", act_slope=slope)
            ctx.x_nm = x_nm
            ctx.save_for_backward(xd, y, wst, w_r, w_nn, None)
            ctx.topo, ctx.relative, ctx.slope, ctx.cin, ctx.has_bias = topo, False, float(slope), cin, nn_b is not None
            ctx.rank1, ctx.transform_first, ctx.emb_param, ctx.in_slope = False, True, None, None
            ctx.out_premasked = bool(out_premasked)
            # ``link``: shared with the PathwayPool that consumes y and pre-masks its gradient (out_premasked).  gy then IS dL/dz
            # and its only reader is this layer's backward aggregation, so the pool may write it NODE-MAJOR (row i * B + b: the B
            # replica rows a CSR entry gathers are one contiguous block) -- requested here, confirmed by the pool's backward.
            ctx.link = link if (GZ_NODE_MAJOR and link is not None and out_premasked and cout == 32 and topo.replicas > 1) else None
            if ctx.link is not None:
                ctx.link["gz_node_major"] = True
            return y
        wsplit = (wbuf[1].view(cout, 2 * cin), wbuf[2].view(cout, 2 * cin))
        xcat = torch.empty(n, 2 * cin, dtype=torch.float32, device=xd.device)
        csr = topo.fwd
        gather_sum(xd, csr.rowptr, csr.col, topo.n_single, val=topo.fwd_val, pre=xs_d, post_mode=1, relative=relative,
                   out=xcat[:, cin:], self_out=xcat[:, :cin], replicas=topo.replicas, order=topo.fwd_order,
                   rank1=rank1, tag="sage_aggr_fwd")
        # update GEMM + bias + (Leaky)ReLU: 3xTF32 tensor-core kernel with fused epilogue (cuBLAS fp32 + mlg_bias_act
        # for shapes it does not cover)
        y = tall_matmul(xcat, wcat, None if nn_b is None else nn_b.detach(), act=1, slope=slope, tag="sage_update_gemm",
                        w_split=wsplit)
        ctx.save_for_backward(xcat, y, wbuf, w_r, w_nn, xs_d if rank1 else None)
        ctx.topo, ctx.relative, ctx.slope, ctx.cin, ctx.has_bias = topo, bool(relative), float(slope), cin, nn_b is not None
        ctx.rank1 = rank1
        ctx.emb_d = xd if (rank1 and ctx.needs_input_grad[1]) else None
        ctx.xs_shape = xs.shape if rank1 else None
        ctx.emb_param = x if (rank1 and isinstance(x, torch.nn.Parameter)) else None
        ctx.in_slope = None if (in_slope is None or relative or rank1) else float(in_slope)
        if in_slope is not None and ctx.in_slope is None:
            raise ValueError("SageLayer: in_slope needs a plain (non-relative, materialised) input")
        ctx.out_premasked = bool(out_premasked)
        return y

    @staticmethod
    def _rank1_input_grad(ctx, gz, bits, y):
        """dL/dxs of the factored layer (mlg_sage_rank1_bwd_xs): gz is dL/dz, or dL/dy with the LeakyReLU derivative taken
        from the forward's sign bits ``bits`` or from the output ``y``; rows node-major when the layer wrote its output so."""
        L = _cabi.lib()
        topo = ctx.topo
        n1, B = topo.n_single, topo.replicas
        e12 = ctx.e12
        cout = e12.shape[1] // 2
        fw, bw = topo.fwd, topo.bwd
        g_xs = torch.empty(B * n1, dtype=torch.float32, device=gz.device)
        ws_bytes = L.mlg_sage_rank1_bwd_xs_workspace_bytes(fw.cap, n1, B)
        ws = torch.empty(max(ws_bytes // 4, 1), dtype=torch.float32, device=gz.device)
        nbytes = 4 * cout * gz.shape[0] + 8 * fw.col.numel() + 3 * ws_bytes + 4 * g_xs.numel()
        with torch.cuda.device(gz.device), _cabi.span("sage_rank1_bwd_xs", nbytes):
            _cabi.check(L.mlg_sage_rank1_bwd_xs(
                _cabi.fptr(gz), cout, 1 if getattr(ctx, "h1_nm", False) else 0, _cabi.fptr(y, True), _cabi.lptr(bits, True),
                float(ctx.slope), _vptr(e12), 2 * cout, _vptr(e12[:, cout:]), 2 * cout, _cabi.iptr(fw.rowptr),
                _cabi.iptr(fw.col), _cabi.fptr(topo.fwd_val, True), _cabi.iptr(topo.fwd_order, True), _cabi.iptr(bw.rowptr),
                _cabi.iptr(topo.bwd2fwd), n1, fw.cap, cout, B, _cabi.fptr(g_xs), _cabi.fptr(ws), ws_bytes,
                _cabi.stream_ptr()), "mlg_sage_rank1_bwd_xs")
        return g_xs.view(ctx.xs_shape)

    @staticmethod
    def _backward_factored(ctx, gy):
        emb, y, wst, w_r, w_nn, xs_d = ctx.saved_tensors
        topo, cin = ctx.topo, ctx.cin
        cout = w_nn.shape[0]
        gy = _f32c(gy)
        L = _cabi.lib()
        n1, B = topo.n_single, topo.replicas
        needs = ctx.needs_input_grad
        want_w = needs[0] or needs[2] or needs[3] or needs[4]
        g_xs = None
        if not want_w:
            # input gradient only (attribution): none of the table / weight-gradient work below
            if ctx.out_premasked:
                g_xs = SageLayer._rank1_input_grad(ctx, gy, None, None)
            else:
                g_xs = SageLayer._rank1_input_grad(ctx, gy, ctx.mbits, None if ctx.mbits is not None else y)
            return None, g_xs, None, None, None, None, None, None, None, None, None, None
        by_rows = FACTORED_RANK1 != "gather" and bool(L.mlg_sage_rank1_bwd_rows_supported(cout))
        y_mask = bits = None
        if ctx.out_premasked:
            gz = gy
        elif by_rows and ctx.mbits is not None:
            # the kernel applies LeakyReLU'(y) while it loads the gradient rows, from the forward kernel's sign bits
            gz, bits = gy, ctx.mbits
        else:
            gz = torch.ops.aten.leaky_relu_backward(gy, y, ctx.slope, True) if ctx.slope != 0.0 \
                else torch.ops.aten.threshold_backward(gy, y, 0.0)
        if needs[1]:
            g_xs = SageLayer._rank1_input_grad(ctx, gz, bits, None)
        if by_rows:
            # by target row: gz read once -> per-entry rows h (+ the self / bias reductions), then a segment sum by source
            fw, bw = topo.fwd, topo.bwd
            g12 = torch.empty(n1, 2 * cout, dtype=torch.float32, device=gz.device)      # [g_E_self | g_E_nbr]
            gbr = torch.empty(n1, cout, dtype=torch.float32, device=gz.device)
            h = torch.empty(fw.cap, cout, dtype=torch.float32, device=gz.device)
            nbytes = 4 * cout * gz.shape[0] + 4 * gz.shape[0] + 8 * fw.col.numel() + 4 * (h.numel() + 2 * gbr.numel())
            with torch.cuda.device(gz.device), _cabi.span("sage_rank1_bwd", nbytes):
                xs_t = getattr(ctx, "xs_t", None)
                bwd_rows = L.mlg_sage_rank1_bwd_rows_nm if getattr(ctx, "h1_nm", False) else L.mlg_sage_rank1_bwd_rows
                _cabi.check(bwd_rows(
                    _cabi.fptr(gz), cout, _cabi.fptr(y_mask, True),
                    _cabi.lptr(bits, True), float(ctx.slope),
                    _cabi.fptr(xs_d if xs_t is None else xs_t), 0 if xs_t is None else 1, _cabi.iptr(fw.rowptr),
                    _cabi.iptr(fw.col),
                    _cabi.fptr(topo.fwd_val, True), _cabi.iptr(topo.fwd_order, True), n1, cout, B,
                    _cabi.fptr(h),
                    _cabi.fptr(g12), 2 * cout, _cabi.fptr(gbr), _cabi.stream_ptr()), "mlg_sage_rank1_bwd_rows")
            g_b = None
            if ctx.has_bias:       # column sums of the per-row partials: one streaming pass, fixed order (mlg_wcolsum)
                with _Forked(gz.device, 1, keep=(gbr,)) as fk:      # independent of the segment sum below
                    g_b = grad_slot(ctx.wparams[2], (cout,))
                    if g_b is None:
                        g_b = torch.empty(cout, dtype=torch.float32, device=gz.device)
                    ws_bytes = L.mlg_wcolsum_workspace_bytes(n1, cout)
                    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=gz.device)
                    with torch.cuda.device(gz.device):
                        _cabi.check(L.mlg_wcolsum(_cabi.fptr(gbr), cout, None, n1, cout, None, _cabi.fptr(g_b), _cabi.fptr(ws),
                                                  ws_bytes, _cabi.stream_ptr()), "mlg_wcolsum")
                    fk.hold(g_b, ws)
            gather_sum(h, bw.rowptr, topo.bwd2fwd, n1, out=g12[:, cout:], order=topo.bwd_order, tag="sage_rank1_bwd_seg")
        else:
            slices = L.mlg_gather_sum_slices(n1, cout, B)
            parts = torch.empty(slices * n1 * 3 * cout, dtype=torch.float32, device=gz.device)
            p12 = parts[:slices * n1 * 2 * cout].view(slices, n1, 2 * cout)
            pb = parts[slices * n1 * 2 * cout:].view(slices * n1, cout)
            bw = topo.bwd
            nbytes = 4 * cout * gz.shape[0] + 4 * gz.shape[0] + 8 * bw.col.numel() + 4 * parts.numel()
            with torch.cuda.device(gz.device), _cabi.span("sage_rank1_bwd", nbytes):
                _cabi.check(L.mlg_sage_rank1_bwd(
                    _cabi.fptr(gz), cout, _cabi.fptr(xs_d), _cabi.iptr(bw.rowptr), _cabi.iptr(bw.col),
                    _cabi.fptr(topo.bwd_val, True), _cabi.fptr(topo.inv_cnt, True), _cabi.iptr(topo.bwd_order, True), n1, cout, B,
                    _cabi.fptr(p12), _cabi.fptr(pb), _cabi.stream_ptr()), "mlg_sage_rank1_bwd")
            g12 = p12.sum(0) if slices > 1 else p12[0]                 # [n1, 2cout] = [g_E_self | g_E_nbr]
            g_b = pb.sum(0) if ctx.has_bias else None
        # [2cout, cin] = [g_W1 ; g_(W2 W_r)] = g12^T emb (a 15 405-deep reduction) + the weight un-folding: on a forked stream
        # next to the table -> embedding product
        with _Forked(gz.device, 2, keep=(g12, emb, w_nn, w_r)) as fk:
            g_wst, _ = xty(g12, emb, tag="sage_rank1_wgrad")                       # [2cout, cin], stacked like Wst
            g_wnn, g_wr = _slot_or_empty(ctx.wparams[1], w_nn), _slot_or_empty(ctx.wparams[0], w_r)
            with torch.cuda.device(gz.device):
                _cabi.check(L.mlg_sage_fold_stacked_bwd(_cabi.fptr(g_wst), None, cin, _cabi.fptr(w_nn), _cabi.fptr(w_r), cout,
                                                        cin, w_r.shape[0], _cabi.fptr(g_wnn), _cabi.fptr(g_wr),
                                                        _cabi.stream_ptr()), "mlg_sage_fold_stacked_bwd")
            fk.hold(g_wst, g_wnn, g_wr)
        slot = grad_slot(ctx.emb_param, (n1, cin)) if ctx.emb_param is not None else None
        g_emb = tall_matmul(g12, wst.t(), tag="sage_rank1_demb", w_split=ctx.wst_t_split, out=slot)     # g12 @ Wst
        return g_emb, g_xs, g_wr, g_wnn, g_b, None, None, None, None, None, None, None

    @staticmethod
    def _backward_transform_first(ctx, gy):
        x, y, wst, w_r, w_nn, _ = ctx.saved_tensors
        topo, cin = ctx.topo, ctx.cin
        cout = w_nn.shape[0]
        gy = _f32c(gy)
        if ctx.out_premasked:
            gz = gy
        else:
            gz = torch.ops.aten.leaky_relu_backward(gy, y, ctx.slope, True) if ctx.slope != 0.0 \
                else torch.ops.aten.threshold_backward(gy, y, 0.0)
        L = _cabi.lib()
        n = gz.shape[0]
        bw = topo.bwd
        # G = [g_U | g_V] = [gz | A^T gz]: the by-source aggregation runs on the cout-wide gz rows and copies them alongside
        g_uv = torch.empty(n, 2 * cout, dtype=torch.float32, device=gz.device)
        link = getattr(ctx, "link", None)
        gz_nm = bool(link is not None and link.pop("gz_written_node_major", False))
        x_nm = bool(getattr(ctx, "x_nm", False))
        if x_nm and not gz_nm:      # x (and so g_uv) node-major but the gradient arrived graph-major: one transposing copy
            gz = gz.view(topo.replicas, topo.n_single, cout).transpose(0, 1).contiguous().view(n, cout)
            gz_nm = True
        if gz_nm:
            # gz node-major (written so by the pool): every load instruction of the aggregation reads 512 contiguous bytes;
            # g_uv in the row order of x
            with torch.cuda.device(gz.device), _cabi.span("sage_aggr_bwd", 4 * cout * n * 2 + 8 * bw.col.numel()):
                _cabi.check(L.mlg_gather_sum_nm_ex(_cabi.fptr(gz), cout, _cabi.iptr(bw.rowptr), _cabi.iptr(bw.col),
                                                   _cabi.fptr(topo.bwd_val, True), _cabi.fptr(topo.inv_cnt, True),
                                                   _cabi.iptr(topo.bwd_order, True), topo.n_single, topo.replicas, 0, None, 0, 0,
                                                   0.0, _vptr(g_uv[:, cout:]), 2 * cout, _vptr(g_uv), 2 * cout,
                                                   1 if x_nm else 0, _cabi.stream_ptr()), "mlg_gather_sum_nm_ex")
        else:
            gather_sum(gz, bw.rowptr, bw.col, topo.n_single, val=topo.bwd_val, pre=topo.inv_cnt, out=g_uv[:, cout:],
                       self_out=g_uv[:, :cout], replicas=topo.replicas, order=topo.bwd_order,
                       tag="sage_aggr_bwd")
        needs = ctx.needs_input_grad
        gx = g_wr = g_wnn = g_b = None
        # the weight gradient (tensor-core x^T G over the row pairs + fold) on a forked stream next to the input-gradient GEMM
        # and everything autograd runs after it (the first layer's backward); joined at the end of the backward pass
        if needs[2] or needs[3] or needs[4]:
            with _Forked(gz.device, 0, keep=(g_uv, x, w_nn, w_r)) as fk:
                if n % 2 == 0 and 4 * cout == 128 and 2 * cin == 128:
                    # tensor-core weight gradient on ROW PAIRS: [G_even | G_odd]^T [x_even | x_odd] is 128 x 128; its two
                    # diagonal blocks are the even- and odd-row halves of G^T x (the off-diagonal blocks are discarded)
                    # (the two diagonal blocks are added inside the un-folding kernel)
                    o2, cs2 = xty(g_uv.view(n // 2, 4 * cout), x.view(n // 2, 2 * cin), want_colsum=ctx.has_bias, tag="sage_wgrad")
                    ga, gb, ld = o2, o2[2 * cout:, cin:], 2 * cin
                    if ctx.has_bias:
                        g_b = torch.add(cs2[:cout], cs2[2 * cout:3 * cout], out=grad_slot(ctx.wparams[2], (cout,)))
                else:
                    o2, cs = xty(g_uv, x, want_colsum=ctx.has_bias, tag="sage_wgrad")
                    ga, gb, ld = o2, None, cin
                    if ctx.has_bias:
                        g_b = cs[:cout]
                g_wnn, g_wr = _slot_or_empty(ctx.wparams[1], w_nn), _slot_or_empty(ctx.wparams[0], w_r)
                with torch.cuda.device(gz.device):
                    _cabi.check(L.mlg_sage_fold_stacked_bwd(_vptr(ga), None if gb is None else _vptr(gb), ld, _cabi.fptr(w_nn),
                                                            _cabi.fptr(w_r), cout, cin, w_r.shape[0], _cabi.fptr(g_wnn),
                                                            _cabi.fptr(g_wr), _cabi.stream_ptr()), "mlg_sage_fold_stacked_bwd")
                fk.hold(o2, g_wnn, g_wr, g_b)
        if needs[0]:
            gx = tall_matmul(g_uv, wst.t(), tag="sage_dgrad_gemm", w_split=ctx.wst_t_split)     # dL/dx (the producer masks it itself)
        return gx, None, g_wr, g_wnn, (g_b if ctx.has_bias else None), None, None, None, None, None, None, None

    @staticmethod
    def backward(ctx, gy):
        if ctx.factored:
            return SageLayer._backward_factored(ctx, gy)
        if ctx.transform_first:
            return SageLayer._backward_transform_first(ctx, gy)
        xcat, y, wbuf, w_r, w_nn, xs_d = ctx.saved_tensors
        topo, cin = ctx.topo, ctx.cin
        cout = w_nn.shape[0]
        gy = _f32c(gy)
        if ctx.out_premasked:
            gz = gy          # the consumer already applied this layer's activation derivative
        else:
            gz = torch.ops.aten.leaky_relu_backward(gy, y, ctx.slope, True) if ctx.slope != 0.0 \
                else torch.ops.aten.threshold_backward(gy, y, 0.0)
        needs = ctx.needs_input_grad
        gx = g_wr = g_wnn = g_b = None
        if needs[2] or needs[3] or needs[4]:
            g_wcat, g_b = xty(gz, xcat, want_colsum=ctx.has_bias, tag="sage_wgrad")       # [cout, 2cin], [cout]
            g_wnn, g_wr = _slot_or_empty(ctx.wparams[1], w_nn), _slot_or_empty(ctx.wparams[0], w_r)
            with torch.cuda.device(gz.device):
                _cabi.check(_cabi.lib().mlg_sage_fold_bwd(_cabi.fptr(g_wcat), _cabi.fptr(w_nn), _cabi.fptr(w_r), cout, cin,
                                                          w_r.shape[0], _cabi.fptr(g_wnn), _cabi.fptr(g_wr),
                                                          _cabi.stream_ptr()), "mlg_sage_fold_bwd")
        g_xs = None
        if needs[0] or (ctx.rank1 and needs[1]):
            wcat_t = wbuf[0].view(cout, 2 * cin).t()
            gxcat = tall_matmul(gz, wcat_t, tag="sage_dgrad_gemm",
                                w_split=(wbuf[3].view(2 * cin, cout), wbuf[4].view(2 * cin, cout)))   # [N, 2cin]
            bw = topo.bwd
            if ctx.rank1 and not ctx.relative and topo.replicas > 1 and cin % 4 == 0 and not needs[1]:
                # first layer: only g_emb[n,:] = sum_b xs[b,n] * g_x0[b,n,:] is needed, so the backward aggregation reduces
                # over the replicas in its epilogue (per replica slice; slices added here) and g_x0 is never written
                n1 = topo.n_single
                part = gather_sum(gxcat[:, cin:], bw.rowptr, bw.col, n1, val=topo.bwd_val, pre=topo.inv_cnt,
                                  addend=gxcat[:, :cin], replicas=topo.replicas, order=topo.bwd_order,
                                  tag="sage_aggr_bwd", reduce_scale=xs_d)
                slot = grad_slot(ctx.emb_param, (n1, cin)) if ctx.emb_param is not None else None
                if part.shape[0] > n1:
                    g_emb = torch.sum(part.view(-1, n1, cin), 0, out=slot) if slot is not None else part.view(-1, n1, cin).sum(0)
                else:
                    g_emb = part
                return g_emb, None, g_wr, g_wnn, (g_b if ctx.has_bias else None), None, None, None, None, None, None, None
            gx = gather_sum(gxcat[:, cin:], bw.rowptr, bw.col, topo.n_single, val=topo.bwd_val, pre=topo.inv_cnt,
                            addend=gxcat[:, :cin], replicas=topo.replicas, order=topo.bwd_order, tag="sage_aggr_bwd",
                            mask=None if ctx.in_slope is None else xcat[:, :cin],
                            mask_slope=0.0 if ctx.in_slope is None else ctx.in_slope)
            if ctx.relative:
                gx = gx - gxcat[:, cin:]
            if ctx.rank1:
                L = _cabi.lib()
                n1 = topo.n_single
                if needs[1]:
                    # gradient w.r.t. the node values: g_xs[b,n] = <g_x0[b,n,:], emb[n,:]>
                    g_xs = _embed_scale_input_grad(gx, ctx.emb_d, topo.replicas, n1, cin).view(ctx.xs_shape)
                g_emb = None
                if needs[0]:
                    # gradient of the rank-1 input w.r.t. node_embedding: g_emb[n,:] = sum_b xs[b,n] * g_x0[b,n,:]
                    g_emb = torch.empty(n1, cin, dtype=torch.float32, device=gx.device)
                    with torch.cuda.device(gx.device), _cabi.span("embed_scale_bwd", 4 * gx.numel()):
                        _cabi.check(L.mlg_embed_scale_bwd(_cabi.fptr(xs_d), _cabi.fptr(gx), topo.replicas, n1, cin,
                                                          _cabi.fptr(g_emb), _cabi.stream_ptr()), "mlg_embed_scale_bwd")
                gx = g_emb
        return gx, g_xs, g_wr, g_wnn, (g_b if ctx.has_bias else None), None, None, None, None, None, None, None


class RankOne:
    """Layer input x0[b*N+n, :] = xs[b*N+n] * emb[n, :] kept in factored form (MultilevelGNN's embed-scale
    prologue, models/multilevel_gnn.py:150-151) so that the first SAGE layer can consume it without the
    [B*N, C] tensor ever being written; ``materialize()`` produces it for any consumer that needs it."""

    def __init__(self, xs, emb):
        self.xs, self.emb = xs, emb

    @property
    def shape(self):
        return (self.xs.numel(), self.emb.shape[1])

    def dim(self):
        return 2

    def materialize(self):
        return EmbedScale.apply(self.xs, self.emb)


class EmbedScale(torch.autograd.Function):
    """x0[b*N+n,:] = x[b*N+n] * node_embedding[n,:]   (models/multilevel_gnn.py:150-151)."""

    @staticmethod
    def forward(ctx, xs, emb):
        L = _cabi.lib()
        _cabi.require_cuda(xs, emb)
        N, C = emb.shape
        xs_d = _f32c(xs.detach().reshape(-1))
        emb_d = _f32c(emb.detach())
        B = xs_d.numel() // N
        out = torch.empty(B * N, C, dtype=torch.float32, device=emb.device)
        with torch.cuda.device(emb.device):
            _cabi.check(L.mlg_embed_scale_fwd(_cabi.fptr(xs_d), _cabi.fptr(emb_d), B, N, C, _cabi.fptr(out),
                                              _cabi.stream_ptr()), "mlg_embed_scale_fwd")
        ctx.save_for_backward(xs_d, emb_d if ctx.needs_input_grad[0] else None)
        ctx.dims = (B, N, C)
        ctx.xs_shape = xs.shape
        return out

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        xs_d, emb_d = ctx.saved_tensors
        B, N, C = ctx.dims
        g = _f32c(g)
        g_xs = g_emb = None
        if ctx.needs_input_grad[0]:
            g_xs = _embed_scale_input_grad(g, emb_d, B, N, C).view(ctx.xs_shape)
        if ctx.needs_input_grad[1] or not ctx.needs_input_grad[0]:
            g_emb = torch.empty(N, C, dtype=torch.float32, device=g.device)
            with torch.cuda.device(g.device):
                _cabi.check(L.mlg_embed_scale_bwd(_cabi.fptr(xs_d), _cabi.fptr(g), B, N, C, _cabi.fptr(g_emb),
                                                  _cabi.stream_ptr()), "mlg_embed_scale_bwd")
        return g_xs, g_emb


def _embed_scale_input_grad(g_x0, emb, B, N, C):
    """g_xs [B*N] = <g_x0[b*N+n, :], emb[n, :]>: the gradient w.r.t. the node values of x0 = xs * emb (mlg_embed_scale_bwd_xs)."""
    g_xs = torch.empty(B * N, dtype=torch.float32, device=g_x0.device)
    with torch.cuda.device(g_x0.device), _cabi.span("embed_scale_bwd_xs", 4 * (g_x0.numel() + N * C + B * N)):
        _cabi.check(_cabi.lib().mlg_embed_scale_bwd_xs(_cabi.fptr(_f32c(g_x0)), _cabi.fptr(_f32c(emb)), B, N, C,
                                                       _cabi.fptr(g_xs), _cabi.stream_ptr()), "mlg_embed_scale_bwd_xs")
    return g_xs


class LayerNormFn(torch.autograd.Function):
    """nn.LayerNorm over the last axis of a tall [rows, C] fp32 tensor (mlg_layernorm_fwd / _bwd): one warp per row,
    input gradient and gamma / beta gradients in one backward pass."""

    MIN_ROWS = 4096

    @staticmethod
    def supported(x, normalized_shape):
        return (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and len(normalized_shape) == 1
                and x.shape[1] == normalized_shape[0] and x.shape[0] >= LayerNormFn.MIN_ROWS
                and bool(_cabi.lib().mlg_layernorm_supported(x.shape[1])))

    @staticmethod
    def forward(ctx, x, weight, bias, eps, relu=False):
        """``relu``: max(LN(x), 0) in the same pass (mlg_layernorm_relu_fwd / _bwd)."""
        L = _cabi.lib()
        xd = _f32c(x.detach())
        rows, C = xd.shape
        y = torch.empty_like(xd)
        mean = torch.empty(rows, dtype=torch.float32, device=xd.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=xd.device)
        wd = None if weight is None else _f32c(weight.detach())
        bd = None if bias is None else _f32c(bias.detach())
        fn, name = (L.mlg_layernorm_relu_fwd, "mlg_layernorm_relu_fwd") if relu else (L.mlg_layernorm_fwd, "mlg_layernorm_fwd")
        with torch.cuda.device(xd.device), _cabi.span("layernorm_fwd", 8 * rows * C):
            _cabi.check(fn(_cabi.fptr(xd), _cabi.fptr(wd, True), _cabi.fptr(bd, True), rows, C, float(eps),
                           _cabi.fptr(y), _cabi.fptr(mean), _cabi.fptr(rstd), _cabi.stream_ptr()), name)
        ctx.save_for_backward(xd, wd, bd if relu else None, mean, rstd)
        ctx.has_w, ctx.has_b, ctx.relu = weight is not None, bias is not None, bool(relu)
        return y

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        xd, wd, bd, mean, rstd = ctx.saved_tensors
        rows, C = xd.shape
        g = _f32c(g)
        gx = torch.empty_like(xd)
        need_w = ctx.has_w and ctx.needs_input_grad[1]
        need_b = ctx.has_b and ctx.needs_input_grad[2]
        dgam = torch.empty(C, dtype=torch.float32, device=xd.device) if need_w else None
        dbet = torch.empty(C, dtype=torch.float32, device=xd.device) if need_b else None
        ws_bytes = L.mlg_layernorm_bwd_workspace_bytes(rows, C)
        ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=xd.device)
        with torch.cuda.device(xd.device), _cabi.span("layernorm_bwd", 12 * rows * C):
            if ctx.relu:
                _cabi.check(L.mlg_layernorm_relu_bwd(_cabi.fptr(xd), _cabi.fptr(g), _cabi.fptr(wd, True), _cabi.fptr(bd, True),
                                                     _cabi.fptr(mean), _cabi.fptr(rstd), rows, C, _cabi.fptr(gx),
                                                     _cabi.fptr(dgam, True), _cabi.fptr(dbet, True), _cabi.fptr(ws), ws_bytes,
                                                     _cabi.stream_ptr()), "mlg_layernorm_relu_bwd")
            else:
                _cabi.check(L.mlg_layernorm_bwd(_cabi.fptr(xd), _cabi.fptr(g), _cabi.fptr(wd, True), _cabi.fptr(mean),
                                                _cabi.fptr(rstd), rows, C, _cabi.fptr(gx), _cabi.fptr(dgam, True),
                                                _cabi.fptr(dbet, True), _cabi.fptr(ws), ws_bytes, _cabi.stream_ptr()),
                            "mlg_layernorm_bwd")
        return gx, dgam, dbet, None, None


class MaxPoolCL(torch.autograd.Function):
    """nn.MaxPool2d((kh, kw)) (stride = kernel, floor mode; multilevel_gnn.py:286) of a [B, C, H, W] tensor whose MEMORY is
    channel-last (the permuted view the pooled features / 1x1 convs produce): one kernel, NCHW-contiguous output, no
    layout copy either way (mlg_maxpool_cl_fwd / _bwd)."""

    @staticmethod
    def forward(ctx, x, kh, kw):
        L = _cabi.lib()
        _cabi.require_cuda(x)
        B, C, H, W = x.shape
        x_cl = x.detach().permute(0, 2, 3, 1)
        if not x_cl.is_contiguous() or x.dtype != torch.float32:
            raise ValueError("MaxPoolCL needs a float32 tensor that is contiguous in channel-last memory order")
        out = torch.empty(B, C, H // kh, W // kw, dtype=torch.float32, device=x.device)
        arg = torch.empty(out.shape, dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            _cabi.check(L.mlg_maxpool_cl_fwd(_cabi.fptr(x_cl), B, H, W, C, kh, kw, _cabi.fptr(out),
                                             ctypes_ptr(arg), _cabi.stream_ptr()), "mlg_maxpool_cl_fwd")
        ctx.save_for_backward(arg)
        ctx.dims = (B, C, H, W, kh, kw)
        return out

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        (arg,) = ctx.saved_tensors
        B, C, H, W, kh, kw = ctx.dims
        g = _f32c(g)
        gx_cl = torch.empty(B, H, W, C, dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            _cabi.check(L.mlg_maxpool_cl_bwd(_cabi.fptr(g), ctypes_ptr(arg), B, H, W, C, kh, kw, _cabi.fptr(gx_cl),
                                             _cabi.stream_ptr()), "mlg_maxpool_cl_bwd")
        return gx_cl.permute(0, 3, 1, 2), None, None


def ctypes_ptr(t):
    import ctypes
    return ctypes.c_void_p(t.data_ptr())


class PathwayPool(torch.autograd.Function):
    """Gene -> pathway pool (models/multilevel_gnn.py:205-239).
    forward(x [B*N,C], w [G,P] (already * info_mask), vm [B*N] or None, layout) -> [B,C,S,P], returned as the
    permute(0,3,1,2) VIEW of the channel-last buffer [B,S,P,C] the kernel writes."""

    @staticmethod
    def forward(ctx, x, w, vm, layout, in_slope=None, w_mask=None, link=None):
        """``in_slope``: x is the output of a (Leaky)ReLU with that slope whose producer expects dL/dz (see SageLayer).
        ``w_mask`` [G, 1] or [G]: the projection weights are w * w_mask (learnable_pca_params * info_mask,
        multilevel_gnn.py:222); the product and its backward are folded in (the gradient returned for ``w`` is dL/dw).
        ``vm`` is differentiable: when it requires grad, the backward returns dL/dvm from the same pass as dL/dx."""
        L = _cabi.lib()
        _cabi.require_cuda(x, w)
        vm = None if vm is None else vm.detach()
        ctx.w_param = w
        ctx.w_mask = None
        if w_mask is not None:
            ctx.w_mask = _f32c(w_mask.detach().reshape(-1))
            w = w.detach() * ctx.w_mask.reshape(-1, 1)
        xd, wd = _f32c(x.detach()), _f32c(w.detach())
        B, N, G, S = layout.B, layout.N, layout.G, layout.S
        C, P = xd.shape[1], wd.shape[1]
        out_cl = torch.empty(B, S, P, C, dtype=torch.float32, device=xd.device)
        nbytes = 4 * C * B * N + 4 * B * N + 12 * G + 4 * B * C * S * P              # SURVEY.md section 8d
        with torch.cuda.device(xd.device), _cabi.span("pool_fwd", nbytes):
            _cabi.check(L.mlg_pool_fwd(_cabi.fptr(xd), _cabi.fptr(vm, True), _cabi.lptr(layout.match),
                                       _cabi.fptr(wd), _cabi.iptr(layout.seg.rowptr), _cabi.iptr(layout.seg.col),
                                       B, N, C, G, S, P, int(layout.wrap_negative), _cabi.fptr(out_cl),
                                       _cabi.stream_ptr()), "mlg_pool_fwd")
        ctx.save_for_backward(xd, wd)
        ctx.vm, ctx.layout = vm, layout
        ctx.in_slope = None if in_slope is None else float(in_slope)
        ctx.link = link       # shared with the SageLayer that produced x (see its forward): layout of the gradient handed back
        return out_cl.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        xd, wd = ctx.saved_tensors
        lay, vm = ctx.layout, ctx.vm
        B, N, G, S = lay.B, lay.N, lay.G, lay.S
        C, P = xd.shape[1], wd.shape[1]
        g_cl = g.float().permute(0, 2, 3, 1).contiguous()     # [B,S,P,C]; no copy when g is already channel-last
        gx = gw = None
        if ctx.needs_input_grad[2]:
            return PathwayPool._backward_with_vm(ctx, g_cl)
        if ctx.needs_input_grad[0] and ctx.needs_input_grad[1] and C <= 128 and not lay.wrap_negative:
            slot = grad_slot(ctx.w_param, wd.shape)
            gx, gw = torch.empty_like(xd), (slot if slot is not None else torch.empty_like(wd))
            node = lay.node_csr
            ws = torch.empty(B * G * P, dtype=torch.float32, device=xd.device)
            link = getattr(ctx, "link", None)
            node_major = bool(link is not None and link.get("gz_node_major") and ctx.in_slope is not None
                              and L.mlg_pool_bwd_node_major_supported(C, lay.replicas))
            with torch.cuda.device(xd.device), _cabi.span("pool_bwd", 2 * (4 * C * B * N) + 4 * B * C * S * P):
                _cabi.check(L.mlg_pool_bwd_layout(_cabi.fptr(g_cl), _cabi.fptr(xd), _cabi.fptr(vm, True), _cabi.fptr(wd),
                                                  _cabi.iptr(node.rowptr), _cabi.iptr(node.col), _cabi.iptr(lay.seg_of_slot),
                                                  B, N, C, G, S, P, lay.replicas, _cabi.fptr(gx), _cabi.fptr(gw), _cabi.fptr(ws),
                                                  0 if ctx.in_slope is None else 1, 0.0 if ctx.in_slope is None else ctx.in_slope,
                                                  _cabi.fptr(ctx.w_mask, True), 1 if node_major else 0, _cabi.stream_ptr()),
                            "mlg_pool_bwd_layout")
            if link is not None:
                link["gz_written_node_major"] = node_major      # read (and cleared) by the producer layer's backward
            return gx, gw, None, None, None, None, None
        with torch.cuda.device(xd.device):
            if ctx.needs_input_grad[0]:
                gx = torch.empty_like(xd)
                node = lay.node_csr
                with _cabi.span("pool_bwd_x", 4 * C * B * N + 4 * B * C * S * P):
                    _cabi.check(L.mlg_pool_bwd_x(_cabi.fptr(g_cl), _cabi.fptr(vm, True), _cabi.fptr(wd),
                                                 _cabi.iptr(node.rowptr), _cabi.iptr(node.col),
                                                 _cabi.iptr(lay.seg_of_slot), B, N, C, G, S, P, lay.replicas,
                                                 _cabi.fptr(gx), _cabi.stream_ptr()), "mlg_pool_bwd_x")
            if ctx.needs_input_grad[1]:
                gw = torch.empty_like(wd)
                with _cabi.span("pool_bwd_w", 4 * C * B * N + 4 * B * C * S * P):
                    _cabi.check(L.mlg_pool_bwd_w(_cabi.fptr(g_cl), _cabi.fptr(xd), _cabi.fptr(vm, True),
                                                 _cabi.lptr(lay.match), _cabi.lptr(lay.raw_indice), B, N, C, G, S, P,
                                                 int(lay.wrap_negative), lay.replicas, _cabi.fptr(gw), _cabi.stream_ptr()),
                                "mlg_pool_bwd_w")
        if gx is not None and ctx.in_slope is not None:      # unfused fallback of the activation-derivative mask
            gx = torch.where(xd > 0, gx, gx * ctx.in_slope)
        if gw is not None and ctx.w_mask is not None:
            gw = gw * ctx.w_mask.reshape(-1, 1)
        if getattr(ctx, "link", None) is not None:
            ctx.link["gz_written_node_major"] = False
        return gx, gw, None, None, None, None, None

    @staticmethod
    def _backward_with_vm(ctx, g_cl):
        """Backward when the value mask vm (batch.x) needs a gradient: g_x and g_vm in one pass (mlg_pool_bwd_vm), the weight
        gradient in the same pass when it is needed too (or by mlg_pool_bwd_w where the fused pass does not apply); the
        node-major hand-shake with the producing layer works as on the training path."""
        L = _cabi.lib()
        xd, wd = ctx.saved_tensors
        lay, vm = ctx.layout, ctx.vm
        B, N, G, S = lay.B, lay.N, lay.G, lay.S
        C, P = xd.shape[1], wd.shape[1]
        if C > 128:
            raise NotImplementedError("PathwayPool: the gradient w.r.t. the value mask needs C <= 128 (got %d)" % C)
        fused_w = ctx.needs_input_grad[1] and not lay.wrap_negative
        gx, g_vm = torch.empty_like(xd), torch.empty_like(vm)
        gw = ws = None
        if fused_w:
            slot = grad_slot(ctx.w_param, wd.shape)
            gw = slot if slot is not None else torch.empty_like(wd)
            ws = torch.empty(B * G * P, dtype=torch.float32, device=xd.device)
        node = lay.node_csr
        link = getattr(ctx, "link", None)
        node_major = bool(link is not None and link.get("gz_node_major") and ctx.in_slope is not None
                          and L.mlg_pool_bwd_node_major_supported(C, lay.replicas))
        with torch.cuda.device(xd.device), _cabi.span("pool_bwd_vm", 2 * (4 * C * B * N) + 4 * B * C * S * P + 8 * B * N):
            _cabi.check(L.mlg_pool_bwd_vm(_cabi.fptr(g_cl), _cabi.fptr(xd), _cabi.fptr(vm), _cabi.fptr(wd),
                                          _cabi.iptr(node.rowptr), _cabi.iptr(node.col), _cabi.iptr(lay.seg_of_slot),
                                          B, N, C, G, S, P, lay.replicas, _cabi.fptr(gx), _cabi.fptr(gw, True),
                                          _cabi.fptr(ws, True), 0 if ctx.in_slope is None else 1,
                                          0.0 if ctx.in_slope is None else ctx.in_slope, _cabi.fptr(ctx.w_mask, True),
                                          1 if node_major else 0, _cabi.fptr(g_vm), _cabi.stream_ptr()), "mlg_pool_bwd_vm")
            if ctx.needs_input_grad[1] and not fused_w:
                gw = torch.empty_like(wd)
                with _cabi.span("pool_bwd_w", 4 * C * B * N + 4 * B * C * S * P):
                    _cabi.check(L.mlg_pool_bwd_w(_cabi.fptr(g_cl), _cabi.fptr(xd), _cabi.fptr(vm),
                                                 _cabi.lptr(lay.match), _cabi.lptr(lay.raw_indice), B, N, C, G, S, P,
                                                 int(lay.wrap_negative), lay.replicas, _cabi.fptr(gw), _cabi.stream_ptr()),
                                "mlg_pool_bwd_w")
                if ctx.w_mask is not None:
                    gw = gw * ctx.w_mask.reshape(-1, 1)
        if link is not None:
            link["gz_written_node_major"] = node_major      # read (and cleared) by the producer layer's backward
        return (gx if ctx.needs_input_grad[0] else None), gw, g_vm, None, None, None, None


def _drop_bits(n, device):
    """Uniform int32 words in [0, 2^31) from torch's CUDA generator (graph-safe; torch.manual_seed applies): the dropout
    masks of the fused head kernels (kept iff bits >= p * 2^31)."""
    return torch.empty(n, dtype=torch.int32, device=device).random_()


class HeadConvPool(torch.autograd.Function):
    """Conv2d(32->32,1x1)+ReLU, Conv2d(32->64,1x1)+ReLU, MaxPool2d((kh,kw)), Dropout(p), flatten, cat(age) of
    MultilevelGNN's head (models/multilevel_gnn.py:262-288) as one kernel each way (mlg_head_conv_pool_fwd / _bwd).

    forward(feat [B,32,H,W] whose MEMORY is channel-last, W1 [32,32,1,1], b1, W2 [64,32,1,1], b2, age [B] or None,
            kh, kw, p, training) -> a0 [B, 64*(H//kh)*(W//kw) (+1)]"""

    @staticmethod
    def supported(feat, conv1, conv2):
        return (feat.is_cuda and feat.dtype == torch.float32 and conv1.kernel_size == (1, 1) and conv2.kernel_size == (1, 1)
                and conv1.bias is not None and conv2.bias is not None
                and bool(_cabi.lib().mlg_head_conv_pool_supported(conv1.in_channels, conv1.out_channels, conv2.out_channels))
                and conv2.in_channels == conv1.out_channels and feat.shape[1] == conv1.in_channels)

    @staticmethod
    def forward(ctx, feat, W1, b1, W2, b2, age, kh, kw, p, training):
        L = _cabi.lib()
        _cabi.require_cuda(feat, W1, W2)
        B, C, H, W = feat.shape
        x_cl = feat.detach().permute(0, 2, 3, 1)
        if not x_cl.is_contiguous():
            x_cl = x_cl.contiguous()
        Ho, Wo = H // kh, W // kw
        F_ = W2.shape[0] * Ho * Wo
        ld = F_ + (1 if age is not None else 0)
        p = float(p) if training else 0.0
        bits = _drop_bits(B * F_, feat.device) if p > 0.0 else None
        a0 = torch.empty(B, ld, dtype=torch.float32, device=feat.device)
        w1, w2 = _f32c(W1.detach()).view(W1.shape[0], -1), _f32c(W2.detach()).view(W2.shape[0], -1)
        b1d, b2d = _f32c(b1.detach()), _f32c(b2.detach())
        aged = None if age is None else _f32c(age.detach().reshape(-1))
        nbytes = 4 * (x_cl.numel() + a0.numel())
        with torch.cuda.device(feat.device), _cabi.span("head_conv_pool_fwd", nbytes):
            _cabi.check(L.mlg_head_conv_pool_fwd(_cabi.fptr(x_cl), _cabi.fptr(w1), _cabi.fptr(b1d), _cabi.fptr(w2),
                                                 _cabi.fptr(b2d), _cabi.fptr(aged, True), _cabi.iptr(bits, True), p, B, H, W,
                                                 int(kh), int(kw), _cabi.fptr(a0), ld, _cabi.stream_ptr()),
                        "mlg_head_conv_pool_fwd")
        ctx.save_for_backward(x_cl, w1, b1d, w2, b2d, bits)
        ctx.dims = (B, H, W, int(kh), int(kw), p, ld)
        ctx.params = (W1, b1, W2, b2)
        return a0

    @staticmethod
    def backward(ctx, g):
        L = _cabi.lib()
        x_cl, w1, b1d, w2, b2d, bits = ctx.saved_tensors
        B, H, W, kh, kw, p, ld = ctx.dims
        W1, b1, W2, b2 = ctx.params
        g = _f32c(g)
        gx = torch.empty_like(x_cl)
        dev = x_cl.device

        def dest(param):
            slot = grad_slot(param, param.shape)
            return slot if slot is not None else torch.empty(param.shape, dtype=torch.float32, device=dev)

        if any(ctx.needs_input_grad[1:5]):
            gW1, gb1, gW2, gb2 = dest(W1), dest(b1), dest(W2), dest(b2)
            ws_bytes = L.mlg_head_conv_pool_bwd_workspace_bytes(B, H, W, kh, kw)
            ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=dev)
        else:      # input gradient only: the kernel skips the weight-gradient partials and their reduce
            gW1 = gb1 = gW2 = gb2 = ws = None
            ws_bytes = 0
        with torch.cuda.device(dev), _cabi.span("head_conv_pool_bwd", 4 * (2 * x_cl.numel() + g.numel())):
            _cabi.check(L.mlg_head_conv_pool_bwd(_cabi.fptr(g), ld, _cabi.fptr(x_cl), _cabi.fptr(w1), _cabi.fptr(b1d),
                                                 _cabi.fptr(w2), _cabi.fptr(b2d), _cabi.iptr(bits, True), p, B, H, W, kh, kw,
                                                 _cabi.fptr(gx), _cabi.fptr(gW1, True), _cabi.fptr(gb1, True),
                                                 _cabi.fptr(gW2, True), _cabi.fptr(gb2, True), _cabi.fptr(ws, True), ws_bytes,
                                                 _cabi.stream_ptr()),
                        "mlg_head_conv_pool_bwd")
        g_age = g[:, ld - 1] if (ctx.needs_input_grad[5]) else None
        return gx.permute(0, 3, 1, 2), gW1, gb1, gW2, gb2, g_age, None, None, None, None


class HeadMLP(torch.autograd.Function):
    """Linear(K->D)+ReLU+Dropout(p), Linear(D->2), Softmax (models/multilevel_gnn.py:104-110,288-290) and, when the target
    is given, BCELoss(weight) (train.py:60,118) in two launches forward, one backward (mlg_head_mlp_fwd / _bwd).

    forward(a0 [B,K], W0 [D,K], b0, W3 [2,D], b3, p, training, y [B,2] or None, weight [B,2] or None) -> (pred [B,2], bce [])"""

    @staticmethod
    def supported(a0, lin0, lin3):
        return (a0.is_cuda and a0.dtype == torch.float32 and a0.dim() == 2 and a0.shape[0] <= 64 and lin3.out_features == 2
                and lin0.out_features % 32 == 0 and lin0.out_features <= 512 and lin0.bias is not None
                and lin3.bias is not None and lin3.in_features == lin0.out_features and a0.shape[1] == lin0.in_features)

    @staticmethod
    def forward(ctx, a0, W0, b0, W3, b3, p, training, y, weight):
        L = _cabi.lib()
        _cabi.require_cuda(a0, W0, W3)
        ctx.set_materialize_grads(False)
        R, K = a0.shape
        D = W0.shape[0]
        dev = a0.device
        a0d = a0.detach()
        a0d = a0d if (a0d.stride(1) == 1 and a0d.dtype == torch.float32) else _f32c(a0d)
        w0, w3 = _f32c(W0.detach()), _f32c(W3.detach())
        b0d, b3d = _f32c(b0.detach()), _f32c(b3.detach())
        p = float(p) if training else 0.0
        bits = _drop_bits(R * D, dev) if p > 0.0 else None
        yd = None if y is None else _f32c(y.detach().reshape(R, 2))
        wd = None if weight is None else _f32c(weight.detach().expand(R, 2))
        a1 = torch.empty(R, D, dtype=torch.float32, device=dev)
        pred = torch.empty(R, 2, dtype=torch.float32, device=dev)
        loss = torch.zeros((), dtype=torch.float32, device=dev) if yd is None else torch.empty((), dtype=torch.float32, device=dev)
        ws_bytes = L.mlg_head_mlp_workspace_bytes(R, D, K)
        ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev), _cabi.span("head_mlp_fwd", 4 * (D * K + R * K)):
            _cabi.check(L.mlg_head_mlp_fwd(_vptr(a0d), a0d.stride(0), _cabi.fptr(w0), _cabi.fptr(b0d), _cabi.fptr(w3),
                                           _cabi.fptr(b3d), _cabi.iptr(bits, True), p, _cabi.fptr(yd, True),
                                           _cabi.fptr(wd, True), R, D, K, _cabi.fptr(a1), _cabi.fptr(pred),
                                           _vptr(loss), _cabi.fptr(ws), ws_bytes, _cabi.stream_ptr()), "mlg_head_mlp_fwd")
        ctx.save_for_backward(a0d, a1, pred, w0, w3, yd, wd)
        ctx.p = p
        ctx.params = (W0, b0, W3, b3)
        if yd is None:
            ctx.mark_non_differentiable(loss)
        return pred, loss

    @staticmethod
    def backward(ctx, g_pred, g_loss):
        L = _cabi.lib()
        a0d, a1, pred, w0, w3, yd, wd = ctx.saved_tensors
        if g_pred is None and (g_loss is None or yd is None):
            return (None,) * 9
        W0, b0, W3, b3 = ctx.params
        R, K = a0d.shape
        D = w0.shape[0]
        dev = a0d.device
        gp = None if g_pred is None else _f32c(g_pred)
        gl = None if (g_loss is None or yd is None) else _f32c(g_loss).reshape(1)

        def dest(param):
            slot = grad_slot(param, param.shape)
            return slot if slot is not None else torch.empty(param.shape, dtype=torch.float32, device=dev)

        if any(ctx.needs_input_grad[1:5]):
            gW0, gb0, gW3, gb3 = dest(W0), dest(b0), dest(W3), dest(b3)
        else:      # input gradient only: one pass over W0, no weight-gradient slices
            gW0 = gb0 = gW3 = gb3 = None
        g_a0 = torch.empty(R, K, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(dev), _cabi.span("head_mlp_bwd", 4 * (2 * D * K + 2 * R * K)):
            _cabi.check(L.mlg_head_mlp_bwd(_cabi.fptr(gp, True), _cabi.fptr(gl, True), _cabi.fptr(pred), _cabi.fptr(yd, True),
                                           _cabi.fptr(wd, True), _vptr(a0d), a0d.stride(0), _cabi.fptr(a1), _cabi.fptr(w0),
                                           _cabi.fptr(w3), ctx.p, R, D, K, _cabi.fptr(g_a0, True), K, _cabi.fptr(gW0, True),
                                           _cabi.fptr(gb0, True), _cabi.fptr(gW3, True), _cabi.fptr(gb3, True),
                                           _cabi.stream_ptr()),
                        "mlg_head_mlp_bwd")
        if AFTER_HEAD_BACKWARD is not None:
            AFTER_HEAD_BACKWARD()
        return g_a0, gW0, gb0, gW3, gb3, None, None, None, None


class DiffPoolFused(torch.autograd.Function):
    """DiffPool.forward at the reference's size (models/diff_pooling.py:116-133; 146 -> 37 -> 10 nodes) as one kernel per
    direction (mlg_diffpool_fwd / _bwd, csrc/diffpool_fused.cu).

    forward(x [b,n,c], adj [n,n], dims, *weights) -> (out [b,k,h], link, entropy); ``weights``: 9 tensors per layer in
    the order of include/mlg_b200.h; ``dims``: tuple of (n, c, k, h) per layer."""

    @staticmethod
    def _tables(weights, dims):
        import ctypes
        ws = [_f32c(w.detach()) for w in weights]
        warr = (ctypes.c_void_p * len(ws))(*[w.data_ptr() for w in ws])
        darr = (ctypes.c_int64 * (4 * len(dims)))(*[int(v) for d in dims for v in d])
        return ws, warr, darr

    _NORMS = {}

    @staticmethod
    def _norms(dims, b, device):
        """(numel(adj_l), b * n_l) per layer as device tensors, uploaded once per (dims, b, device)."""
        key = (tuple(tuple(d) for d in dims), b, str(device))
        got = DiffPoolFused._NORMS.get(key)
        if got is None:
            got = (torch.tensor([float(d[0] * d[0] * (1 if i == 0 else b)) for i, d in enumerate(dims)], device=device),
                   torch.tensor([float(b * d[0]) for d in dims], device=device))
            DiffPoolFused._NORMS[key] = got
        return got

    @staticmethod
    def supported(dims):
        import ctypes
        darr = (ctypes.c_int64 * (4 * len(dims)))(*[int(v) for d in dims for v in d])
        return 1 <= len(dims) <= 2 and bool(_cabi.lib().mlg_diffpool_supported(len(dims), darr))

    @staticmethod
    def forward(ctx, x, adj, dims, *weights):
        L = _cabi.lib()
        _cabi.require_cuda(x, adj, *weights)
        xd, ad = _f32c(x.detach()), _f32c(adj.detach())
        b = xd.shape[0]
        ws, warr, darr = DiffPoolFused._tables(weights, dims)
        nl = len(dims)
        out = torch.empty(b, dims[-1][2], dims[-1][3], dtype=torch.float32, device=xd.device)
        stats = torch.empty(b, nl, 2, dtype=torch.float32, device=xd.device)
        # forward state for backward (S, Z, pooled X / A, row norms: ~90 KB per sample at the reference size) -- only when a
        # backward pass can follow; without it the backward kernel recomputes the forward pass
        state = None
        if any(ctx.needs_input_grad):
            state = torch.empty(b * int(L.mlg_diffpool_state_floats(nl, darr)), dtype=torch.float32, device=xd.device)
        flops = 2.0 * b * sum(n * n * c + 2 * n * c * (k + h) + n * k * h + 2 * n * n * k + n * k * k for n, c, k, h in dims)
        with torch.cuda.device(xd.device), _cabi.span("diffpool_fwd", flops):
            _cabi.check(L.mlg_diffpool_fwd(_cabi.fptr(xd), _cabi.fptr(ad), warr, nl, darr, b, _cabi.fptr(out),
                                           _cabi.fptr(stats), _cabi.fptr(state) if state is not None else None,
                                           _cabi.stream_ptr()), "mlg_diffpool_fwd")
        # link_l = ||adj_l - S S^T||_F / numel(adj_l) over the whole batch (adj_0 is the shared [n, n] matrix, deeper
        # adjacencies are batched [b, k, k]); entropy_l = mean over (sample, node)
        tot = stats.sum(0)                                              # [layers, 2]
        numel, rows = DiffPoolFused._norms(dims, b, xd.device)
        fro = tot[:, 0].sqrt()
        link = (fro / numel).sum()
        ent = (tot[:, 1] / rows).sum()
        ctx.save_for_backward(xd, ad, fro, numel, rows, *ws)
        ctx.dims = dims
        ctx.state = state
        ctx.n_weights = len(weights)
        ctx.set_materialize_grads(False)
        return out, link, ent

    @staticmethod
    def backward(ctx, g_out, g_link, g_ent):
        L = _cabi.lib()
        xd, ad, fro, numel, rows = ctx.saved_tensors[:5]
        ws = list(ctx.saved_tensors[5:])
        dims = ctx.dims
        nl = len(dims)
        b = xd.shape[0]
        dev = xd.device
        import ctypes
        warr = (ctypes.c_void_p * len(ws))(*[w.data_ptr() for w in ws])
        darr = (ctypes.c_int64 * (4 * nl))(*[int(v) for d in dims for v in d])
        g_out = torch.zeros(b, dims[-1][2], dims[-1][3], dtype=torch.float32, device=dev) if g_out is None else _f32c(g_out)
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        gl = zero if g_link is None else g_link.float()
        ge = zero if g_ent is None else g_ent.float()
        coef = torch.stack([gl / (fro * numel), (ge / rows)], dim=1).contiguous()     # [layers, 2]
        nfl = int(L.mlg_diffpool_grad_floats(nl, darr))
        ctas = int(L.mlg_diffpool_ctas(b))
        gx = torch.empty_like(xd)
        gw = torch.empty(nfl, dtype=torch.float32, device=dev)
        wsp = torch.empty(ctas * nfl, dtype=torch.float32, device=dev)
        flops = 6.0 * b * sum(n * n * c + 2 * n * c * (k + h) + n * k * h + 2 * n * n * k + n * k * k for n, c, k, h in dims)
        with torch.cuda.device(dev), _cabi.span("diffpool_bwd", flops):
            _cabi.check(L.mlg_diffpool_bwd(_cabi.fptr(g_out), _cabi.fptr(coef), _cabi.fptr(xd), _cabi.fptr(ad), warr, nl, darr,
                                           b, _cabi.fptr(gx), _cabi.fptr(gw),
                                           _cabi.fptr(ctx.state) if ctx.state is not None else None, _cabi.fptr(wsp),
                                           wsp.numel() * 4, _cabi.stream_ptr()), "mlg_diffpool_bwd")
        grads, off = [], 0
        for w in ws:
            grads.append(gw[off:off + w.numel()].view_as(w))
            off += w.numel()
        return (gx, None, None) + tuple(grads)


class DecoderGrouped(torch.autograd.Function):
    """All per-pathway decoder blocks Linear-ReLU-Linear of VAE.foreach_decoder (models/vae.py:54-74,216-222) in one launch
    per direction (mlg_decoder_fwd / _bwd, csrc/decoder_grouped.cu).  x [B, S, F], packed: every block's parameters (layout:
    models/decoder.py), table [S, 8] int64 on the device -> pred [B, total_out]."""

    @staticmethod
    def forward(ctx, x, packed, table, d_max, total_out, total_hidden):
        L = _cabi.lib()
        _cabi.require_cuda(x, packed, table)
        xd, pd = _f32c(x.detach()), _f32c(packed.detach())
        B, S, F = xd.shape
        out = torch.empty(B, total_out, dtype=torch.float32, device=xd.device)
        need = any(ctx.needs_input_grad)
        h = torch.empty(B, total_hidden, dtype=torch.float32, device=xd.device) if need else None
        flops = 2.0 * B * (F * total_hidden + pd.numel())
        with torch.cuda.device(xd.device), _cabi.span("decoder_fwd", flops):
            _cabi.check(L.mlg_decoder_fwd(_cabi.fptr(xd), _cabi.fptr(pd), _cabi.lptr(table), B, S, F, d_max, total_out,
                                          total_hidden, _cabi.fptr(out), _cabi.fptr(h, allow_none=True),
                                          _cabi.stream_ptr()), "mlg_decoder_fwd")
        if need:
            ctx.save_for_backward(xd, pd, table, h)
            ctx.meta = (d_max, total_out, total_hidden)
            ctx.packed_param = packed
        return out

    @staticmethod
    def backward(ctx, g_out):
        L = _cabi.lib()
        xd, pd, table, h = ctx.saved_tensors
        d_max, total_out, total_hidden = ctx.meta
        B, S, F = xd.shape
        g = _f32c(g_out)
        gx = torch.empty_like(xd) if ctx.needs_input_grad[0] else None
        # every element of a block's arrays has exactly one writer; the alignment gaps between the arrays stay zero
        gp = grad_slot(ctx.packed_param, pd.shape)
        if gp is None:
            gp = torch.zeros_like(pd)
        flops = 4.0 * B * (F * total_hidden + pd.numel())
        with torch.cuda.device(xd.device), _cabi.span("decoder_bwd", flops):
            _cabi.check(L.mlg_decoder_bwd(_cabi.fptr(g), _cabi.fptr(xd), _cabi.fptr(h), _cabi.fptr(pd), _cabi.lptr(table), B, S,
                                          F, d_max, total_out, total_hidden, _cabi.fptr(gx, allow_none=True), _cabi.fptr(gp),
                                          _cabi.stream_ptr()), "mlg_decoder_bwd")
        return gx, gp, None, None, None, None
