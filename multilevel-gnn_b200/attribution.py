"""Gene and pathway attribution for MultilevelGNN on the B200 kernels.

``Attributor`` answers "which genes and pathways drove this patient's prediction" with the gradient of the predicted class
probability with respect to the patient's omics values (``batch.x``): saliency, input x gradient, integrated gradients
(IG), or expected gradients (IG averaged over a background cohort: SHAP-style values).  IG for one patient evaluates
``points`` interpolants of that patient, all on the same gene network: one replicated-topology batch.  ``capture`` records the forward and the input-only backward (no weight-gradient kernel runs) as
ONE CUDA graph with its own memory pool; ``attribute`` replays it over a plan of patient slots and accumulates per-patient
results on the device (mlg_attr_accumulate: slot order fixed, so a patient's result has the same bits in any slot and any
batch), with one host synchronisation per call.

    attr = Attributor(model, args, batch_size=32, method="integrated_gradients", points=32, target=1, baseline=None)
    attr.capture(device_batch)                 # keyed batch, as Evaluator.capture
    res = attr.attribute(dataset, topo)        # records with x / y / age, as Evaluator.evaluate
    res.nodes [n, N]; res.genes [n, 5135, 3]; res.pathways [n, 146, 3]; res.pred [n, 2]; res.delta [n]

    attr = Attributor(model, args, batch_size=32, method="expected_gradients", background=train_x, samples=32, seed=0)
"""
from collections import namedtuple

import torch

from . import _cabi
from .train import StaticBatchFeed, frozen_parameters

METHODS = ("saliency", "input_x_gradient", "integrated_gradients", "expected_gradients")

AttributionResult = namedtuple("AttributionResult", "nodes genes pathways pred delta")


def ig_alphas(points):
    """Interpolation coefficients alpha_k = k / (points - 1), k = 0 .. points - 1 (float64)."""
    if points < 2:
        raise ValueError("integrated gradients needs points >= 2 (got %d)" % points)
    return torch.arange(points, dtype=torch.float64) / (points - 1)


def trapezoid_weights(points):
    """Trapezoid-rule weights over the ``points`` interpolants of [0, 1]: 1 / (points - 1), halved at both ends."""
    w = torch.full((points,), 1.0 / (points - 1), dtype=torch.float64)
    w[0] *= 0.5
    w[-1] *= 0.5
    return w


def slot_plan(n, batch_size, per_patient):
    """Replays that visit ``per_patient`` slots (interpolants) of each of ``n`` patients, ``batch_size`` slots per replay.
    per_patient <= batch_size: floor(batch_size / per_patient) whole patients per replay; otherwise a patient's interpolants
    span ceil(per_patient / batch_size) replays.  A tail replay fills the first slots.  Returns a list of int64 tensors
    [slots, 2] of (patient, interpolant k), patients ascending and k ascending within a patient."""
    if n < 1 or batch_size < 1 or per_patient < 1:
        raise ValueError("slot_plan: n, batch_size and per_patient must be positive")
    plan = []
    if per_patient <= batch_size:
        per_replay = batch_size // per_patient
        for p0 in range(0, n, per_replay):
            pats = torch.arange(p0, min(n, p0 + per_replay))
            plan.append(torch.stack([pats.repeat_interleave(per_patient), torch.arange(per_patient).repeat(pats.numel())], 1))
    else:
        for p in range(n):
            for k0 in range(0, per_patient, batch_size):
                ks = torch.arange(k0, min(per_patient, k0 + batch_size))
                plan.append(torch.stack([torch.full_like(ks, p), ks], 1))
    return plan


_M64 = (1 << 64) - 1
_GOLDEN = 0x9E3779B97F4A7C15


def _mix64(z):
    """splitmix64's output function (Steele, Lea and Flood, OOPSLA 2014) of a 64-bit state."""
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def eg_draws(seed, index, S, M):
    """Expected gradients' draws for the patient at position ``index`` of the dataset: (j [S] int64 in [0, M), alpha [S]
    float64 in (0, 1)).  A pure function of (seed, index, S, M), so a patient's draws do not depend on batch_size, on the
    other patients or on call order.  Draw k is the k-th output of a splitmix64 stream keyed by (seed, index): counter
    based, computed directly.  j = (high 32 bits * M) >> 32; alpha = (u + 0.5) * 2^-23 with u the low 23 bits: the midpoints
    of 2^23 equal bins, each exact in fp32."""
    if S < 1 or M < 1 or index < 0:
        raise ValueError("eg_draws: needs S >= 1, M >= 1 and index >= 0")
    key = _mix64(((_mix64((seed + _GOLDEN) & _M64) ^ index) + _GOLDEN) & _M64)
    j, alpha = [], []
    for k in range(S):
        h = _mix64((key + (k + 1) * _GOLDEN) & _M64)
        j.append(((h >> 32) * M) >> 32)
        alpha.append(((h & 0x7FFFFF) + 0.5) * 2.0 ** -23)
    return torch.tensor(j, dtype=torch.int64), torch.tensor(alpha, dtype=torch.float64)


def eg_plan(j, alpha, batch_size, completeness):
    """Sample pass of expected gradients for n patients with draws j, alpha [n, S]: slot_plan over S slots per patient (2S
    with ``completeness``).  Slot k < S holds draw k with weight 1 / S; slot S + k holds draw k at alpha = 0 with weight 0,
    and its prediction F(x'_{j_k}) (at the patient's age) is kept at position patient * S + k (-1: not kept).  Returns per
    replay (slots [s, 2] of (patient, k), j [s], alpha [s], w [s], f0 position [s])."""
    n, S = j.shape
    out = []
    for slots in slot_plan(n, batch_size, 2 * S if completeness else S):
        p, k = slots[:, 0], slots[:, 1]
        draw = k % S
        sample = k < S
        out.append((slots, j[p, draw], torch.where(sample, alpha[p, draw], torch.zeros((), dtype=alpha.dtype)),
                    sample.double() / S, torch.where(sample, torch.full_like(k, -1), p * S + draw)))
    return out


def gene_view(nodes):
    """[n, N] per-node values -> [n, N // 3, 3] per (gene, omic): gene g owns nodes 3g, 3g + 1, 3g + 2."""
    return nodes.reshape(nodes.shape[0], -1, 3)


def pathway_reduce(contrib, pca_dim, reorder_idxs=None):
    """Per-element contributions at the pooled features [B, C, 146, 3 * pca_dim] -> [B, 146, 3] per (pathway, omic): summed over
    the channels and over the pca_dim columns of each omic (the last axis is (omic, p), models/multilevel_gnn.py:233).  With
    ``reorder_idxs`` (the model reordered the pathways, x[:, :, reorder_idxs]) the result is put back in the reference's
    pathway order: row r is pathway r."""
    B, C, S = contrib.shape[0], contrib.shape[1], contrib.shape[2]
    red = contrib.reshape(B, C, S, 3, pca_dim).sum((1, 4))
    if reorder_idxs is None:
        return red
    out = torch.empty_like(red)
    out[:, reorder_idxs.to(red.device)] = red
    return out


class Attributor(StaticBatchFeed):
    """Captured attribution of ``pred[:, target]`` (the softmax probability) with respect to the node values.

    method: "saliency" (dp/dx), "input_x_gradient" (x * dp/dx) or "integrated_gradients" (trapezoid rule on ``points``
    interpolants alpha * x + (1 - alpha) * x', alpha_k = k / (points - 1); ``delta`` = F(x) - F(x') - sum of the attributions,
    the completeness gap).  baseline: x' (None = zeros, or an [N] reference profile such as a cohort mean); age is held at
    the patient's value and not attributed.  Pathway attributions are gradient x activation at the pooled features at
    alpha = 1, per (pathway, omic) in the reference's pathway order.

    "expected_gradients" measures the patient against a cohort instead of one reference profile:
        phi_i(x) = E_{x' ~ background, alpha ~ U(0,1)} [(x_i - x'_i) dF/dx_i (x' + alpha (x - x'))],
        sum_i phi_i(x) = F(x) - E_{x'} F(x')   (in expectation),
    estimated from ``samples`` = S draws (j_k, alpha_k) per patient (``eg_draws``: a function of ``seed`` and the patient's
    position in the dataset only, so a patient's result has the same bits in any batch or slot).  background: [M, N]
    reference profiles, e.g. the training split's x.  A sample pass replays S interpolants per patient (x' = background[j_k])
    and sums (x - x'_{j_k}) * g_k / S on the device (mlg_attr_eg_accumulate); a pass at alpha = 1 supplies ``pred`` and the
    pathway attributions.  The pathway attributions are the same gradient x activation at alpha = 1 as for the other methods,
    not a cohort-relative SHAP value of the pathway.  With ``completeness`` each patient also gets S slots at alpha = 0
    (F(x'_{j_k}) at the patient's own age), and ``delta`` = F(x) - mean_k F(x'_{j_k}) - sum_i phi_i, the sampled
    completeness gap: zero in expectation over alpha given the drawn j.  Without it, ``delta`` is None.

    Eval semantics (no dropout) on the fused training-forward route.  The parameters are read in place and receive no
    gradient: they are frozen while the graph is captured (requires_grad, the model's mode and the grad mode are restored
    afterwards), so the graph holds no weight-gradient kernel and writes no ``.grad``; if their storage moved since capture
    (e.g. a Trainer re-homed them), ``attribute`` re-captures first."""

    def __init__(self, model, args, batch_size=32, method="integrated_gradients", points=32, target=1, baseline=None,
                 background=None, samples=32, seed=0, completeness=False):
        if method not in METHODS:
            raise ValueError("Attributor: method must be one of %s (got %r)" % (METHODS, method))
        self.background = None
        if method == "expected_gradients":
            if background is None:
                raise ValueError("Attributor: expected_gradients needs a background [M, N] of reference profiles")
            if baseline is not None:
                raise ValueError("Attributor: expected_gradients takes a background, not a baseline")
            bg = torch.as_tensor(background).detach().to("cpu", torch.float32, copy=True)
            n_nodes = 3 * model.node_num
            if bg.dim() != 2 or bg.shape[0] < 1 or bg.shape[1] != n_nodes:
                raise ValueError("Attributor: background must be [M >= 1, %d] (got %s)" % (n_nodes, tuple(bg.shape)))
            if not bool(torch.isfinite(bg).all()):
                raise ValueError("Attributor: background values must be finite")
            if int(samples) < 1:
                raise ValueError("Attributor: samples must be >= 1 (got %d)" % int(samples))
            self.background = bg.contiguous()
        elif background is not None:
            raise ValueError("Attributor: background is only used by expected_gradients (method %r)" % method)
        self.samples, self.seed, self.completeness = int(samples), int(seed), bool(completeness)
        self.model, self.args = model, args
        self.batch_size = int(batch_size)
        if not 1 <= self.batch_size <= 64:
            raise ValueError("Attributor: batch_size must be in [1, 64] (the fused head's limit)")
        self.method = method
        self.points = int(points) if method == "integrated_gradients" else 1
        if method == "integrated_gradients":
            ig_alphas(self.points)
        self.target = int(target)
        self.baseline = None if baseline is None else torch.as_tensor(baseline, dtype=torch.float32).reshape(-1)
        self.graph = None
        self.static_batch = None
        self._copy_stream = None
        self._example = None

    def _param_ptrs(self):
        return [p.data_ptr() for p in self.model.parameters()]

    # one replay: interpolate, forward, input-only backward (recorded as one graph)
    def _replay_body(self):
        B = self.batch_size
        xs = self.static_batch.x.view(B, -1)
        if self.method == "integrated_gradients":
            a = self.alpha.view(B, 1)
            xin = torch.addcmul(self._base * (1.0 - a), a, xs)      # alpha * x + (1 - alpha) * x': exact at both ends
        elif self.method == "expected_gradients":
            xin = torch.empty_like(xs)
            _cabi.check(_cabi.lib().mlg_attr_eg_interp(_cabi.fptr(xs), _cabi.fptr(self._bank), self._bank.shape[0],
                                                       _cabi.iptr(self.j), _cabi.fptr(self.alpha), B, xs.shape[1],
                                                       _cabi.fptr(xin), _cabi.iptr(self._bad), _cabi.stream_ptr()),
                        "mlg_attr_eg_interp")
        else:
            xin = xs.clone()
        xin.requires_grad_(True)
        batch = type(self.static_batch)(**vars(self.static_batch))
        batch.x = xin.view(-1, 1)
        pred, feat = self.model(batch)
        g_x, g_feat = torch.autograd.grad(pred[:, self.target].sum(), [xin, feat])
        pw = pathway_reduce(feat.detach() * g_feat, self.model.pca_dim)
        self.out_g, self.out_pw, self.out_pred = g_x, pw.reshape(B, -1), pred.detach()

    def capture(self, batch, warmup=2):
        """Record the graph over ``batch`` (a keyed device batch of ``batch_size`` graphs, as Evaluator.capture)."""
        B = int(batch.age.shape[0])
        if B != self.batch_size:
            raise ValueError("Attributor.capture: the batch holds %d graphs, batch_size is %d" % (B, self.batch_size))
        if getattr(batch, "topology_key", None) is None:
            raise ValueError("Attributor.capture: needs a keyed batch (data.collate / data.to_device)")
        from .synth import GraphBatch
        from .data import PER_SAMPLE_FIELDS
        self._example = batch
        static = GraphBatch(**{k: v for k, v in vars(batch).items()})
        for k in PER_SAMPLE_FIELDS:
            setattr(static, k, getattr(batch, k).clone())
        self.static_batch = static
        self._copy_stream = None
        dev = static.x.device
        n_nodes = static.x.numel() // B
        self.alpha = torch.ones(B, dtype=torch.float32, device=dev)
        self._base = (torch.zeros(n_nodes, dtype=torch.float32, device=dev) if self.baseline is None
                      else self.baseline.to(dev).reshape(n_nodes).clone())
        if self.method == "expected_gradients":
            if self.background.shape[1] != n_nodes:
                raise ValueError("Attributor.capture: the background has %d nodes, the batch %d"
                                 % (self.background.shape[1], n_nodes))
            self._bank = self.background.to(dev, copy=True)
            self.j = torch.zeros(B, dtype=torch.int32, device=dev)
            self._bad = torch.zeros(1, dtype=torch.int32, device=dev)
        with frozen_parameters(self.model, grad_enabled=True):
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    self._replay_body()
            cur.wait_stream(side)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._replay_body()
        self._ptrs = self._param_ptrs()
        return self

    def eager(self):
        """One uncaptured pass of what a replay runs, on the static buffers (same kernels, launched from the host); the
        outputs land in ``out_g`` / ``out_pw`` / ``out_pred`` as after a replay."""
        with frozen_parameters(self.model, grad_enabled=True):
            self._replay_body()

    def _step_fields(self, host_batch):
        from .data import PER_SAMPLE_FIELDS
        return list(PER_SAMPLE_FIELDS)

    def _check_topology(self, host_batch):
        pass

    @staticmethod
    def _fill(dst, src):
        dst[:src.shape[0]].copy_(src, non_blocking=True)

    def _device_plan(self, plan, dev):
        """Per replay: alphas [B], node weights [B], alpha = 1 / alpha = 0 indicators [B], per-patient slot pointers; one upload."""
        B, m = self.batch_size, self.points
        if self.method == "integrated_gradients":
            al, tw = ig_alphas(m).float(), trapezoid_weights(m).float()
        else:
            al, tw = torch.ones(1), torch.ones(1)
        rows = []
        for slots in plan:
            k = slots[:, 1]
            pat = slots[:, 0]
            t = torch.zeros(4, B)
            t[0, :len(k)] = al[k]
            t[1, :len(k)] = tw[k]
            t[2, :len(k)] = (k == m - 1).float()
            t[3, :len(k)] = (k == 0).float()
            ptr = torch.zeros(B + 1, dtype=torch.int32)
            first = int(pat[0])
            counts = torch.bincount(pat - first)
            ptr[1:counts.numel() + 1] = torch.cumsum(counts, 0).to(torch.int32)
            rows.append((t, ptr, first, counts.numel(), bool(k[0] == 0)))
        tab = torch.stack([r[0] for r in rows]).pin_memory().to(dev, non_blocking=True)
        ptrs = torch.stack([r[1] for r in rows]).pin_memory().to(dev, non_blocking=True)
        return tab, ptrs, [(r[2], r[3], r[4]) for r in rows]

    def _accumulate(self, g, ld, w, ptr, n_out, N, fresh, acc):
        _cabi.check(_cabi.lib().mlg_attr_accumulate(_cabi.fptr(g) if ld == N else ctypes_ptr(g), ld, _cabi.fptr(w),
                                                    _cabi.iptr(ptr), n_out, N, 0 if fresh else 1, _cabi.fptr(acc),
                                                    _cabi.stream_ptr()), "mlg_attr_accumulate")

    def _replays(self, dataset, topo, plan, before, after):
        """One replay per entry of ``plan`` on its slots' records, collated on the host and staged on a side stream while
        the device works; ``before(s)`` sets replay s's per-slot inputs, ``after(s)`` consumes its outputs."""
        from .data import collate

        def host(s):
            return collate([dataset[int(p)] for p in plan[s][:, 0]], topo)

        nxt = host(0)
        self.prefetch(nxt)
        for s in range(len(plan)):
            nxt_s = host(s + 1) if s + 1 < len(plan) else None      # collated on the host while the device works
            self._take_staged()
            before(s)
            self.graph.replay()
            after(s)
            if nxt_s is not None:
                self.prefetch(nxt_s)

    def _pathways(self, host_pw, n):
        """[n, S3] summed pooled contributions -> [n, 146, 3] in the reference's pathway order."""
        reorder = self.model.reorder_idxs if (self.args.reorder_pathway and self.model.reorder_idxs is not None) else None
        pathways = host_pw.view(n, host_pw.shape[1] // 3, 3)
        if reorder is not None:
            out = torch.empty_like(pathways)
            out[:, reorder] = pathways
            pathways = out
        return pathways

    def attribute(self, dataset, topo):
        """Attributions of every record of ``dataset`` (records with x / y / age, as data.collate takes them; ``topo`` the
        dataset's FoldTopology) -> AttributionResult of host tensors, in dataset order."""
        if self.graph is None:
            raise RuntimeError("Attributor: call capture(batch) first")
        want = "%s-b%d" % (topo.key, self.batch_size)
        if self.static_batch.topology_key != want:
            raise ValueError("Attributor: captured for topology_key=%r, this dataset's topology is %r"
                             % (self.static_batch.topology_key, want))
        if self._param_ptrs() != self._ptrs:
            self.capture(self._example)          # parameters were re-homed since capture: the graph reads stale storage
        n = len(dataset)
        if n == 0:
            raise ValueError("Attributor: empty dataset")
        if self.method == "expected_gradients":
            return self._expected_gradients(dataset, topo)
        B = self.batch_size
        plan = slot_plan(n, B, self.points)
        dev = self.out_g.device
        N = self.out_g.shape[1]
        S3 = self.out_pw.shape[1]
        tab, ptrs, meta = self._device_plan(plan, dev)
        acc = torch.empty(n, N, dtype=torch.float32, device=dev)
        pw = torch.empty(n, S3, dtype=torch.float32, device=dev)
        pred = torch.empty(n, 2, dtype=torch.float32, device=dev)
        f0 = torch.empty(n, 1, dtype=torch.float32, device=dev)
        xs = torch.empty(n, N, dtype=torch.float32, device=dev)

        def before(s):
            self.alpha.copy_(tab[s, 0])

        def after(s):
            first, cnt, fresh = meta[s]
            L = slice(first, first + cnt)
            self._accumulate(self.out_g, N, tab[s, 1], ptrs[s], cnt, N, fresh, acc[L])
            self._accumulate(self.out_pw, S3, tab[s, 2], ptrs[s], cnt, S3, fresh, pw[L])
            self._accumulate(self.out_pred, 2, tab[s, 2], ptrs[s], cnt, 2, fresh, pred[L])
            self._accumulate(self.out_pred[:, self.target:], 2, tab[s, 3], ptrs[s], cnt, 1, fresh, f0[L])
            self._accumulate(self.static_batch.x.view(B, N), N, tab[s, 2], ptrs[s], cnt, N, fresh, xs[L])

        self._replays(dataset, topo, plan, before, after)
        if self.method == "saliency":
            nodes = acc
        elif self.method == "input_x_gradient":
            nodes = xs * acc
        else:
            nodes = (xs - self._base) * acc
        host_nodes, host_pw, host_pred, host_f0 = (t.cpu() for t in (nodes, pw, pred, f0))     # the one synchronisation
        delta = None
        if self.method == "integrated_gradients":
            delta = (host_pred[:, self.target].double() - host_f0[:, 0].double() - host_nodes.double().sum(1)).float()
        return AttributionResult(host_nodes, gene_view(host_nodes), self._pathways(host_pw, n), host_pred, delta)

    def _eg_device_plan(self, rows, dev, dummy):
        """Sample pass tables per replay (eg_plan rows): alpha and weights [2, B] fp32, bank rows and slot pointers [2B + 1]
        int32, F(x'_j) destinations [B] int64 (``dummy`` for slots whose prediction is not kept); one upload each."""
        B = self.batch_size
        ft, it, dst, meta = [], [], [], []
        for slots, j, alpha, w, pos in rows:
            m = slots.shape[0]
            f = torch.zeros(2, B)
            f[0, :m], f[1, :m] = alpha.float(), w.float()
            i = torch.zeros(2 * B + 1, dtype=torch.int32)
            i[:m] = j.to(torch.int32)
            pat = slots[:, 0]
            first = int(pat[0])
            counts = torch.bincount(pat - first)
            i[B + 1:B + 1 + counts.numel()] = torch.cumsum(counts, 0).to(torch.int32)
            d = torch.full((B,), dummy, dtype=torch.int64)
            d[:m] = torch.where(pos < 0, torch.full_like(pos, dummy), pos)
            ft.append(f), it.append(i), dst.append(d)
            meta.append((first, counts.numel(), bool(slots[0, 1] == 0), bool((w > 0).any()), bool((pos >= 0).any())))
        up = [torch.stack(t).pin_memory().to(dev, non_blocking=True) for t in (ft, it, dst)]
        return up[0], up[1], up[2], meta

    def _expected_gradients(self, dataset, topo):
        n, B, S = len(dataset), self.batch_size, self.samples
        M = self._bank.shape[0]
        dev = self.out_g.device
        N = self.out_g.shape[1]
        S3 = self.out_pw.shape[1]
        draws = [eg_draws(self.seed, i, S, M) for i in range(n)]
        rows = eg_plan(torch.stack([d[0] for d in draws]), torch.stack([d[1] for d in draws]), B, self.completeness)
        ftab, itab, dst, meta = self._eg_device_plan(rows, dev, n * S)
        plan1 = slot_plan(n, B, 1)
        tab, ptrs, meta1 = self._device_plan(plan1, dev)
        acc = torch.empty(n, N, dtype=torch.float32, device=dev)
        f0 = torch.zeros(n * S + 1, dtype=torch.float32, device=dev)       # last entry: the slots whose value is not kept
        pw = torch.empty(n, S3, dtype=torch.float32, device=dev)
        pred = torch.empty(n, 2, dtype=torch.float32, device=dev)
        self._bad.zero_()
        xs = self.static_batch.x.view(B, N)

        def before(s):
            self.alpha.copy_(ftab[s, 0])
            self.j.copy_(itab[s, :B])

        def after(s):
            first, cnt, fresh, weighted, kept = meta[s]
            if weighted or fresh:
                _cabi.check(_cabi.lib().mlg_attr_eg_accumulate(
                    _cabi.fptr(self.out_g), _cabi.fptr(xs), _cabi.fptr(self._bank), M, _cabi.iptr(self.j),
                    _cabi.fptr(ftab[s, 1]), _cabi.iptr(itab[s, B:]), cnt, N, 0 if fresh else 1,
                    _cabi.fptr(acc[first:first + cnt]), _cabi.iptr(self._bad), _cabi.stream_ptr()), "mlg_attr_eg_accumulate")
            if kept:
                f0.index_copy_(0, dst[s], self.out_pred[:, self.target])

        self._replays(dataset, topo, [r[0] for r in rows], before, after)

        def before1(s):
            self.alpha.copy_(tab[s, 0])                # alpha = 1: the interpolant is x, whatever bank row j holds

        def after1(s):
            first, cnt, fresh = meta1[s]
            L = slice(first, first + cnt)
            self._accumulate(self.out_pw, S3, tab[s, 2], ptrs[s], cnt, S3, fresh, pw[L])
            self._accumulate(self.out_pred, 2, tab[s, 2], ptrs[s], cnt, 2, fresh, pred[L])

        self._replays(dataset, topo, plan1, before1, after1)
        host_nodes, host_pw, host_pred, host_f0, bad = (t.cpu() for t in (acc, pw, pred, f0, self._bad))  # one sync
        if int(bad[0]):
            raise RuntimeError("Attributor: a background row index was outside [0, %d)" % M)
        delta = None
        if self.completeness:
            ref = host_f0[:n * S].view(n, S).double().mean(1)
            delta = (host_pred[:, self.target].double() - ref - host_nodes.double().sum(1)).float()
        return AttributionResult(host_nodes, gene_view(host_nodes), self._pathways(host_pw, n), host_pred, delta)


def ctypes_ptr(t):
    """Device pointer of a (possibly strided) float32 CUDA view; the kernel indexes it with its own leading dimension."""
    import ctypes
    if not t.is_cuda or t.dtype != torch.float32:
        raise ValueError("expected a float32 CUDA tensor")
    return ctypes.c_void_p(t.data_ptr())
