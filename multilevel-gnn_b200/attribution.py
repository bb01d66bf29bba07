"""Gene and pathway attribution for MultilevelGNN on the B200 kernels.

``Attributor`` answers "which genes and pathways drove this patient's prediction" with the gradient of the predicted class
probability with respect to the patient's omics values (``batch.x``): saliency, input x gradient, or integrated gradients
(IG).  IG for one patient evaluates ``points`` interpolants of that patient, all on the same gene network: one
replicated-topology batch.  ``capture`` records the forward and the input-only backward (no weight-gradient kernel runs) as
ONE CUDA graph with its own memory pool; ``attribute`` replays it over a plan of patient slots and accumulates per-patient
results on the device (mlg_attr_accumulate: slot order fixed, so a patient's result has the same bits in any slot and any
batch), with one host synchronisation per call.

    attr = Attributor(model, args, batch_size=32, method="integrated_gradients", points=32, target=1, baseline=None)
    attr.capture(device_batch)                 # keyed batch, as Evaluator.capture
    res = attr.attribute(dataset, topo)        # records with x / y / age, as Evaluator.evaluate
    res.nodes [n, N]; res.genes [n, 5135, 3]; res.pathways [n, 146, 3]; res.pred [n, 2]; res.delta [n]
"""
import contextlib
from collections import namedtuple

import torch

from . import _cabi
from .train import StaticBatchFeed

METHODS = ("saliency", "input_x_gradient", "integrated_gradients")

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

    Eval semantics (no dropout) on the fused training-forward route.  The parameters are read in place and receive no
    gradient: they are frozen while the graph is captured (requires_grad, the model's mode and the grad mode are restored
    afterwards), so the graph holds no weight-gradient kernel and writes no ``.grad``; if their storage moved since capture
    (e.g. a Trainer re-homed them), ``attribute`` re-captures first."""

    def __init__(self, model, args, batch_size=32, method="integrated_gradients", points=32, target=1, baseline=None):
        if method not in METHODS:
            raise ValueError("Attributor: method must be one of %s (got %r)" % (METHODS, method))
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
        with self._frozen():
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

    @contextlib.contextmanager
    def _frozen(self):
        """Eval mode, grad mode on, every parameter frozen (no weight-gradient work, no .grad); all restored on exit."""
        params = list(self.model.parameters())
        flags = [p.requires_grad for p in params]
        was_training, was_grad = self.model.training, torch.is_grad_enabled()
        try:
            for p in params:
                p.requires_grad_(False)
            self.model.train(False)
            torch.set_grad_enabled(True)
            yield
        finally:
            for p, f in zip(params, flags):
                p.requires_grad_(f)
            self.model.train(was_training)
            torch.set_grad_enabled(was_grad)

    def eager(self):
        """One uncaptured pass of what a replay runs, on the static buffers (same kernels, launched from the host); the
        outputs land in ``out_g`` / ``out_pw`` / ``out_pred`` as after a replay."""
        with self._frozen():
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

    def attribute(self, dataset, topo):
        """Attributions of every record of ``dataset`` (records with x / y / age, as data.collate takes them; ``topo`` the
        dataset's FoldTopology) -> AttributionResult of host tensors, in dataset order."""
        from .data import collate
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

        def host(s):
            return collate([dataset[int(p)] for p in plan[s][:, 0]], topo)

        nxt = host(0)
        self.prefetch(nxt)
        for s in range(len(plan)):
            nxt_s = host(s + 1) if s + 1 < len(plan) else None      # collated on the host while the device works
            self._take_staged()
            first, cnt, fresh = meta[s]
            self.alpha.copy_(tab[s, 0])
            self.graph.replay()
            L = slice(first, first + cnt)
            self._accumulate(self.out_g, N, tab[s, 1], ptrs[s], cnt, N, fresh, acc[L])
            self._accumulate(self.out_pw, S3, tab[s, 2], ptrs[s], cnt, S3, fresh, pw[L])
            self._accumulate(self.out_pred, 2, tab[s, 2], ptrs[s], cnt, 2, fresh, pred[L])
            self._accumulate(self.out_pred[:, self.target:], 2, tab[s, 3], ptrs[s], cnt, 1, fresh, f0[L])
            self._accumulate(self.static_batch.x.view(B, N), N, tab[s, 2], ptrs[s], cnt, N, fresh, xs[L])
            if nxt_s is not None:
                self.prefetch(nxt_s)
        if self.method == "saliency":
            nodes = acc
        elif self.method == "input_x_gradient":
            nodes = xs * acc
        else:
            nodes = (xs - self._base) * acc
        host_nodes, host_pw, host_pred, host_f0 = (t.cpu() for t in (nodes, pw, pred, f0))     # the one synchronisation
        reorder = self.model.reorder_idxs if (self.args.reorder_pathway and self.model.reorder_idxs is not None) else None
        pathways = host_pw.view(n, S3 // 3, 3)
        if reorder is not None:
            out = torch.empty_like(pathways)
            out[:, reorder] = pathways
            pathways = out
        delta = None
        if self.method == "integrated_gradients":
            delta = (host_pred[:, self.target].double() - host_f0[:, 0].double() - host_nodes.double().sum(1)).float()
        return AttributionResult(host_nodes, gene_view(host_nodes), pathways, host_pred, delta)


def ctypes_ptr(t):
    """Device pointer of a (possibly strided) float32 CUDA view; the kernel indexes it with its own leading dimension."""
    import ctypes
    if not t.is_cuda or t.dtype != torch.float32:
        raise ValueError("expected a float32 CUDA tensor")
    return ctypes.c_void_p(t.data_ptr())
