"""The caller of the hot path: one training step as the reference's ``train()`` runs it
(train.py:38-68; optimizer / criterion set-up train.py:112-125), plus the data-parallel wrapper the
reference lacks (SURVEY.md section 8e): patient graphs are independent, so every rank steps on its own
batch and the replicas are synchronised by ONE fused kernel after backward over NVLink peer memory
(gradient reduce-scatter -> Adam on the owned shard -> parameter all-gather, csrc/peer_adam.cu) -- or,
selectably, one NCCL all-reduce (op=AVG)
over the flat fp32 gradient bucket followed by a replicated flat Adam.  Parameters that never receive a
gradient (``lin_l.weight`` of every SAGEConv, ``info_mask``) are left out of the bucket and of the
optimizer state.
"""
import contextlib
from typing import NamedTuple, Optional

import torch
import torch.distributed as dist


def shard_indices(n_items, rank, world, per_rank_batch, epoch_seed=0, drop_last=True):
    """Per-epoch partition of the patient list: one shuffled permutation (same seed on every rank), rank r takes
    batches r, r+world, ... of size ``per_rank_batch`` -- disjoint across ranks (train.py:303-323 uses a single
    DataLoader with shuffle + drop_last; this is its data-parallel split).  Returns a list of index tensors."""
    g = torch.Generator()
    g.manual_seed(epoch_seed)
    perm = torch.randperm(n_items, generator=g)
    step = per_rank_batch * world
    n_steps = n_items // step if drop_last else -(-n_items // step)
    out = []
    for s in range(n_steps):
        lo = s * step + rank * per_rank_batch
        out.append(perm[lo:lo + per_rank_batch])
    return out


class GradBucket:
    """Flat fp32 gradient bucket: every ``p.grad`` is a view into one contiguous buffer, so the data-parallel
    synchronisation is ONE all-reduce with no packing/unpacking (NCCL: op=AVG folds the 1/world scale in;
    gloo has no AVG, so SUM + scale).  Parameters that never get a gradient are not in the bucket.
    ``align``: the bucket length is rounded up to a multiple of it (the fused peer update needs a multiple of 4 * world);
    the padding elements stay zero."""

    def __init__(self, params, flat=None, align=1):
        self.params = list(params)
        dev = self.params[0].device
        self.offsets, off = {}, 0
        for p in self.params:
            self.offsets[id(p)] = off
            off += p.numel()
        n = GradBucket.padded_size(self.params, align)
        self.n = n
        # ``flat``: caller-provided storage (PeerArena: peer-mapped device memory, padded past n)
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev) if flat is None else flat
        assert self.flat.numel() >= n and self.flat.is_contiguous()
        for p in self.params:
            o = self.offsets[id(p)]
            p.grad = self.flat[o:o + p.numel()].view_as(p)
            # backward kernels that produce a whole parameter gradient may write it here directly (functional.grad_slot)
            p._mlg_grad_slot = {"view": p.grad, "claimed": False}

    @staticmethod
    def padded_size(params, align):
        return -(-sum(p.numel() for p in params) // align) * align

    def zero(self):
        self.flat.zero_()

    def store(self, grads):
        """Write a list of gradients (one per bucket parameter, None = no gradient) into the bucket with one
        multi-tensor copy.  Replaces zero() + AccumulateGrad's per-parameter in-place add (one tiny kernel per
        parameter: ~20 launches per step on the gbm model)."""
        if any(g is None for g in grads):
            if not hasattr(self, "_has_none"):
                self._has_none = True
            for p, g in zip(self.params, grads):
                if g is None:
                    p.grad.zero_()
        dst, src = [], []
        for p, g in zip(self.params, grads):
            p._mlg_grad_slot["claimed"] = False
            if g is not None and g.data_ptr() != p.grad.data_ptr():    # same pointer: written in place by its kernel
                dst.append(p.grad)
                src.append(g)
        if dst:
            torch._foreach_copy_(dst, src)

    def all_reduce(self, world):
        if world <= 1:
            return
        if dist.get_backend() == "nccl":
            dist.all_reduce(self.flat, op=dist.ReduceOp.AVG)
        else:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.flat.mul_(1.0 / world)


class FlatAdam:
    """torch.optim.Adam (amsgrad off) as ONE kernel over flat buffers (mlg_adam_step): parameters are re-homed as views
    of one contiguous fp32 buffer laid out like the gradient bucket; the step counter is a device scalar so the
    update replays inside a CUDA graph.  lr / betas / eps / weight_decay as in train.py:112."""

    def __init__(self, bucket, lr, betas, eps=1e-8, weight_decay=0.0):
        self.bucket, self.lr, self.betas, self.eps, self.wd = bucket, lr, betas, eps, weight_decay
        flat_g = bucket.flat
        self.flat_p = torch.zeros_like(flat_g)
        for p in bucket.params:
            n, off = p.numel(), bucket.offsets[id(p)]
            self.flat_p[off:off + n].copy_(p.data.reshape(-1))
            p.data = self.flat_p[off:off + n].view_as(p)
        self.exp_avg = torch.zeros_like(flat_g)
        self.exp_avg_sq = torch.zeros_like(flat_g)
        self.step_dev = torch.zeros(1, dtype=torch.float32, device=flat_g.device)

    def step(self):
        from . import _cabi
        L = _cabi.lib()
        with torch.cuda.device(self.flat_p.device):
            _cabi.check(L.mlg_adam_step(_cabi.fptr(self.flat_p), _cabi.fptr(self.bucket.flat), _cabi.fptr(self.exp_avg),
                                        _cabi.fptr(self.exp_avg_sq), _cabi.fptr(self.step_dev), self.flat_p.numel(),
                                        float(self.lr), float(self.betas[0]), float(self.betas[1]), float(self.eps),
                                        float(self.wd), _cabi.stream_ptr()), "mlg_adam_step")


class _DeviceSpan:
    """A raw device allocation exposed through __cuda_array_interface__ so that torch can alias it (no copy)."""

    def __init__(self, ptr, n_floats):
        self.__cuda_array_interface__ = {"shape": (n_floats,), "typestr": "<f4", "data": (ptr, False), "version": 3,
                                         "strides": None}


class PeerArena:
    """This rank's peer-visible device memory [gradient bucket | parameters | flag block] (mlg_peer_alloc) and the mappings
    of every other rank's arena (CUDA IPC handles exchanged once through torch.distributed)."""

    def __init__(self, n_padded, world, rank, device, exchange=True):
        from . import _cabi
        L = _cabi.lib()
        self.world, self.rank, self.device = world, rank, device
        assert n_padded % 4 == 0
        self.n_padded = n_padded
        self.bytes = 2 * 4 * self.n_padded + int(L.mlg_peer_flag_bytes())
        with torch.cuda.device(device):
            self.base = L.mlg_peer_alloc(self.bytes)
        if not self.base:
            raise RuntimeError("mlg_peer_alloc failed: %s" % _cabi.last_error())
        self._opened = []
        self._hold = (_DeviceSpan(self.base, self.n_padded), _DeviceSpan(self.base + 4 * self.n_padded, self.n_padded))
        self.grad = torch.as_tensor(self._hold[0], device=device)
        self.param = torch.as_tensor(self._hold[1], device=device)
        self.peer_base = [None] * world
        self.peer_base[rank] = self.base
        if exchange and world > 1:
            self._exchange()

    def _exchange(self):
        import ctypes
        from . import _cabi
        L = _cabi.lib()
        handle = ctypes.create_string_buffer(64)
        _cabi.check(L.mlg_peer_export(self.base, handle), "mlg_peer_export")
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle.raw))
        with torch.cuda.device(self.device):
            for r, h in enumerate(handles):
                if r == self.rank:
                    continue
                buf = ctypes.create_string_buffer(h, 64)
                ptr = L.mlg_peer_open(buf)
                if not ptr:
                    raise RuntimeError("mlg_peer_open(rank %d) failed: %s" % (r, _cabi.last_error()))
                self._opened.append(ptr)
                self.peer_base[r] = ptr

    def pointer_tables(self):
        """(grads, params, flags): ctypes arrays of ``world`` device pointers, indexed by rank."""
        import ctypes
        arr = ctypes.c_void_p * self.world
        g = arr(*[b for b in self.peer_base])
        p = arr(*[b + 4 * self.n_padded for b in self.peer_base])
        f = arr(*[b + 8 * self.n_padded for b in self.peer_base])
        return g, p, f

    def status(self):
        """Non-zero when a wait of the update kernel gave up on this rank (device read: synchronises)."""
        import ctypes
        from . import _cabi
        out = ctypes.c_int(0)
        _cabi.check(_cabi.lib().mlg_peer_status(self.base + 8 * self.n_padded, ctypes.byref(out)), "mlg_peer_status")
        return out.value

    def close(self):
        from . import _cabi
        L = _cabi.lib()
        for ptr in self._opened:
            L.mlg_peer_close(ptr)
        self._opened = []
        # the arena itself stays allocated for the life of the process: parameters and gradients alias it


class PeerAdam:
    """Data-parallel optimizer step as ONE kernel over NVLink peer memory (mlg_peer_adam_step): reduce-scatter of the
    gradient buckets, torch.optim.Adam on the owned 1/world shard (ZeRO-1: the moment buffers exist once per box),
    all-gather of the updated parameters -- no NCCL call, no second graph, every rank bitwise in step.  Parameters are
    re-homed as views of the arena's parameter buffer (like FlatAdam).  A wait that times out is a hard failure on every
    rank (``failed()``)."""

    def __init__(self, bucket, arena, lr, betas, eps=1e-8, weight_decay=0.0, timeout_s=5.0):
        self.bucket, self.arena = bucket, arena
        self.lr, self.betas, self.eps, self.wd, self.timeout_s = lr, betas, eps, weight_decay, timeout_s
        self.flat_p = arena.param
        for p in bucket.params:
            n, off = p.numel(), bucket.offsets[id(p)]
            self.flat_p[off:off + n].copy_(p.data.reshape(-1))
            p.data = self.flat_p[off:off + n].view_as(p)
        dev = arena.device
        self.exp_avg = torch.zeros(bucket.n // arena.world, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros_like(self.exp_avg)
        self.step_dev = torch.zeros(1, dtype=torch.float32, device=dev)
        self._tables = arena.pointer_tables()
        # pinned host word the kernel sets on a failed wait: read by the host without synchronising the device
        self.host_status = torch.zeros(1, dtype=torch.int32).pin_memory()

    def failed(self):
        return int(self.host_status[0]) != 0

    def step(self):
        import ctypes
        from . import _cabi
        a = self.arena
        g, p, f = self._tables
        with torch.cuda.device(a.device):
            _cabi.check(_cabi.lib().mlg_peer_adam_step(
                g, p, f, a.world, a.rank, self.bucket.n, _cabi.fptr(self.exp_avg), _cabi.fptr(self.exp_avg_sq),
                _cabi.fptr(self.step_dev), float(self.lr), float(self.betas[0]), float(self.betas[1]), float(self.eps),
                float(self.wd), float(self.timeout_s), ctypes.c_void_p(self.host_status.data_ptr()), _cabi.stream_ptr()),
                "mlg_peer_adam_step")


def peer_update_available(world, device):
    """True when every rank of the job sits on one box with CUDA peer access to every other rank's GPU (NVLink /
    NVSwitch) -- the precondition of PeerAdam.  Collective: every rank must call it."""
    if world <= 1 or device.type != "cuda" or not dist.is_initialized() or dist.get_backend() != "nccl" or world > 8:
        return False
    ids = [None] * world
    dist.all_gather_object(ids, (torch.cuda.current_device(), __import__("socket").gethostname()))
    mine = torch.cuda.current_device()
    ok = len({h for _, h in ids}) == 1 and len({d for d, _ in ids}) == world
    ok = ok and all(d == mine or torch.cuda.can_device_access_peer(mine, d) for d, _ in ids)
    flag = torch.tensor([1 if ok else 0], device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item())


class _PendingLoss:
    """A loss value on its way to pinned host memory (Trainer.loss_to_host); slot[1] != 0: a keyless batch uploaded after
    capture() did not match the captured topology."""

    def __init__(self, slot, event):
        self.slot, self.event = slot, event

    def get(self):
        self.event.synchronize()
        if float(self.slot[1]) != 0.0:
            raise RuntimeError("Trainer: a batch uploaded after capture() carried a different topology than the captured graph")
        return float(self.slot[0])


@contextlib.contextmanager
def frozen_parameters(model, grad_enabled):
    """Eval mode, every parameter frozen (no weight-gradient work, no .grad) and the grad mode set to ``grad_enabled``; all
    restored on exit.  The attribution and knockout graphs are recorded under it: they read the parameters in place."""
    params = list(model.parameters())
    flags = [p.requires_grad for p in params]
    was_training, was_grad = model.training, torch.is_grad_enabled()
    try:
        for p in params:
            p.requires_grad_(False)
        model.train(False)
        torch.set_grad_enabled(grad_enabled)
        yield
    finally:
        for p, f in zip(params, flags):
            p.requires_grad_(f)
        model.train(was_training)
        torch.set_grad_enabled(was_grad)


class StaticBatchFeed:
    """Host -> device feeding of a captured CUDA graph's static input buffers (``self.static_batch``), shared by ``Trainer``
    and ``Evaluator``: ``load_batch`` copies a (pinned) host batch in on the current stream; ``prefetch`` starts the copy of
    the NEXT batch on a side stream into staging buffers while the current replay runs, and ``_take_staged`` moves it into
    the static buffers (device-to-device) right before the next replay."""

    # fields that are dataset constants when a batch carries a ``topology_key``: the key promises that the edge list,
    # edge weights, node->graph vector and pooling layout are identical for every batch with that key (one gene network
    # shared by all patients, dataloader/multiloader.py:687-698) -- exactly what MultilevelGNN.forward already assumes
    # when it caches the CSR / pool layout under that key.  They are uploaded once, not per step.
    STATIC_TOPOLOGY_FIELDS = ("edge_index", "edge_attr", "batch", "gene_pca_match", "raw_indice")

    def _step_fields(self, host_batch):
        key = getattr(self.static_batch, "topology_key", None)
        same = key is not None and getattr(host_batch, "topology_key", None) == key
        return [k for k, v in vars(self.static_batch).items()
                if torch.is_tensor(v) and not (same and k in self.STATIC_TOPOLOGY_FIELDS)]

    def h2d_bytes(self, host_batch):
        """Bytes ``load_batch`` / ``prefetch`` copy host -> device for this batch."""
        return sum(getattr(host_batch, k).numel() * getattr(host_batch, k).element_size()
                   for k in self._step_fields(host_batch))

    def _check_topology(self, host_batch):
        """The CSR, pooling layout, degree tables and visiting orders are built in the warm-up steps and BAKED into the
        captured graph: a batch with another edge list / match table would silently train on the stale topology.  A keyed
        batch (data.collate / data.TopologyLoader) must carry the key the graph was captured with.  A batch WITHOUT a key
        (the reference's loader: every batch re-sends its own copy of the topology, train.py:42) is accepted, uploaded in
        full, and its topology fields are compared ON THE DEVICE with the captured ones; a mismatch raises when the host
        next reads a loss (``loss_to_host(...).get()``) or calls ``check_topology_flag()``."""
        key = getattr(self.static_batch, "topology_key", None)
        other = getattr(host_batch, "topology_key", None)
        if other is not None and other != key:
            raise ValueError("Trainer: the topology is frozen at capture(); this batch has topology_key=%r, the captured "
                             "graph %r -- re-capture for a new topology, or step eagerly" % (other, key))

    def _verify_uploaded_topology(self, fields):
        """After a full upload into the static buffers: flag |= any(static != captured) per topology field (device only)."""
        ref = getattr(self, "_topo_ref", None)
        if ref is None:
            return
        for k in fields:
            if k in ref:
                self._topo_bad.logical_or_((getattr(self.static_batch, k) != ref[k]).any())
                self._topo_compared = True      # from now on the flag travels to the host with every loss

    def check_topology_flag(self):
        """Host-side check (one sync) that no keyless batch with a different topology was fed to the captured graph."""
        if getattr(self, "_topo_bad", None) is not None and bool(self._topo_bad.item()):
            raise RuntimeError("Trainer: a batch uploaded after capture() carried a different edge list / pooling layout than "
                               "the captured graph was built for (topology is frozen at capture())")

    def load_batch(self, host_batch):
        """Copy a (pinned) host batch into the captured graph's static device buffers (async H2D).  Only per-step
        fields are copied: the topology fields are frozen at capture()."""
        self._check_topology(host_batch)
        fields = self._step_fields(host_batch)
        for k in fields:
            self._fill(getattr(self.static_batch, k), getattr(host_batch, k))
        self._verify_uploaded_topology(fields)

    def prefetch(self, host_batch):
        """Start the H2D copy of the NEXT batch on a side stream into staging buffers while the current step's
        graph is still running; ``step_prefetched`` then moves it into the static buffers (device-to-device)
        and replays.  This is the double buffering the reference's synchronous ``batch.to(device)``
        (train.py:42) lacks."""
        self._check_topology(host_batch)
        if self._copy_stream is None or set(self._staging) != set(self._step_fields(host_batch)):
            if self._copy_stream is not None:
                torch.cuda.current_stream().synchronize()        # switching keyed <-> keyless batches: new staging set
            self._copy_stream = torch.cuda.Stream()
            self._staging = {k: torch.empty_like(getattr(self.static_batch, k)) for k in self._step_fields(host_batch)}
            self._staged = torch.cuda.Event()
            self._consumed = torch.cuda.Event()
            self._consumed.record()
        self._copy_stream.wait_event(self._consumed)        # staging may not be overwritten before it was consumed
        with torch.cuda.stream(self._copy_stream):
            if set(self._staging) != set(self._step_fields(host_batch)):
                raise ValueError("prefetch: this batch's topology_key differs from the one the staging buffers were "
                                 "sized for; use step(batch) for a batch with a different topology")
            for k, v in self._staging.items():
                self._fill(v, getattr(host_batch, k))
            self._staged.record()

    @staticmethod
    def _fill(dst, src):
        """The H2D copy of one field into its device buffer (static or staging)."""
        dst.copy_(src, non_blocking=True)

    def _take_staged(self):
        """Move the batch ``prefetch`` staged into the static buffers (device-to-device, on the current stream)."""
        cur = torch.cuda.current_stream()
        cur.wait_event(self._staged)
        # staging -> static buffers: one multi-tensor launch per dtype instead of one copy kernel per field
        torch._foreach_copy_([getattr(self.static_batch, k) for k in self._staging], list(self._staging.values()))
        self._consumed.record()
        self._verify_uploaded_topology(self._staging)


class Trainer(StaticBatchFeed):
    """One training step of train.py:38-68 on the B200 kernels; ``capture()`` turns the whole step (forward, loss,
    backward, optimizer update -- with several ranks the fused NVLink reduce-scatter / Adam / all-gather kernels) into ONE
    CUDA graph replayed per step (the NCCL path keeps its all-reduce between two graphs)."""

    def __init__(self, model, args, criterion_weight=None, world_size=1, fused_adam=True, peer_update=None):
        """peer_update: None = use the fused NVLink peer-memory update (PeerAdam) whenever the job allows it (one box,
        NCCL process group, peer access between all ranks, no gradient clipping -- clipping needs the averaged gradient
        on every rank before the update); False = NCCL all-reduce + replicated FlatAdam; True = require PeerAdam."""
        self.model, self.args, self.world = model, args, world_size
        # reference flags this trainer does not implement must not be silently ignored (train.py:52-57 per-sample
        # criterion weights with reduction='none'; train.py:113-116 StepLR)
        for flag in ("weighted_loss", "batch_weighted_loss"):
            if getattr(args, flag, False):
                raise NotImplementedError("Trainer: args.%s (per-sample BCE weights, train.py:52-57) is not implemented" % flag)
        if getattr(args, "step", 0) and getattr(args, "step", 0) > 0:
            raise NotImplementedError("Trainer: args.step > 0 (StepLR, train.py:113-116) is not implemented: lr is a launch "
                                      "constant of the captured update kernel")
        self.params = [p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")]
        dev = self.params[0].device
        self.peer = None
        want_peer = (peer_update is not False and fused_adam and world_size > 1 and dev.type == "cuda"
                     and not args.clip_grad)
        if want_peer and not peer_update_available(world_size, dev):
            if peer_update:
                raise RuntimeError("peer_update=True but the ranks do not all have CUDA peer access on one box")
            want_peer = False
        if want_peer:
            align = 4 * world_size
            self.peer = PeerArena(GradBucket.padded_size(self.params, align), world_size, dist.get_rank(), dev)
            self.bucket = GradBucket(self.params, flat=self.peer.grad, align=align)
        else:
            self.bucket = GradBucket(self.params)
        self.flat = self.bucket.flat
        if self.peer is not None:
            self.opt = PeerAdam(self.bucket, self.peer, lr=args.lr, betas=(args.beta1, args.beta2), weight_decay=args.wd)
        elif fused_adam and dev.type == "cuda":
            self.opt = FlatAdam(self.bucket, lr=args.lr, betas=(args.beta1, args.beta2), weight_decay=args.wd)
        else:
            self.opt = torch.optim.Adam(self.params, lr=args.lr, betas=(args.beta1, args.beta2), weight_decay=args.wd)
        self.weight = criterion_weight
        self.crit = torch.nn.BCELoss(weight=criterion_weight) if args.weight_balance else torch.nn.BCELoss()
        self.graph = None
        self.graph_update = None
        self.static_batch = None
        self.static_loss = None
        self._copy_stream = None

    def loss(self, batch):
        fused = getattr(self.model, "forward_with_loss", None)
        if fused is not None and batch.x.is_cuda:
            # BCE(weight) comes out of the head kernel that produces pred (models/multilevel_gnn.py::forward_with_loss)
            w = self.weight if self.args.weight_balance else None
            pred, feat, loss = fused(batch, batch.y.reshape(-1, 2).to(torch.float32), w)
        else:
            pred, feat = self.model(batch)
            loss = self.crit(pred.to(torch.float32), batch.y.reshape(-1, 2).to(torch.float32))
        return loss + self.model.get_feature_loss(feat)

    def _fwd_bwd(self, batch):
        self.model.train()
        loss = self.loss(batch)
        # == optimizer.zero_grad(); loss.backward() with the gradients landing in the bucket views (p.grad)
        from . import functional as Fn
        Fn.GRAD_SLOTS_ENABLED = loss.is_cuda
        try:
            grads = torch.autograd.grad(loss, self.params, allow_unused=True)
        finally:
            Fn.GRAD_SLOTS_ENABLED = False
        self.bucket.store(grads)
        return loss.detach()

    def _update(self):
        if self.args.clip_grad:
            torch.nn.utils.clip_grad_norm_(self.params, max_norm=20, norm_type=2)
        self.opt.step()

    def _step_eager(self, batch):
        loss = self._fwd_bwd(batch)
        if self.peer is None:
            self.bucket.all_reduce(self.world)
        self._update()         # PeerAdam: the update kernel reduces the gradients over NVLink itself
        return loss

    def capture(self, batch, warmup=3):
        """Capture the step as CUDA graphs over ``batch``'s device tensors (they become the static input
        buffers).  The CSR / pool layouts are built during the warm-up steps (their one-time host syncs are not
        capturable).  Single GPU: ONE graph (fwd, loss, bwd, Adam).  Data parallel with PeerAdam: also ONE graph
        (fwd, loss, bwd, the fused reduce-scatter/Adam/all-gather kernel).  Data parallel over NCCL: graph A (fwd,
        loss, bwd) -> the NCCL all-reduce issued eagerly on the same stream -> graph B (Adam); the collective stays
        outside the capture so that NCCL's own stream/event management never interferes with it."""
        self.static_batch = batch
        # reference copies of the topology fields: keyless batches (full upload) are verified against them on the device
        self._topo_ref = {k: getattr(batch, k).clone() for k in self.STATIC_TOPOLOGY_FIELDS
                          if torch.is_tensor(getattr(batch, k, None))}
        self._topo_bad = torch.zeros((), dtype=torch.bool, device=self.flat.device)
        self._topo_compared = False
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._step_eager(batch)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        if self.world > 1 and self.peer is None:
            self.graph_update = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.static_loss = self._fwd_bwd(batch)
            with torch.cuda.graph(self.graph_update, pool=self.graph.pool()):
                self._update()
        else:
            self.graph_update = None
            with torch.cuda.graph(self.graph):
                self.static_loss = self._step_eager(batch)
        return self

    def _replay(self):
        self.graph.replay()
        if self.graph_update is not None:
            self.bucket.all_reduce(self.world)
            self.graph_update.replay()
        return self.static_loss

    def step_prefetched(self):
        if self.peer is not None and self.opt.failed():
            raise RuntimeError("Trainer: the fused NVLink update timed out waiting for a peer rank")
        self._take_staged()
        return self._replay()

    def loss_to_host(self, loss):
        """Start the device->host copy of a step's loss into a pinned slot and return a handle whose ``get()`` waits for
        THAT copy only.  train.py:62 reads ``loss.item()`` right after the step, which idles the GPU for a launch latency
        every step; reading step i's loss while step i+1 runs gives the host the same number one step later."""
        if getattr(self, "_loss_ring", None) is None:
            self._loss_ring = [torch.zeros(2, dtype=torch.float32).pin_memory() for _ in range(4)]
            self._loss_events = [torch.cuda.Event() for _ in range(4)]
            self._loss_slot = 0
        i = self._loss_slot
        self._loss_slot = (i + 1) % len(self._loss_ring)
        self._loss_ring[i][:1].copy_(loss.reshape(1), non_blocking=True)
        if getattr(self, "_topo_compared", False):      # keyed batches never upload a topology: nothing to report
            self._loss_ring[i][1:].copy_(self._topo_bad.reshape(1), non_blocking=True)
        self._loss_events[i].record()
        return _PendingLoss(self._loss_ring[i], self._loss_events[i])

    def step(self, batch=None):
        """forward, loss, backward, (all-reduce), Adam.  Returns the loss as a device scalar (the
        reference's ``loss.item()`` host sync is the caller's choice).  With a captured graph, ``batch`` must
        be the static batch (or None); use ``load_batch`` to feed new data."""
        if self.peer is not None and self.opt.failed():
            # a rank gave up waiting for a peer inside the fused update kernel (rank skew beyond the timeout, a dead rank): the
            # kernels skipped that update on every rank and refuse to run again -- stop here instead of training on
            raise RuntimeError("Trainer: the fused NVLink update timed out waiting for a peer rank; parameters were left "
                               "untouched by the failed step.  Restart the job (or run with peer_update=False).")
        if self.graph is not None:
            if batch is not None and batch is not self.static_batch:
                self.load_batch(batch)
            return self._replay()
        return self._step_eager(batch)


def reassemble(gathered, n_items):
    """Rows gathered from every rank of an unshuffled plan (data.TopologyLoader(shuffle=False, drop_last=False).index_batches())
    -- [world, steps, B, ...], slot (r, s, j) holding row j of rank r's batch s, padding included -- back in dataset order: slot
    (r, s, j) is dataset row s*B*world + r*B + j, so the valid rows are the first ``n_items`` of the (s, r, j)-ordered slots."""
    w, st, b = gathered.shape[:3]
    return gathered.transpose(0, 1).reshape(st * w * b, *gathered.shape[3:])[:n_items]


class EvalResult(NamedTuple):
    """The metrics of one split and, when asked for, pred [n, 2] on the host in dataset order."""
    auc: float
    acc: float
    bce: float
    n: int
    pred: Optional[torch.Tensor] = None


class Evaluator(StaticBatchFeed):
    """The reference's per-epoch ``eval()`` of a split (train.py:71-109, called on train / valid / test every epoch) on the B200:
    ``capture()`` records ONE forward-only CUDA graph of ``MultilevelGNN.predict`` (eval mode, its own memory pool) over a
    batch of ``batch_size`` graphs; ``evaluate(dataset, topo)`` replays it over an unshuffled plan that visits every sample
    exactly once (data-parallel: each rank its own shard), gathers pred and y, and computes BCE, accuracy and ROC AUC in one
    kernel (mlg_eval_metrics) -- one host synchronisation per split.

    The graph reads the parameters in place, so it always evaluates the latest optimizer update; if a parameter's storage
    moved since capture (e.g. a Trainer re-homed it into its flat buffer), ``evaluate`` re-captures first.
    ``criterion_weight`` is the Trainer's: the BCE uses it, as its class row, only when ``args.weight_balance``."""

    def __init__(self, model, args, batch_size=None, criterion_weight=None, world_size=1):
        self.model, self.args, self.world = model, args, world_size
        self.rank = dist.get_rank() if world_size > 1 else 0
        self.batch_size = int(batch_size or args.batch_size)
        self.class_w = None
        if criterion_weight is not None and args.weight_balance:
            w = torch.as_tensor(criterion_weight, dtype=torch.float32).reshape(-1, 2)
            if not torch.equal(w, w[:1].expand_as(w)):
                raise ValueError("Evaluator: a [B, 2] criterion weight must have equal rows (a class weight); per-position "
                                 "weights have no meaning across a split")
            self.class_w = w[0].contiguous()
        self.graph = None
        self.static_batch = None
        self._copy_stream = None
        self._example = None

    def _param_ptrs(self):
        return [p.data_ptr() for p in self.model.parameters()]

    def capture(self, batch, warmup=2):
        """Record the forward-only graph over ``batch`` (a device batch of ``batch_size`` graphs with a ``topology_key``, e.g.
        data.to_device(data.collate(...))).  Its per-sample fields (x, y, age) are cloned into the static input buffers; the
        topology fields are the batch's own (device-resident, shared).  The CSR / pool layouts are built in the warm-up."""
        B = int(batch.age.shape[0])
        if B != self.batch_size:
            raise ValueError("Evaluator.capture: the batch holds %d graphs, batch_size is %d" % (B, self.batch_size))
        if getattr(batch, "topology_key", None) is None:
            raise ValueError("Evaluator.capture: needs a keyed batch (data.collate / data.to_device)")
        from .synth import GraphBatch
        from .data import PER_SAMPLE_FIELDS
        self._example = batch
        static = GraphBatch(**{k: v for k, v in vars(batch).items()})
        for k in PER_SAMPLE_FIELDS:
            if not torch.is_tensor(getattr(batch, k, None)):
                raise ValueError("Evaluator.capture: the batch has no %r" % k)
            setattr(static, k, getattr(batch, k).clone())
        self.static_batch = static
        self._copy_stream = None
        dev = static.x.device
        if self.class_w is not None:
            self.class_w = self.class_w.to(dev)
        # predict runs in eval mode and restores the model's mode afterwards
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.model.predict(static)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_pred = self.model.predict(static)[0]
        self._ptrs = self._param_ptrs()
        return self

    # the batches are built here from the dataset: only the per-sample fields travel, into the first B' sample slots
    def _step_fields(self, host_batch):
        from .data import PER_SAMPLE_FIELDS
        return list(PER_SAMPLE_FIELDS)

    def _check_topology(self, host_batch):
        pass

    @staticmethod
    def _fill(dst, src):
        dst[:src.shape[0]].copy_(src, non_blocking=True)

    def evaluate(self, dataset, topo, with_pred=True):
        """Forward-only pass over the whole split ``dataset`` (records with x / y / age, as data.collate takes them; ``topo``
        the split's FoldTopology) -> EvalResult(auc, acc, bce, n, pred).  Data parallel: every rank calls it with the same
        dataset and gets the same result.  A short tail batch fills the first B' slots of the static buffers (the graphs of
        a batch do not interact in the forward, so the padding rows only produce predictions that are dropped); a rank whose
        last batch is empty still replays, so all ranks step together."""
        from .data import TopologyLoader, collate
        if self.graph is None:
            raise RuntimeError("Evaluator: call capture(batch) first")
        want = "%s-b%d" % (topo.key, self.batch_size)
        if self.static_batch.topology_key != want:
            raise ValueError("Evaluator: captured for topology_key=%r, this split's topology is %r"
                             % (self.static_batch.topology_key, want))
        if self._param_ptrs() != self._ptrs:
            self.capture(self._example)          # parameters were re-homed since capture: the graph reads stale storage
        n = len(dataset)
        if n == 0:
            raise ValueError("Evaluator: empty split")
        B = self.batch_size
        plan = TopologyLoader(dataset, topo, B, shuffle=False, drop_last=False, rank=self.rank, world=self.world).index_batches()
        steps = len(plan)
        dev = self.static_pred.device
        out = torch.empty(steps, 2, B, 2, dtype=torch.float32, device=dev)      # per step: [pred | y] of the B slots
        y_static = self.static_batch.y.view(B, 2)

        def host(s):
            idx = plan[s]
            return collate([dataset[int(i)] for i in idx], topo) if idx.numel() else None

        nxt = host(0)
        if nxt is not None:
            self.prefetch(nxt)
        for s in range(steps):
            staged = nxt is not None
            nxt = host(s + 1) if s + 1 < steps else None      # collated on the host while the device works
            if staged:
                self._take_staged()
            self.graph.replay()
            out[s, 0].copy_(self.static_pred)        # D2D, outside the graph
            out[s, 1].copy_(y_static)
            if nxt is not None:
                self.prefetch(nxt)
        if self.world > 1:
            gathered = torch.empty(self.world * steps, 2, B, 2, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(gathered, out)
            gathered = gathered.view(self.world, steps, 2, B, 2)
        else:
            gathered = out.view(1, steps, 2, B, 2)
        rows = reassemble(gathered.permute(0, 1, 3, 2, 4), n)         # [n, 2 (pred | y), 2]
        res = torch.empty(3 + (2 * n if with_pred else 0), dtype=torch.float32, device=dev)
        pred = rows[:, 0].contiguous()
        y = rows[:, 1].contiguous()
        if with_pred:
            res[3:].copy_(pred.view(-1))
        eval_metrics(pred, y, self.class_w, out=res[:3])
        host_res = res.cpu()                     # the one host synchronisation of the split
        auc, acc, bce = float(host_res[2]), float(host_res[1]), float(host_res[0])
        return EvalResult(auc, acc, bce, n, host_res[3:].view(n, 2).clone() if with_pred else None)


def eval_metrics(pred, y, class_w=None, out=None):
    """[bce, acc, auc] (float32 device tensor) of pred [n, 2] against y [n, 2] in one launch (mlg_eval_metrics): BCELoss(weight)
    with the class row ``class_w`` [2], argmax accuracy, and the exact ROC AUC of pred[:, 1] (NaN with one class only)."""
    from . import _cabi
    L = _cabi.lib()
    _cabi.require_cuda(pred, y, class_w)
    pred = pred.detach().float().contiguous()
    y = y.detach().float().reshape(-1, 2).contiguous()
    n = pred.shape[0]
    if pred.shape != (n, 2) or y.shape[0] != n:
        raise ValueError("eval_metrics: pred and y must both be [n, 2]")
    cw = None if class_w is None else class_w.detach().float().reshape(2).contiguous()
    if out is None:
        out = torch.empty(3, dtype=torch.float32, device=pred.device)
    ws_bytes = int(L.mlg_eval_metrics_workspace_bytes(n))
    ws = torch.empty(-(-ws_bytes // 8), dtype=torch.float64, device=pred.device)
    with torch.cuda.device(pred.device), _cabi.span("eval_metrics", 16 * n):
        _cabi.check(L.mlg_eval_metrics(_cabi.fptr(pred), _cabi.fptr(y), n, _cabi.fptr(cw, True), _cabi.fptr(out), _cabi.ptr(ws),
                                       ws_bytes, _cabi.stream_ptr()), "mlg_eval_metrics")
    return out
