"""Pathway Shapley values for MultilevelGNN against a background cohort, on the B200 kernels.

``PathwayShapley`` answers "how much of this patient's predicted probability, relative to the cohort's expected prediction,
does each pathway (or pathway x omic segment, or omic) account for?" with Shapley values whose players are sets of cells of
the head's input grid ``pca_feature`` [B, 32, 146, 3P]: the values add up exactly to F(x) - E_j F(background_j), where each
coalition is evaluated through the head's own non-linearities (ReLUs, max-pool, softmax) -- not linearised.

    shap = PathwayShapley(model, args, background=train_x, players="pathway", samples=32, seed=0, target=1, batch_size=32)
    shap.capture(device_batch)          # keyed batch of batch_size graphs (data.collate / data.to_device), as Evaluator.capture
    res = shap.explain(dataset, topo)   # records with x / y / age, as Evaluator.evaluate / Knockout.screen
    res.values [n, K]; res.base [n]; res.pred [n, 2]; res.delta [n]

The trunk is not involved: one captured ``predict`` graph gives every patient's and every background row's grid, the head's
own per-cell convs (mlg_head_conv_pool_fwd with a 1 x 1 window) give per-cell tables, and mlg_shap_chains walks the
permutations incrementally through the max-pool and the first Linear (csrc/pathway_shapley.cu).
"""
import itertools
from collections import namedtuple

import torch
import torch.nn as nn

from . import _cabi
from .attribution import _GOLDEN, _M64, _mix64
from .train import StaticBatchFeed, frozen_parameters

ShapleyResult = namedtuple("ShapleyResult", "values base pred delta")

PATHWAYS = 146
SEGMENTS = 3 * PATHWAYS
EXACT_MAX_PLAYERS = 8


def parse_players(players):
    """Players -> list of int64 tensors of segment ids (segment = 3 * pathway + omic, in the reference's pathway order).
    "pathway": 146 players {3p, 3p + 1, 3p + 2}; "segment": 438 singletons; "omic": 3 players {3p + o for every p};
    otherwise a non-empty list of disjoint, non-empty sequences of ids in [0, 438)."""
    if isinstance(players, str):
        if players == "pathway":
            return [torch.arange(3 * p, 3 * p + 3) for p in range(PATHWAYS)]
        if players == "segment":
            return [torch.tensor([s]) for s in range(SEGMENTS)]
        if players == "omic":
            return [torch.arange(o, SEGMENTS, 3) for o in range(3)]
        raise ValueError("players must be 'pathway', 'segment', 'omic' or a list of segment-id sequences (got %r)" % players)
    out, seen = [], torch.zeros(SEGMENTS, dtype=torch.bool)
    for k, grp in enumerate(players):
        t = torch.as_tensor(grp).reshape(-1)
        if t.numel() == 0:
            raise ValueError("player %d: no segment" % k)
        if t.is_floating_point() or t.is_complex() or t.dtype == torch.bool:
            raise ValueError("player %d: segment ids must be integers (got %s)" % (k, t.dtype))
        t = torch.unique(t.to(torch.int64))
        if int(t.min()) < 0 or int(t.max()) >= SEGMENTS:
            raise ValueError("player %d: segment id out of range [0, %d)" % (k, SEGMENTS))
        if bool(seen[t].any()):
            raise ValueError("player %d: overlaps an earlier player (players must be disjoint)" % k)
        seen[t] = True
        out.append(t)
    if not out:
        raise ValueError("players: no player given")
    return out


def segment_row(reorder_idxs=None):
    """Grid row of every pathway [146]: with the model's pathway reorder (x[:, :, reorder_idxs]) pathway p sits at the
    position q with reorder_idxs[q] == p, as attribution.pathway_reduce maps it back."""
    if reorder_idxs is None:
        return torch.arange(PATHWAYS)
    r = torch.as_tensor(reorder_idxs).to("cpu", torch.int64).reshape(-1)
    row = torch.empty(PATHWAYS, dtype=torch.int64)
    row[r] = torch.arange(PATHWAYS)
    return row


def player_tables(groups, pca_dim, kh, kw, reorder_idxs=None):
    """(owner int32 [146 * 3P], win_ptr int32 [K + 1], win_idx int32) for the grid [146, 3P] and the (kh, kw) floor-mode
    max-pool: owner[cell] = the player holding the cell (-1: none); player k's windows, ascending, are
    win_idx[win_ptr[k]:win_ptr[k + 1]] (window = ho * Wo + wo).  A cell outside every window (floor mode) joins no window."""
    P = int(pca_dim)
    Wg = 3 * P
    Ho, Wo = PATHWAYS // kh, Wg // kw
    row = segment_row(reorder_idxs)
    owner = torch.full((PATHWAYS, Wg), -1, dtype=torch.int32)
    ptr, idx = [0], []
    for k, segs in enumerate(groups):
        wins = set()
        for s in segs.tolist():
            q, o = int(row[s // 3]), s % 3
            owner[q, o * P:(o + 1) * P] = k
            if q // kh < Ho:
                wins.update(q // kh * Wo + c // kw for c in range(o * P, (o + 1) * P) if c // kw < Wo)
        idx.extend(sorted(wins))
        ptr.append(len(idx))
    return owner.reshape(-1), torch.tensor(ptr, dtype=torch.int32), torch.tensor(idx, dtype=torch.int32)


def _stream(seed, a, b):
    return _mix64(((_mix64((seed + _GOLDEN) & _M64) ^ a) + _GOLDEN + b) & _M64)


def shapley_perms(seed, S, K):
    """The S permutations of K players [S, K] int64, in antithetic pairs: row 2m is pi_m, row 2m + 1 its reverse.  pi_m is a
    Fisher-Yates shuffle driven by a splitmix64 stream keyed by (seed, m) only: shared by every patient."""
    if S < 2 or S % 2 or K < 1:
        raise ValueError("shapley_perms: needs an even S >= 2 and K >= 1")
    out = torch.empty(S, K, dtype=torch.int64)
    for m in range(S // 2):
        key = _stream(seed, m, 0x5EED_0000_0001)
        p = list(range(K))
        for t in range(K - 1, 0, -1):
            h = _mix64((key + (K - t) * _GOLDEN) & _M64)
            u = ((h >> 32) * (t + 1)) >> 32
            p[t], p[u] = p[u], p[t]
        out[2 * m] = torch.tensor(p)
        out[2 * m + 1] = torch.tensor(p[::-1])
    return out


def shapley_rows(seed, index, S, M):
    """Background rows [S] int64 in [0, M) of the patient at position ``index`` of the dataset: pair m (rows 2m, 2m + 1)
    uses j_m, the m-th output of a splitmix64 stream keyed by (seed, index)."""
    if S < 2 or S % 2 or M < 1 or index < 0:
        raise ValueError("shapley_rows: needs an even S >= 2, M >= 1 and index >= 0")
    key = _stream(seed, index, 0x5EED_0000_0002)
    j = [((_mix64((key + (m + 1) * _GOLDEN) & _M64) >> 32) * M) >> 32 for m in range(S // 2)]
    return torch.tensor(j, dtype=torch.int64).repeat_interleave(2)


def shapley_draws(seed, index, S, M, K):
    """Sampled mode's draws for the patient at position ``index``: (perm [S, K], j [S]).  A pure function of its arguments:
    perm depends on (seed, m) only, j on (seed, index, m), so a patient's values do not depend on batch_size, on the other
    patients or on its slot."""
    return shapley_perms(seed, S, K), shapley_rows(seed, index, S, M)


def exact_perms(K):
    """All K! permutations of K players [K!, K] int64, in lexicographic order."""
    return torch.tensor(list(itertools.permutations(range(K))), dtype=torch.int64).reshape(-1, K)


def head_geometry(model):
    """(kh, kw, Ho, Wo, H) of the head every shipped config builds -- the conditions of MultilevelGNN._fused_head_ok without
    its 64-row limit; anything else raises NotImplementedError."""
    cm, hd, pool = model.conv_model, model.head, model.pooling
    why = None
    ks = pool.kernel_size if isinstance(pool.kernel_size, tuple) else (pool.kernel_size,) * 2
    if not (len(cm) == 4 and isinstance(cm[0], nn.Conv2d) and isinstance(cm[2], nn.Conv2d) and type(cm[1]) is nn.ReLU
            and type(cm[3]) is nn.ReLU and len(hd) == 5 and isinstance(hd[0], nn.Linear) and type(hd[1]) is nn.ReLU
            and isinstance(hd[2], nn.Dropout) and isinstance(hd[3], nn.Linear) and isinstance(hd[4], nn.Softmax)):
        why = "the head is not conv/ReLU/conv/ReLU + Linear/ReLU/Dropout/Linear/Softmax"
    elif any(m._forward_hooks or m._forward_pre_hooks or m._backward_hooks for m in list(cm) + list(hd) + [pool, model.drop1]):
        why = "hooks on a head module"
    elif not (cm[0].kernel_size == (1, 1) and cm[2].kernel_size == (1, 1) and cm[0].in_channels == 32
              and cm[0].out_channels == 32 and cm[2].in_channels == 32 and cm[2].out_channels == 64
              and cm[0].bias is not None and cm[2].bias is not None):
        why = "the convs are not 1x1 32 -> 32 -> 64 with biases"
    elif not (pool.stride in (ks, pool.kernel_size) and pool.padding in (0, (0, 0)) and pool.dilation in (1, (1, 1))
              and not pool.ceil_mode and not pool.return_indices):
        why = "the max-pool is not stride = kernel, floor mode"
    else:
        Ho, Wo = PATHWAYS // ks[0], (3 * model.pca_dim) // ks[1]
        H = hd[0].out_features
        f_in = 64 * Ho * Wo + (1 if model.args.use_age else 0)
        if not (Ho >= 1 and Wo >= 1 and hd[0].in_features == f_in and hd[3].out_features == 2 and hd[3].in_features == H
                and H % 32 == 0 and H <= 512 and hd[0].bias is not None and hd[3].bias is not None and hd[4].dim in (1, -1)):
            why = "the Linear layers do not match the grid (or H % 32 != 0, H > 512)"
    if why is not None:
        raise NotImplementedError("PathwayShapley: unsupported head: " + why)
    return int(ks[0]), int(ks[1]), Ho, Wo, H


class PathwayShapley(StaticBatchFeed):
    """Shapley values of ``pred[:, target]`` (the softmax probability) whose players are sets of pooled segments of the head's
    input grid, against a background cohort.

    Players.  Segment id = 3 * pathway + omic in the reference's pathway order; with ``reorder_pathway`` pathway p sits at
    grid row q with reorder_idxs[q] == p (as attribution.pathway_reduce maps it).  A segment covers grid row q and columns
    o * P .. o * P + P - 1 (P = pca_dim).  players: "pathway" (K = 146, each pathway's 3 segments), "segment" (K = 438),
    "omic" (K = 3, each omic's 146 segments) or a list of disjoint segment-id sequences; overlapping groups, ids outside
    [0, 438) or an empty list raise ValueError.  Segments in no player stay at the patient's values throughout.

    Value function.  v(S) = F(grid with the cells of the players in S from the patient and the other players' cells from
    background row j), at the patient's age: interventional Shapley against the background at the head's input, eval
    semantics (no dropout).  background: [M, N] profiles (e.g. the training split's x), finite, M >= 1; their grids come from
    the same captured ``predict`` as the patients', recomputed on every ``explain`` call.

    Sampled mode (``samples`` = S, even, >= 2): S / 2 antithetic pairs (pi_m, reversed pi_m), both chains of a pair with one
    background row j_{p,m} (``shapley_draws``: pi_m depends on (seed, m) only and is shared by all patients, j on (seed,
    dataset index, m), so a patient's bits do not depend on batch_size, batch company or slot).  phi_k = mean over the
    patient's S chains of the change in F when k joins.  Exact mode (``samples="exact"``, K <= 8): every one of the K!
    permutations with every background row, weight 1 / (K! M): the exact Shapley values against the uniform background.

    Result (host tensors, dataset order): ``values`` [n, K] float32 in player order; ``base`` [n] float64, the mean over the
    patient's chains of F(start state) (E_j F(background_j) with the non-player segments at the patient's values);
    ``pred`` [n, 2], predict's output; ``delta`` [n] float64 = pred[:, target] - base - values.sum(1), zero up to the fp32
    rounding of the incremental updates.  A player whose cells change no window maximum gets exactly 0 (the dummy property):
    with gbm's floor-mode (4, 2) pool grid rows 144 and 145 are never read, with lgg's (4, 2) pool on 9 columns column 8.

    Cost.  ``explain`` packs the first Linear's weight by pooling window once per call ([Ho * Wo][64][H] fp32: 7 MB for gbm,
    19 MB for lgg, 172 MB for kirc).  One permutation of 146 pathways then reads it about once (kirc, 1 x 1 windows) or four
    times (gbm / lgg, windows four rows high), shared by the 16 chains of a CTA.  The parameters are read in place and frozen
    while the graph is recorded (no weight-gradient kernel runs, no ``.grad`` is written); if their storage moved since
    capture (e.g. a Trainer re-homed them), ``explain`` re-captures first.  One host synchronisation per call."""

    def __init__(self, model, args, background, players="pathway", samples=32, seed=0, target=1, batch_size=32):
        self.model, self.args = model, args
        if target not in (0, 1):
            raise ValueError("PathwayShapley: target must be 0 or 1 (got %r)" % (target,))
        self.target = int(target)
        self.batch_size = int(batch_size)
        if self.batch_size < 2:
            raise ValueError("PathwayShapley: batch_size must be >= 2 (the factored first layer runs on replicated graphs)")
        bg = torch.as_tensor(background).detach().to("cpu", torch.float32, copy=True)
        n_nodes = 3 * model.node_num
        if bg.dim() != 2 or bg.shape[0] < 1 or bg.shape[1] != n_nodes:
            raise ValueError("PathwayShapley: background must be [M >= 1, %d] (got %s)" % (n_nodes, tuple(bg.shape)))
        if not bool(torch.isfinite(bg).all()):
            raise ValueError("PathwayShapley: background values must be finite")
        self.background = bg.contiguous()
        self.groups = parse_players(players)
        self.K = len(self.groups)
        if isinstance(samples, str):
            if samples != "exact":
                raise ValueError("PathwayShapley: samples must be an even int >= 2 or 'exact' (got %r)" % samples)
            if self.K > EXACT_MAX_PLAYERS:
                raise ValueError("PathwayShapley: exact mode enumerates K! permutations; allowed for K <= %d (got K = %d)"
                                 % (EXACT_MAX_PLAYERS, self.K))
            self.samples = "exact"
        else:
            if isinstance(samples, bool) or int(samples) != samples or int(samples) < 2 or int(samples) % 2:
                raise ValueError("PathwayShapley: samples must be even and >= 2 (antithetic pairs) (got %r)" % (samples,))
            self.samples = int(samples)
        self.seed = int(seed)
        self.kh, self.kw, self.Ho, self.Wo, self.H = head_geometry(model)
        self.Hg, self.Wg = PATHWAYS, 3 * model.pca_dim
        self.graph = None
        self.static_batch = None
        self._copy_stream = None
        self._example = None
        self._tables = None

    def _param_ptrs(self):
        return [p.data_ptr() for p in self.model.parameters()]

    def _reorder(self):
        return self.model.reorder_idxs if (self.args.reorder_pathway and self.model.reorder_idxs is not None) else None

    # one replay: predict over the static batch, then the head's per-cell convs of its grids
    def _body(self):
        B = self.batch_size
        pred, feat = self.model.predict(self.static_batch)
        x_cl = feat.permute(0, 2, 3, 1)
        if not x_cl.is_contiguous():
            x_cl = x_cl.contiguous()
        cm = self.model.conv_model
        ld = 64 * self.Hg * self.Wg
        cells = torch.empty(B, ld, dtype=torch.float32, device=x_cl.device)
        with _cabi.span("head_conv_pool_fwd", 4 * (x_cl.numel() + cells.numel())):
            _cabi.check(_cabi.lib().mlg_head_conv_pool_fwd(
                _cabi.fptr(x_cl), _cabi.fptr(cm[0].weight.view(32, 32)), _cabi.fptr(cm[0].bias),
                _cabi.fptr(cm[2].weight.view(64, 32)), _cabi.fptr(cm[2].bias), None, None, 0.0, B, self.Hg, self.Wg, 1, 1,
                _cabi.fptr(cells), ld, _cabi.stream_ptr()), "mlg_head_conv_pool_fwd")
        self.out_pred, self.out_cells = pred, cells

    def capture(self, batch, warmup=2):
        """Record the graph over ``batch`` (a keyed device batch of ``batch_size`` graphs, as Evaluator.capture)."""
        B = int(batch.age.shape[0])
        if B != self.batch_size:
            raise ValueError("PathwayShapley.capture: the batch holds %d graphs, batch_size is %d" % (B, self.batch_size))
        if getattr(batch, "topology_key", None) is None:
            raise ValueError("PathwayShapley.capture: needs a keyed batch (data.collate / data.to_device)")
        from .synth import GraphBatch
        from .data import PER_SAMPLE_FIELDS
        self._example = batch
        static = GraphBatch(**{k: v for k, v in vars(batch).items()})
        for k in PER_SAMPLE_FIELDS:
            setattr(static, k, getattr(batch, k).clone())
        self.static_batch = static
        self._copy_stream = None
        dev = static.x.device
        if self.model.reorder_idxs is not None and self.model.reorder_idxs.device != dev:
            # the head reorders the pathways with this index; a graph cannot copy it from pageable host memory on every replay
            self.model.reorder_idxs = self.model.reorder_idxs.to(dev)
        self._bad = torch.zeros(1, dtype=torch.int32, device=dev)
        with frozen_parameters(self.model, grad_enabled=False):
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    self._body()
            cur.wait_stream(side)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._body()
        self._ptrs = self._param_ptrs()
        return self

    def eager(self):
        """One uncaptured pass of what a replay runs, on the static buffers; the outputs land in ``out_pred`` / ``out_cells``
        as after a replay."""
        with frozen_parameters(self.model, grad_enabled=False):
            self._body()

    def _step_fields(self, host_batch):
        from .data import PER_SAMPLE_FIELDS
        return list(PER_SAMPLE_FIELDS)

    def _check_topology(self, host_batch):
        pass

    @staticmethod
    def _fill(dst, src):
        dst[:src.shape[0]].copy_(src, non_blocking=True)

    def _grids(self, records, topo, out_cells, out_pred=None):
        """Replays over ``records`` in batches of batch_size (collated on the host while the device works): per record its
        per-cell table (and predict's output)."""
        from .data import collate
        B, n = self.batch_size, len(records)
        starts = list(range(0, n, B))

        def host(j):
            return collate(records[starts[j]:starts[j] + B], topo)

        self.prefetch(host(0))
        for j, s in enumerate(starts):
            nxt = host(j + 1) if j + 1 < len(starts) else None
            self._take_staged()
            self.graph.replay()
            m = min(B, n - s)
            out_cells[s:s + m].copy_(self.out_cells[:m])
            if out_pred is not None:
                out_pred[s:s + m].copy_(self.out_pred[:m])
            if nxt is not None:
                self.prefetch(nxt)

    def _head_tables(self, dev):
        """The first Linear packed by window [Ho * Wo, 64, H], its age column (or None), and the player tables (once)."""
        W1 = self.model.head[0].weight.detach()
        F = 64 * self.Ho * self.Wo
        w1p = W1[:, :F].reshape(self.H, 64, self.Ho * self.Wo).permute(2, 1, 0).contiguous()
        w1age = W1[:, F].contiguous() if self.args.use_age else None
        if self._tables is None:
            owner, ptr, idx = player_tables(self.groups, self.model.pca_dim, self.kh, self.kw, self._reorder())
            self._tables = [t.to(dev) if t.numel() else torch.zeros(1, dtype=torch.int32, device=dev)
                            for t in (owner, ptr, idx)]
        return w1p, w1age

    def explain(self, dataset, topo):
        """Shapley values of every record of ``dataset`` (records with x / y / age, as data.collate takes them; ``topo`` the
        dataset's FoldTopology) -> ShapleyResult of host tensors, in dataset order."""
        import types
        if self.graph is None:
            raise RuntimeError("PathwayShapley: call capture(batch) first")
        want = "%s-b%d" % (topo.key, self.batch_size)
        if self.static_batch.topology_key != want:
            raise ValueError("PathwayShapley: captured for topology_key=%r, this dataset's topology is %r"
                             % (self.static_batch.topology_key, want))
        if self._param_ptrs() != self._ptrs:
            self.capture(self._example)          # parameters were re-homed since capture: the graph reads stale storage
        n = len(dataset)
        if n == 0:
            raise ValueError("PathwayShapley: empty dataset")
        M, K = self.background.shape[0], self.K
        dev = self._bad.device
        ld = 64 * self.Hg * self.Wg
        records = [dataset[i] for i in range(n)]
        if self.samples == "exact":
            perm = exact_perms(K)
            G = perm.shape[0]
            n_cp = n * M
            chain_pat = torch.arange(n).repeat_interleave(M)
            chain_bg = torch.arange(M).repeat(n).unsqueeze(0).expand(G, n_cp)
        else:
            G = self.samples
            perm = shapley_perms(self.seed, G, K)
            n_cp = n
            chain_pat = torch.arange(n)
            chain_bg = torch.stack([shapley_rows(self.seed, i, G, M) for i in range(n)], 1)     # [G, n]
        R = G * n_cp // n                                       # chains per patient, rows p * R .. p * R + R - 1
        up = [t.to(torch.int32).contiguous().pin_memory().to(dev, non_blocking=True) for t in (perm, chain_pat, chain_bg)]
        slot_ptr = torch.arange(0, n * R + 1, R, dtype=torch.int32).pin_memory().to(dev, non_blocking=True)
        w = torch.full((n * R,), 1.0 / R, dtype=torch.float32, device=dev)
        age = torch.tensor([float(torch.as_tensor(r.age).reshape(())) for r in records], dtype=torch.float32)
        age = age.pin_memory().to(dev, non_blocking=True)

        pat = torch.empty(n, ld, dtype=torch.float32, device=dev)
        bgt = torch.empty(M, ld, dtype=torch.float32, device=dev)
        pred = torch.empty(n, 2, dtype=torch.float32, device=dev)
        bg_records = [types.SimpleNamespace(x=self.background[j], age=0.0, y=torch.zeros(2)) for j in range(M)]
        with frozen_parameters(self.model, grad_enabled=False):
            self._grids(records, topo, pat, pred)
            self._grids(bg_records, topo, bgt)
            w1p, w1age = self._head_tables(dev)
            owner, win_ptr, win_idx = self._tables
            hd = self.model.head
            contrib = torch.empty(n * R, K, dtype=torch.float32, device=dev)
            p0 = torch.empty(n * R, dtype=torch.float32, device=dev)
            pT = torch.empty(n * R, dtype=torch.float32, device=dev)
            self._bad.zero_()
            L = _cabi.lib()
            with _cabi.span("shap_chains", 4 * w1p.numel()):
                _cabi.check(L.mlg_shap_chains(
                    _cabi.fptr(pat), n, _cabi.fptr(bgt), M, ld, self.Hg, self.Wg, self.kh, self.kw, _cabi.fptr(w1p),
                    _cabi.fptr(hd[0].bias), _cabi.fptr(w1age, True), _cabi.fptr(age), _cabi.fptr(hd[3].weight),
                    _cabi.fptr(hd[3].bias), self.target, self.H, _cabi.iptr(owner), _cabi.iptr(win_ptr), _cabi.iptr(win_idx),
                    K, _cabi.iptr(up[0]), G, _cabi.iptr(up[1]), _cabi.iptr(up[2]), n_cp, _cabi.fptr(contrib),
                    _cabi.fptr(p0), _cabi.fptr(pT), _cabi.iptr(self._bad), _cabi.stream_ptr()), "mlg_shap_chains")
            values = torch.empty(n, K, dtype=torch.float32, device=dev)
            _cabi.check(L.mlg_attr_accumulate(_cabi.fptr(contrib), K, _cabi.fptr(w), _cabi.iptr(slot_ptr), n, K, 0,
                                              _cabi.fptr(values), _cabi.stream_ptr()), "mlg_attr_accumulate")
        self.last_chains = (contrib, p0, pT)
        host_values, host_p0, host_pred, bad = (t.cpu() for t in (values, p0, pred, self._bad))    # the one synchronisation
        if int(bad[0]):
            raise RuntimeError("PathwayShapley: a chain's background row index was outside [0, %d)" % M)
        base = host_p0.view(n, R).double().mean(1)
        delta = host_pred[:, self.target].double() - base - host_values.double().sum(1)
        return ShapleyResult(host_values, base, host_pred, delta)
