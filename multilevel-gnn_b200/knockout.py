"""In-silico knockout screens for MultilevelGNN on the B200 kernels.

``Knockout`` answers "if this gene's mRNA / CNV / methylation were at the baseline (zero, or a cohort profile), how would
this patient's predicted probability change?" exactly -- through the LeakyReLU, pooling and softmax non-linearities that a
gradient linearises away -- by occlusion: every group of nodes of a screen is set to the baseline in turn and the model is
evaluated again.  Only the neighbourhood a knockout reaches is recomputed (csrc/knockout.cu): the first-layer rows T1 that
read a node of the group, the second-layer rows T2 that read a T1 row, and the pooled segments that hold a slot of a T2
node; the model's own head then runs on a batch of knockouts, with one unperturbed row per patient in the same launch.

    ko = Knockout(model, args, groups="gene", baseline=None, target=1, batch_size=32)
    ko.capture(device_batch)            # keyed batch of batch_size graphs, as Evaluator.capture / Attributor.capture
    res = ko.screen(dataset, topo)      # records with x / y / age, as Evaluator.evaluate
    res.delta [n, K]: pred(x with group k at the baseline)[target] - pred(x)[target];  res.pred [n, 2]: the base prediction

``capture`` records two CUDA graphs: the base forward of ``batch_size`` patients (it keeps the second layer's [U | V] rows,
the first layer's per-gene tables and the pooled tensor) and one replay of ``ROWS`` head rows (the incremental trunk, the
head, the per-row differences).  ``screen`` replays the first once per batch of patients and the second once per chunk of
knockouts, gathers the results on the device and synchronises with the host once.
"""
from collections import namedtuple

import torch

from . import _cabi
from . import functional as Fn
from .train import StaticBatchFeed, frozen_parameters

KnockoutResult = namedtuple("KnockoutResult", "delta pred")


def parse_groups(groups, n_nodes):
    """Groups of node indices -> (ptr int64 [K + 1], nodes int64): group k is nodes[ptr[k]:ptr[k + 1]], ascending and
    without repeats.  "gene": K = n_nodes / 3 groups {3g, 3g + 1, 3g + 2} (gene g's mRNA, CNV and methylation nodes);
    "node": K = n_nodes singletons; otherwise a sequence of index sequences (e.g. one pathway's nodes per group; a group
    may be empty)."""
    if isinstance(groups, str):
        if groups == "gene":
            if n_nodes % 3:
                raise ValueError("groups='gene' needs 3 nodes per gene (got %d nodes)" % n_nodes)
            return torch.arange(0, n_nodes + 1, 3, dtype=torch.int64), torch.arange(n_nodes, dtype=torch.int64)
        if groups == "node":
            return torch.arange(n_nodes + 1, dtype=torch.int64), torch.arange(n_nodes, dtype=torch.int64)
        raise ValueError("groups must be 'gene', 'node' or a list of node-index sequences (got %r)" % groups)
    parts = []
    for i, g in enumerate(groups):
        t = torch.as_tensor(g).reshape(-1)
        if t.numel() and (t.is_floating_point() or t.is_complex() or t.dtype == torch.bool):
            raise ValueError("group %d: node indices must be integers (got %s)" % (i, t.dtype))
        t = t.to(torch.int64)
        if t.numel() and (int(t.min()) < 0 or int(t.max()) >= n_nodes):
            raise ValueError("group %d: node index out of range [0, %d)" % (i, n_nodes))
        parts.append(torch.unique(t))
    if not parts:
        raise ValueError("groups: no group given")
    counts = torch.tensor([p.numel() for p in parts], dtype=torch.int64)
    return torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]), torch.cat(parts)


def _spread(ptr, nodes, rowptr, col, n_nodes):
    """One hop of the forward CSR: per group, the rows whose entries read a node of the group, plus the group itself (the
    transpose of the CSR applied to the group indicators).  Returns (ptr, nodes), ascending within a group."""
    K = ptr.numel() - 1
    deg = rowptr[1:] - rowptr[:-1]
    rows = torch.repeat_interleave(torch.arange(n_nodes, dtype=torch.int64), deg)       # row of every CSR entry
    at = torch.sparse_coo_tensor(torch.stack([col.to(torch.int64), rows]), torch.ones(rows.numel()), (n_nodes, n_nodes),
                                 check_invariants=True)
    grp = torch.repeat_interleave(torch.arange(K, dtype=torch.int64), ptr[1:] - ptr[:-1])
    m = torch.sparse_coo_tensor(torch.stack([grp, nodes]), torch.ones(nodes.numel()), (K, n_nodes), check_invariants=True)
    reach = (torch.sparse.mm(m, at.coalesce()) + m).coalesce()
    idx = reach.indices()
    counts = torch.bincount(idx[0], minlength=K)
    return torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]), idx[1].clone()


def neighbourhood_tables(ptr, nodes, rowptr, col, n_nodes):
    """T1 and T2 per group, each as (ptr, nodes): T1 = the group and the rows that read one of its nodes, T2 = T1 and the
    rows that read a T1 row.  ``rowptr`` / ``col``: the forward CSR (row i lists the nodes it reads, self loop included)."""
    rowptr, col = rowptr.to(torch.int64).cpu(), col.to(torch.int64).cpu()
    t1 = _spread(ptr, nodes, rowptr, col, n_nodes)
    return t1, _spread(t1[0], t1[1], rowptr, col, n_nodes)


def slot_tables(t2_ptr, t2_nodes, match, seg_of_slot, n_nodes, n_segments):
    """The pool entries a group reaches: per group its touched segments (s_ptr [K + 1], s_seg ascending) and per touched
    segment its entries (e_ptr, with e_slot = the slot, ascending, and e_t2 = the slot's node's position in the group's T2
    list).  A slot whose node is missing (match < 0) contributes nothing and is not listed."""
    K = t2_ptr.numel() - 1
    match, seg_of_slot = match.to(torch.int64).cpu(), seg_of_slot.to(torch.int64).cpu()
    G = match.numel()
    slots = torch.nonzero(match >= 0).flatten()
    node = match[slots]
    order = torch.argsort(node * G + slots)
    ns_slot = slots[order]                                               # slots grouped by node, ascending within a node
    ns_cnt = torch.bincount(node, minlength=n_nodes)
    ns_ptr = torch.cat([torch.zeros(1, dtype=torch.int64), ns_cnt.cumsum(0)])
    cnt = ns_cnt[t2_nodes]
    ent = torch.repeat_interleave(torch.arange(t2_nodes.numel(), dtype=torch.int64), cnt)      # T2 entry of every pool entry
    start = torch.repeat_interleave(cnt.cumsum(0) - cnt, cnt)
    slot = ns_slot[ns_ptr[t2_nodes[ent]] + torch.arange(ent.numel(), dtype=torch.int64) - start]
    grp = torch.repeat_interleave(torch.arange(K, dtype=torch.int64), t2_ptr[1:] - t2_ptr[:-1])[ent]
    key = grp * n_segments + seg_of_slot[slot]
    order = torch.argsort(key * G + slot)
    key, slot, t2 = key[order], slot[order], (ent - t2_ptr[grp])[order]
    uniq, counts = torch.unique_consecutive(key, return_counts=True)
    s_cnt = torch.bincount(uniq // n_segments, minlength=K)
    zero = torch.zeros(1, dtype=torch.int64)
    return (torch.cat([zero, s_cnt.cumsum(0)]), uniq % n_segments, torch.cat([zero, counts.cumsum(0)]), slot, t2)


def replay_plan(n_patients, n_groups, rows):
    """Chunks of ``rows`` head rows that hold every (patient, group) of ``n_patients`` x ``n_groups``, patients ascending,
    groups ascending within a patient; each patient present in a chunk has ONE base row there (group -1), placed before its
    knockouts.  A patient's groups may span several chunks; the last chunk fills its first rows and pads the rest (patient
    -1, its own base row).  Returns int64 [chunks, rows, 3]: (patient, group or -1, row of that patient's base row)."""
    if n_patients < 1 or n_groups < 1 or rows < 2:
        raise ValueError("replay_plan: needs n_patients >= 1, n_groups >= 1 and rows >= 2")
    seg_pos, seg_pat, seg_k, seg_cnt = [], [], [], []      # runs of one patient's rows inside one chunk: base row + groups
    pos = 0
    for p in range(n_patients):
        k = 0
        while k < n_groups:
            free = rows - pos % rows
            if free < 2:
                pos += free
                free = rows
            take = min(free - 1, n_groups - k)
            seg_pos.append(pos)
            seg_pat.append(p)
            seg_k.append(k)
            seg_cnt.append(take)
            pos += take + 1
            k += take
    n_chunks = -(-pos // rows)
    lens = torch.tensor(seg_cnt, dtype=torch.int64) + 1
    start = torch.tensor(seg_pos, dtype=torch.int64)
    seg = torch.repeat_interleave(torch.arange(lens.numel()), lens)
    off = torch.arange(int(lens.sum())) - torch.repeat_interleave(lens.cumsum(0) - lens, lens)
    out = torch.empty(n_chunks * rows, 3, dtype=torch.int64)
    out[:, 0] = -1
    out[:, 1] = -1
    out[:, 2] = torch.arange(n_chunks * rows) % rows
    at = start[seg] + off
    out[at, 0] = torch.tensor(seg_pat, dtype=torch.int64)[seg]
    out[at, 1] = torch.where(off == 0, -1, torch.tensor(seg_k, dtype=torch.int64)[seg] + off - 1)
    out[at, 2] = start[seg] % rows
    return out.view(n_chunks, rows, 3)


class Knockout(StaticBatchFeed):
    """Captured knockout screen of ``pred[:, target]`` (the softmax probability).

    groups: "gene" (K = 5 135 groups {3g, 3g + 1, 3g + 2}), "node" (K = N singletons) or a list of node-index sequences;
    an index outside [0, N) raises ValueError, an empty group has delta 0.  baseline: None (zeros) or an [N] profile such as
    the cohort mean.  The knocked-out values feed the first layer and the value-attention mask, as ``forward`` would see
    them; age is unchanged.  Eval semantics, no dropout, as ``predict``.

    The parameters are read in place and frozen while the graphs are recorded (no weight-gradient kernel runs, no ``.grad``
    is written); if their storage moved since capture (e.g. a Trainer re-homed them), ``screen`` re-captures first.

    The incremental trunk covers the route ``predict`` takes for the shipped configs: the factored first layer (64 wide),
    the transform-first second layer (64 -> 32, non-relative SAGE) on node-major rows, the value mask ``mult`` and the fused
    pool, with any pca_dim / pool kernel, reorder_pathway and use_age; the head is the model's own.  Other routes raise
    NotImplementedError."""

    # head rows per replay: base rows and knockouts together.  128 rows take the model's generic head (the fused head stops at
    # 64 rows); measured faster than 64 rows on the fused head for gene screens of all three shipped configs (B200, 1000 W,
    # tools/knockout_bench.py, profiles/r05_knockout_*.json: gbm 11.8 vs 12.8, kirc 38.2 vs 54.2, lgg 14.9 vs 17.4 ms per patient)
    ROWS = 128

    def __init__(self, model, args, groups="gene", baseline=None, target=1, batch_size=32):
        self.model, self.args = model, args
        self.groups = groups
        self.batch_size = int(batch_size)
        if self.batch_size < 2:
            raise ValueError("Knockout: batch_size must be >= 2 (the factored first layer runs on replicated graphs)")
        if target not in (0, 1):
            raise ValueError("Knockout: target must be 0 or 1 (got %r)" % (target,))
        self.target = int(target)
        self.baseline = None if baseline is None else torch.as_tensor(baseline, dtype=torch.float32).reshape(-1)
        self._check_config()
        self.graph = None
        self.static_batch = None
        self._copy_stream = None
        self._example = None
        self._tables = None

    def _check_config(self):
        a, m = self.args, self.model
        why = None
        if a.gnn_name.lower() != "sage":
            why = "gnn_name=%r (the incremental trunk is written for non-relative SAGE layers)" % a.gnn_name
        elif len(m.gnn_model) != 2:
            why = "%d GNN layers (the incremental trunk covers two)" % len(m.gnn_model)
        elif a.dense_gnn or a.resgnn or a.repeat_mask:
            why = "dense / residual GNN or repeat_mask (the knockout would reach beyond two hops of rows)"
        elif not a.node_embedding or a.input_emb_drop is not None:
            why = "no factored first layer (node_embedding off or input_emb_drop set)"
        elif not (a.value_att_mask and a.merge_mode == "mult"):
            why = "value mask %r (the incremental pool is written for the multiplicative value mask)" % (
                a.merge_mode if a.value_att_mask else None)
        elif not a.pca_match_mask:
            why = "pca_match_mask=False (missing slots read another patient's node)"
        elif a.device_num != 1:
            why = "device_num=%d" % a.device_num
        elif any(m._hooked(l) for l in m.gnn_model):
            why = "forward hooks on a GNN layer (the layer's rows must be seen in the reference's order)"
        if why is not None:
            raise NotImplementedError("Knockout: not supported for this model: " + why)

    def _param_ptrs(self):
        return [p.data_ptr() for p in self.model.parameters()]

    # ---------------------------------------------------------------------------------------------------------------
    def _base_body(self):
        """The forward of the static batch up to the pool, keeping the tensors the incremental trunk starts from."""
        keep = {}
        Fn.KEEP_STATE = keep
        try:
            pooled = self.model.pool_genes(self.static_batch, fused=True)
        finally:
            Fn.KEEP_STATE = None
        if "rank1" not in keep or "tfirst" not in keep or not keep["tfirst"][5]:
            raise NotImplementedError("Knockout: the forward did not take the factored first layer and the node-major "
                                      "transform-first second layer (layer widths or a route switch differ from the shipped "
                                      "configs)")
        topo1, e12, b1, slope1 = keep["rank1"]
        topo2, uv, wst, b2, slope2, _ = keep["tfirst"]
        if e12.shape[1] != 128 or uv.shape[1] != 64 or wst.shape != (64, 64):
            raise NotImplementedError("Knockout: the incremental trunk is written for layer widths 64 -> 32 (got %d -> %d)"
                                      % (e12.shape[1] // 2, uv.shape[1] // 2))
        pooled_cl = pooled.permute(0, 2, 3, 1)                 # [B, S, P, C], the pool kernel's own buffer
        if not pooled_cl.is_contiguous() or pooled_cl.shape[3] != 32:
            raise NotImplementedError("Knockout: the pool did not write the channel-last 32-channel tensor")
        w_pool = self.model.learnable_pca_params.detach() * self.model.info_mask.detach().reshape(-1, 1)
        self._base = dict(topo=topo1, e12=e12, b1=b1, slope1=slope1, uv=uv, wst=wst, b2=b2, slope2=slope2, pooled=pooled_cl,
                          w_pool=w_pool.float().contiguous())

    def _trunk(self):
        st, tb = self._base, self._tables
        topo = st["topo"]
        R = self.ROWS
        B, S, P, C = st["pooled"].shape
        out = torch.empty(R, S, P, C, dtype=torch.float32, device=self._xbase.device)
        L = _cabi.lib()
        with _cabi.span("knockout_trunk", 0):
            _cabi.check(L.mlg_knockout_trunk(
                _cabi.fptr(self.static_batch.x), _cabi.fptr(self._xbase), topo.n_single, B, _cabi.fptr(st["e12"]),
                st["e12"].stride(0), _cabi.fptr(st["b1"], True), st["slope1"], _cabi.fptr(st["wst"]),
                _cabi.fptr(st["b2"], True), _cabi.fptr(st["uv"]), st["slope2"], _cabi.iptr(topo.fwd.rowptr),
                _cabi.iptr(topo.fwd.col), _cabi.fptr(topo.fwd_val, True), _cabi.fptr(st["w_pool"]), _cabi.fptr(st["pooled"]),
                S, P, _cabi.iptr(tb["g_ptr"]), _cabi.iptr(tb["g_nodes"]), _cabi.iptr(tb["t1_ptr"]), _cabi.iptr(tb["t1_nodes"]),
                _cabi.iptr(tb["t2_ptr"]), _cabi.iptr(tb["t2_nodes"]), _cabi.iptr(tb["s_ptr"]), _cabi.iptr(tb["s_seg"]),
                _cabi.iptr(tb["e_ptr"]), _cabi.iptr(tb["e_slot"]), _cabi.iptr(tb["e_t2"]), _cabi.lptr(self._plan[0]),
                _cabi.lptr(self._plan[1]), R, tb["max_t1"], tb["max_t2"], _cabi.ptr(self._ws), self._ws.numel(),
                _cabi.fptr(out), _cabi.stream_ptr()), "mlg_knockout_trunk")
        return out

    def _chunk_body(self):
        """One replay: the incremental trunk for the ROWS rows of the static plan, the model's head on them, and per row
        pred[target] minus that of the patient's base row."""
        out = self._trunk()
        age = self.static_batch.age.index_select(0, self._plan[0])
        pred, _ = self.model.post_pool(out.permute(0, 3, 1, 2), age, require_grad=False)
        pt = pred[:, self.target]
        self.out_delta = pt - pt.index_select(0, self._plan[2])
        self.out_pred = pred

    # ---------------------------------------------------------------------------------------------------------------
    def _build_tables(self, dev):
        """Per (topology, groups): the group / T1 / T2 / pool-entry tables (host torch, once) and the trunk's workspace."""
        topo = self._base["topo"]
        n = topo.n_single
        key = (self.static_batch.topology_key.rsplit("-b", 1)[0], n)
        if self._tables is not None and self._tables["key"] == key:
            return
        ptr, nodes = parse_groups(self.groups, n)
        (t1p, t1n), (t2p, t2n) = neighbourhood_tables(ptr, nodes, topo.fwd.rowptr, topo.fwd.col, n)
        match = self.static_batch.gene_pca_match.reshape(self.batch_size, -1)[0]
        seg = self.static_batch.raw_indice.reshape(self.batch_size, -1)[0]
        S = self._base["pooled"].shape[1]
        s_ptr, s_seg, e_ptr, e_slot, e_t2 = slot_tables(t2p, t2n, match, seg, n, S)
        i32 = lambda t: t.to(torch.int32).to(dev)
        tb = dict(key=key, K=ptr.numel() - 1, g_ptr=i32(ptr), g_nodes=i32(nodes), t1_ptr=i32(t1p), t1_nodes=i32(t1n),
                  t2_ptr=i32(t2p), t2_nodes=i32(t2n), s_ptr=i32(s_ptr), s_seg=i32(s_seg), e_ptr=i32(e_ptr),
                  e_slot=i32(e_slot), e_t2=i32(e_t2),
                  max_t1=int((t1p[1:] - t1p[:-1]).max()), max_t2=int((t2p[1:] - t2p[:-1]).max()))
        for name in ("t1_nodes", "t2_nodes", "e_slot", "g_nodes"):     # the kernel indexes int32 tables with int32 offsets
            if tb[name].numel() >= 2 ** 31:
                raise ValueError("Knockout: the %s table exceeds 2^31 entries" % name)
        nbytes = int(_cabi.lib().mlg_knockout_workspace_bytes(self.ROWS, tb["max_t1"], tb["max_t2"]))
        self._ws = torch.empty(-(-nbytes // 16) * 16, dtype=torch.uint8, device=dev)
        self._tables = tb

    def capture(self, batch, warmup=2):
        """Record the two graphs over ``batch`` (a keyed device batch of ``batch_size`` graphs, as Evaluator.capture).  The
        per-group tables are built here, on the host, once per (topology, groups)."""
        B = int(batch.age.shape[0])
        if B != self.batch_size:
            raise ValueError("Knockout.capture: the batch holds %d graphs, batch_size is %d" % (B, self.batch_size))
        if getattr(batch, "topology_key", None) is None:
            raise ValueError("Knockout.capture: needs a keyed batch (data.collate / data.to_device)")
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
        self._xbase = (torch.zeros(n_nodes, dtype=torch.float32, device=dev) if self.baseline is None
                       else self.baseline.to(dev).reshape(n_nodes).clone())
        if self.model.reorder_idxs is not None and self.model.reorder_idxs.device != dev:
            # the head reorders the pathways with this index; a graph cannot copy it from pageable host memory on every replay
            self.model.reorder_idxs = self.model.reorder_idxs.to(dev)
        self._plan = torch.zeros(3, self.ROWS, dtype=torch.int64, device=dev)
        self._plan[1].fill_(-1)
        self._plan[2].copy_(torch.arange(self.ROWS, device=dev))
        with frozen_parameters(self.model, grad_enabled=False):
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                self._base_body()                       # builds the CSR / pool layout (host syncs) before any capture
                self._build_tables(dev)
                for _ in range(warmup):
                    self._base_body()
                    self._chunk_body()
            cur.wait_stream(side)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._base_body()
            self.graph_chunk = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_chunk, pool=self.graph.pool()):
                self._chunk_body()
        self._ptrs = self._param_ptrs()
        return self

    def eager(self):
        """One uncaptured pass of what the two replays run (base forward, then the chunk of the current static plan), on the
        static buffers; the outputs land in ``out_delta`` / ``out_pred`` as after a replay."""
        with frozen_parameters(self.model, grad_enabled=False):
            self._base_body()
            self._chunk_body()

    def _step_fields(self, host_batch):
        from .data import PER_SAMPLE_FIELDS
        return list(PER_SAMPLE_FIELDS)

    def _check_topology(self, host_batch):
        pass

    @staticmethod
    def _fill(dst, src):
        dst[:src.shape[0]].copy_(src, non_blocking=True)

    def screen(self, dataset, topo):
        """Knockout deltas for every record of ``dataset`` (records with x / y / age, as data.collate takes them; ``topo``
        the dataset's FoldTopology) -> KnockoutResult(delta [n, K], pred [n, 2]) of host tensors, in dataset order."""
        from .data import collate
        if self.graph is None:
            raise RuntimeError("Knockout: call capture(batch) first")
        want = "%s-b%d" % (topo.key, self.batch_size)
        if self.static_batch.topology_key != want:
            raise ValueError("Knockout: captured for topology_key=%r, this dataset's topology is %r"
                             % (self.static_batch.topology_key, want))
        if self._param_ptrs() != self._ptrs:
            self.capture(self._example)          # parameters were re-homed since capture: the graphs read stale storage
        n = len(dataset)
        if n == 0:
            raise ValueError("Knockout: empty dataset")
        B, R, K = self.batch_size, self.ROWS, self._tables["K"]
        dev = self._plan.device
        starts = list(range(0, n, B))
        plans, idx, per_batch = [], [], []
        for s in starts:
            ch = replay_plan(min(B, n - s), K, R)                                      # [chunks, R, 3]
            per_batch.append(ch.shape[0])
            p, k, base = ch[..., 0], ch[..., 1], ch[..., 2]
            real = p >= 0
            plans.append(torch.stack([torch.where(real, p, 0), k, base], 1))
            glob = p + s
            idx.append(torch.stack([torch.where(real & (k >= 0), glob * K + k, n * K), torch.where(real & (k < 0), glob, n)], 1))
        plan_dev = torch.cat(plans).pin_memory().to(dev, non_blocking=True)           # [chunks, 3, R]
        idx_dev = torch.cat(idx).pin_memory().to(dev, non_blocking=True)              # [chunks, 2, R]
        delta = torch.zeros(n * K + 1, dtype=torch.float32, device=dev)
        pred = torch.zeros(n + 1, 2, dtype=torch.float32, device=dev)

        def host(j):
            return collate([dataset[i] for i in range(starts[j], min(n, starts[j] + B))], topo)

        self.prefetch(host(0))
        c = 0
        for j in range(len(starts)):
            nxt = host(j + 1) if j + 1 < len(starts) else None      # collated on the host while the device works
            self._take_staged()
            self.graph.replay()
            if nxt is not None:
                self.prefetch(nxt)
            for _ in range(per_batch[j]):
                self._plan.copy_(plan_dev[c])
                self.graph_chunk.replay()
                delta.index_copy_(0, idx_dev[c, 0], self.out_delta)
                pred.index_copy_(0, idx_dev[c, 1], self.out_pred)
                c += 1
        host_delta, host_pred = delta.cpu(), pred.cpu()          # the one host synchronisation
        return KnockoutResult(host_delta[:n * K].view(n, K), host_pred[:n])
