"""Batch construction for the hot path: the replacement of torch_geometric's ``DataLoader`` / ``Batch`` collate as the
reference uses it (train.py:17,316-327 over ``MyData.__getitem__``, dataloader/multiloader.py:76-94).

What the reference does per step: every patient ``Data`` carries its own copy of the SAME edge list, edge weights and
pooling tables (one gene network per fold, multiloader.py:687-698); PyG's collate concatenates B copies (adding node
offsets to ``edge_index``) and ``batch.to(device)`` uploads all of it -- 78 MB per step at the gbm shape, of which only
2 MB (node values, labels, age) differ between steps.

Here the fold-constant part is a ``FoldTopology`` (single-graph edge list + pooling tables + a content key); ``collate``
stacks only the per-patient fields into pinned host memory and attaches the B-fold replicated topology -- built ONCE per
(topology, batch size) and shared by every batch, on the host and, after the first upload, on the device -- together with
``topology_key``.  ``MultilevelGNN.forward`` caches its CSR / pool layout under that key (graph.topology /
graph.pool_layout ``static_key``) and ``Trainer.load_batch`` / ``prefetch`` copy only the per-step fields of a keyed
batch (and refuse a batch whose key differs from the captured graph's).  ``TopologyLoader`` iterates an epoch the way
train.py:322-323 does (shuffle, drop_last) with the data-parallel split of ``train.shard_indices``.
"""
import hashlib

import torch

from .synth import GraphBatch
from .train import shard_indices


class FoldTopology:
    """The fold-constant inputs of MultilevelGNN.forward: ONE patient's edge list (``edge_index`` [2, E] with node ids in
    [0, n_nodes), ``edge_attr`` [E, 1]) and the pooling tables ``gene_pca_match`` [G], ``raw_indice`` [G].  ``key`` is a
    content hash, so two folds with different gene selections can never share cached CSR / pool layouts."""

    def __init__(self, edge_index, edge_attr, gene_pca_match, raw_indice, n_nodes):
        self.edge_index = edge_index.to(torch.int64).contiguous()
        self.edge_attr = edge_attr.to(torch.float32).reshape(-1, 1).contiguous()
        self.gene_pca_match = gene_pca_match.to(torch.int64).reshape(-1).contiguous()
        self.raw_indice = raw_indice.to(torch.int64).reshape(-1).contiguous()
        self.n_nodes = int(n_nodes)
        if self.edge_index.numel() and (int(self.edge_index.min()) < 0 or int(self.edge_index.max()) >= self.n_nodes):
            raise ValueError("FoldTopology: edge_index must address nodes of ONE graph (0 <= id < n_nodes)")
        h = hashlib.sha1()
        for t in (self.edge_index, self.edge_attr, self.gene_pca_match, self.raw_indice):
            h.update(t.numpy().tobytes())
        h.update(str(self.n_nodes).encode())
        self.key = "topo-" + h.hexdigest()[:16]
        self._host, self._device = {}, {}

    @classmethod
    def from_sample(cls, data, n_nodes=None):
        """From one ``Data`` record of the reference's dataset (all records of a fold carry the same copies)."""
        n = int(data.x.shape[0]) if n_nodes is None else n_nodes
        return cls(data.edge_index, data.edge_attr, data.gene_pca_match.reshape(-1), data.raw_indice.reshape(-1), n)

    def replicated(self, batch_size, pin=True):
        """The B-fold fields exactly as PyG's collate lays them out: edge_index [2, B*E] with cumulative node offsets
        (graph-major), edge_attr [B*E, 1], gene_pca_match / raw_indice [B, G], batch [B*N].  Built once per batch size."""
        got = self._host.get(batch_size)
        if got is None:
            off = (torch.arange(batch_size) * self.n_nodes).view(-1, 1, 1)
            got = dict(
                edge_index=(self.edge_index.unsqueeze(0) + off).permute(1, 0, 2).reshape(2, -1).contiguous(),
                edge_attr=self.edge_attr.repeat(batch_size, 1),
                gene_pca_match=self.gene_pca_match.unsqueeze(0).repeat(batch_size, 1),
                raw_indice=self.raw_indice.unsqueeze(0).repeat(batch_size, 1),
                batch=torch.arange(batch_size).repeat_interleave(self.n_nodes))
            if pin and torch.cuda.is_available():
                got = {k: v.pin_memory() for k, v in got.items()}
            self._host[batch_size] = got
        return got

    def on_device(self, batch_size, device):
        """The replicated fields resident on ``device`` (uploaded once per batch size)."""
        k = (batch_size, str(device))
        if k not in self._device:
            self._device[k] = {n: v.to(device, non_blocking=True) for n, v in self.replicated(batch_size).items()}
        return self._device[k]


PER_SAMPLE_FIELDS = ("x", "y", "age")


def collate(samples, topo, pin=True):
    """List of per-patient records (attributes ``x`` [N] or [N, 1], ``y`` [2], ``age`` float or 0-d tensor) -> one
    GraphBatch with the layout of PyG's ``Batch`` (x [B*N, 1], y [2B], age [B] + the replicated topology) carrying
    ``topology_key``.  Only x / y / age are freshly allocated; the topology tensors are the shared per-batch-size ones."""
    B = len(samples)
    if B == 0:
        raise ValueError("collate: empty batch")
    x = torch.stack([torch.as_tensor(s.x, dtype=torch.float32).reshape(-1) for s in samples])
    if x.shape[1] != topo.n_nodes:
        raise ValueError("collate: a sample has %d nodes, the topology %d" % (x.shape[1], topo.n_nodes))
    fields = dict(x=x.reshape(-1, 1),
                  age=torch.stack([torch.as_tensor(s.age, dtype=torch.float32).reshape(()) for s in samples]))
    if all(getattr(s, "y", None) is not None for s in samples):
        fields["y"] = torch.cat([torch.as_tensor(s.y, dtype=torch.float32).reshape(-1) for s in samples])
    if pin and torch.cuda.is_available():
        fields = {k: v.pin_memory() for k, v in fields.items()}
    fields.update(topo.replicated(B, pin=pin))
    b = GraphBatch(**fields)
    b.topology_key = "%s-b%d" % (topo.key, B)
    return b


def to_device(batch, topo, device):
    """Upload a collated batch: per-step fields are copied, the topology fields are the device-resident shared ones."""
    B = batch.age.shape[0]
    out = GraphBatch(**{k: getattr(batch, k).to(device, non_blocking=True) for k in PER_SAMPLE_FIELDS if hasattr(batch, k)})
    for k, v in topo.on_device(B, device).items():
        setattr(out, k, v)
    out.topology_key = batch.topology_key
    return out


class TopologyLoader:
    """for batch in TopologyLoader(dataset, topo, batch_size=32, rank=r, world=w): ...  -- one epoch of keyed, pinned
    batches; ``set_epoch`` reshuffles (same permutation on every rank, disjoint slices per rank, drop_last like
    train.py:322-323)."""

    def __init__(self, dataset, topo, batch_size, shuffle=True, drop_last=True, rank=0, world=1, seed=0, pin=True):
        self.dataset, self.topo, self.batch_size = dataset, topo, batch_size
        self.shuffle, self.drop_last, self.rank, self.world, self.seed, self.pin = shuffle, drop_last, rank, world, seed, pin
        self.epoch = 0

    def set_epoch(self, epoch):
        self.epoch = epoch

    def index_batches(self):
        """The epoch's index tensors, one per batch of this rank.  Unshuffled without drop_last (evaluation): step s takes rows
        [s*B*world + rank*B, ... + B) clipped to the dataset -- a tail batch may be short, a rank's last one empty, and every
        rank has the same number of steps.  ``__iter__`` skips the empty ones."""
        n = len(self.dataset)
        if self.shuffle:
            return shard_indices(n, self.rank, self.world, self.batch_size, epoch_seed=self.seed + self.epoch,
                                 drop_last=self.drop_last)
        step = self.batch_size * self.world
        n_steps = n // step if self.drop_last else -(-n // step)
        idx = torch.arange(n)
        return [idx[s * step + self.rank * self.batch_size: s * step + (self.rank + 1) * self.batch_size]
                for s in range(n_steps)]

    def __len__(self):
        return len(self.index_batches())

    def __iter__(self):
        for idx in self.index_batches():
            if idx.numel() == 0:
                continue
            yield collate([self.dataset[int(i)] for i in idx], self.topo, pin=self.pin)
