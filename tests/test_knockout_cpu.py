"""Host-side parts of the knockout screen (multilevel_gnn_b200.knockout), no GPU needed:

* the per-group neighbourhood tables T1 / T2 against a dense breadth-first reach on small random graphs with self loops,
  a hub and a node that no row reads;
* the pool-entry tables (touched segments, entries in slot order, missing slots left out) against a direct enumeration;
* group parsing and validation;
* the replay plan: one base row per patient present, groups spanning several chunks, the tail chunk.

The incremental trunk itself and the screen are checked on the GPU (tests/test_gpu_knockout.py)."""
import pytest
import torch

from multilevel_gnn_b200 import knockout as K


def _random_csr(n, n_edges, hub, seed):
    """Forward CSR (row i lists the nodes it reads, self loop included), as graph.Topology builds it with self_loops=True:
    random edges, node ``hub`` read by ~half of the rows, node n - 1 read by no row but its own."""
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n - 1, (n_edges,), generator=g)
    dst = torch.randint(0, n, (n_edges,), generator=g)
    hub_dst = torch.nonzero(torch.rand(n, generator=g) < 0.5).flatten()
    src = torch.cat([src, torch.full_like(hub_dst, hub)])
    dst = torch.cat([dst, hub_dst])
    keep = src != dst
    src, dst = src[keep], dst[keep]
    src = torch.cat([src, torch.arange(n)])
    dst = torch.cat([dst, torch.arange(n)])
    order = torch.argsort(dst * n + src, stable=True)
    src, dst = src[order], dst[order]
    rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), torch.bincount(dst, minlength=n).cumsum(0)])
    return rowptr.to(torch.int32), src.to(torch.int32)


def _dense_reach(rowptr, col, n, group):
    A = torch.zeros(n, n, dtype=torch.bool)
    for i in range(n):
        A[i, col[rowptr[i]:rowptr[i + 1]].long()] = True
    t0 = torch.zeros(n, dtype=torch.bool)
    t0[list(group)] = True
    t1 = t0 | (A & t0.view(1, n)).any(1)
    t2 = t1 | (A & t1.view(1, n)).any(1)
    return torch.nonzero(t1).flatten(), torch.nonzero(t2).flatten()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_neighbourhood_tables_vs_dense_reach(seed):
    n = 60
    rowptr, col = _random_csr(n, 150, hub=7, seed=seed)
    groups = [[3], [7], [n - 1], [0, 1, 2], [], [7, 20, 40], list(range(0, n, 5))]
    ptr, nodes = K.parse_groups(groups, n)
    (t1p, t1n), (t2p, t2n) = K.neighbourhood_tables(ptr, nodes, rowptr, col, n)
    for k, g in enumerate(groups):
        r1, r2 = _dense_reach(rowptr, col, n, g)
        assert torch.equal(t1n[t1p[k]:t1p[k + 1]], r1), (k, g)
        assert torch.equal(t2n[t2p[k]:t2p[k + 1]], r2), (k, g)
    assert t1p[2 + 1] - t1p[2] == 1                      # a node no other row reads reaches only itself
    assert t1p[1 + 1] - t1p[1] > n // 3                  # the hub reaches about half of the rows
    assert t1p[4] == t1p[5] and t2p[4] == t2p[5]         # an empty group reaches nothing


def test_slot_tables_vs_enumeration():
    n, G, S = 40, 90, 7
    g = torch.Generator().manual_seed(3)
    rowptr, col = _random_csr(n, 80, hub=5, seed=3)
    match = torch.randint(0, n, (G,), generator=g)
    match[torch.rand(G, generator=g) < 0.1] = -1
    seg = torch.sort(torch.randint(0, S, (G,), generator=g)).values
    groups = [[5], [0, 1, 2], [], [39]]
    ptr, nodes = K.parse_groups(groups, n)
    _, (t2p, t2n) = K.neighbourhood_tables(ptr, nodes, rowptr, col, n)
    s_ptr, s_seg, e_ptr, e_slot, e_t2 = K.slot_tables(t2p, t2n, match, seg, n, S)
    for k in range(len(groups)):
        t2 = t2n[t2p[k]:t2p[k + 1]].tolist()
        want = {}
        for q in range(G):
            if int(match[q]) in t2:
                want.setdefault(int(seg[q]), []).append((q, t2.index(int(match[q]))))
        segs = s_seg[s_ptr[k]:s_ptr[k + 1]].tolist()
        assert segs == sorted(want), k
        for j, s in enumerate(segs):
            e = slice(int(e_ptr[s_ptr[k] + j]), int(e_ptr[s_ptr[k] + j + 1]))
            assert list(zip(e_slot[e].tolist(), e_t2[e].tolist())) == want[s], (k, s)
    assert int(s_ptr[3] - s_ptr[2]) == 0


def test_parse_groups():
    ptr, nodes = K.parse_groups("gene", 12)
    assert ptr.tolist() == [0, 3, 6, 9, 12] and torch.equal(nodes, torch.arange(12))
    ptr, nodes = K.parse_groups("node", 5)
    assert ptr.tolist() == [0, 1, 2, 3, 4, 5]
    ptr, nodes = K.parse_groups([[4, 1, 4], [], torch.tensor([0])], 5)
    assert ptr.tolist() == [0, 2, 2, 3] and nodes.tolist() == [1, 4, 0]
    for bad in ([[5]], [[-1]], [[0.5]], [[True]]):
        with pytest.raises(ValueError):
            K.parse_groups(bad, 5)
    for bad in ("genes", []):
        with pytest.raises(ValueError):
            K.parse_groups(bad, 6)
    with pytest.raises(ValueError):
        K.parse_groups("gene", 10)


@pytest.mark.parametrize("n,k,rows", [(3, 5135, 64), (5, 10, 64), (4, 63, 64), (3, 62, 64), (2, 1, 2), (7, 3, 8), (1, 200, 128)])
def test_replay_plan(n, k, rows):
    chunks = K.replay_plan(n, k, rows)
    seen = []
    for ch in chunks:
        assert ch.shape == (rows, 3)
        real = ch[:, 0] >= 0
        m = int(real.sum())
        assert bool(real[:m].all()) and not bool(real[m:].any())      # filled from the first row, padding after
        pats = ch[:m, 0].unique().tolist()
        for p in pats:
            rows_p = torch.nonzero(ch[:m, 0] == p).flatten()
            base = rows_p[ch[rows_p, 1] < 0]
            assert base.numel() == 1 and int(base[0]) == int(rows_p[0])      # one base row, first of the patient's rows
            assert bool((ch[rows_p, 2] == base[0]).all())
        for r in range(m):
            if ch[r, 1] >= 0:
                seen.append((int(ch[r, 0]), int(ch[r, 1])))
        assert bool((ch[m:, 2] == torch.arange(m, rows)).all())              # padding rows are their own base
    assert seen == [(p, g) for p in range(n) for g in range(k)]
    if k >= rows:
        assert len(chunks) >= n * k // (rows - 1)


def test_replay_plan_rejects():
    for args in ((0, 1, 4), (1, 0, 4), (1, 1, 1)):
        with pytest.raises(ValueError):
            K.replay_plan(*args)


def test_knockout_rejects_unsupported_routes():
    import multilevel_gnn_b200 as m
    for overrides in (dict(gnn_name="rsage"), dict(resgnn=True), dict(dense_gnn=True), dict(repeat_mask=True),
                      dict(merge_mode="add"), dict(num_layers=3), dict(pca_match_mask=False)):
        args = m.configs.make_args("gbm", **overrides)
        model = m.MultilevelGNN(args)
        with pytest.raises(NotImplementedError):
            K.Knockout(model, args)
    args = m.configs.make_args("gbm")
    model = m.MultilevelGNN(args)
    h = model.gnn_model[1].register_forward_hook(lambda *a: None)
    with pytest.raises(NotImplementedError):
        K.Knockout(model, args)
    h.remove()
    K.Knockout(model, args)
    for bad in (dict(batch_size=1), dict(target=2)):
        with pytest.raises(ValueError):
            K.Knockout(model, args, **bad)
