"""CPU checks of PathwayShapley's host logic: the draws are a pure function (every pi_m a permutation, pair members reverses
of each other, pi depending on (seed, m) only, j on (seed, index, m) and in [0, M)); the player and window tables (gbm rows
144 / 145 and lgg column 8 in no window, the reorder mapping, lgg's "omic" players sharing windows, invalid player lists);
the constructor's validation; and a float64 restatement of the chain algorithm on the same tables against brute-force
``model.post_pool`` on every prefix grid of a few permutations, for a random head of each shipped shape."""
import pytest
import torch

import multilevel_gnn_b200 as mlg
from multilevel_gnn_b200 import shapley as S


def test_draws_are_a_pure_function():
    K, M, Sm = 146, 7, 12
    perm, j = S.shapley_draws(5, 3, Sm, M, K)
    assert perm.shape == (Sm, K) and j.shape == (Sm,)
    for row in perm:
        assert torch.equal(torch.sort(row).values, torch.arange(K))
    for m in range(Sm // 2):
        assert torch.equal(perm[2 * m + 1], perm[2 * m].flip(0))
        assert j[2 * m] == j[2 * m + 1]
    # pi depends on (seed, m) only: another patient, M, or a longer draw gives the same permutations
    for idx, MM, SS in ((0, 7, 12), (9, 3, 12), (3, 7, 20)):
        p2, j2 = S.shapley_draws(5, idx, SS, MM, K)
        assert torch.equal(p2[:Sm], perm)
        assert int(j2.min()) >= 0 and int(j2.max()) < MM
    assert not torch.equal(S.shapley_draws(6, 3, Sm, M, K)[0], perm)
    # j depends on (seed, index, m): repeat and call order, a longer draw extends a shorter one
    ref = [S.shapley_rows(5, i, 32, M) for i in range(10)]
    for i in (9, 0, 4):
        assert torch.equal(S.shapley_rows(5, i, 32, M), ref[i])
        assert torch.equal(S.shapley_rows(5, i, 8, M), ref[i][:8])
    assert len({tuple(r.tolist()) for r in ref}) == 10
    allj = torch.cat([S.shapley_rows(1, i, 64, M) for i in range(50)])
    assert set(allj.tolist()) == set(range(M))
    for bad in ((5, 0, 3, M, K), (5, 0, 0, M, K), (5, 0, 4, 0, K), (5, -1, 4, M, K)):
        with pytest.raises(ValueError):
            S.shapley_draws(*bad)
    ex = S.exact_perms(4)
    assert ex.shape == (24, 4) and len({tuple(r.tolist()) for r in ex}) == 24


def _cells_of_windows(ptr, idx, kh, kw, Wg):
    Wo = Wg // kw
    out = set()
    for w in idx.tolist():
        ho, wo = divmod(w, Wo)
        out.update((ho * kh + dh, wo * kw + dw) for dh in range(kh) for dw in range(kw))
    return out


def test_player_tables():
    # gbm: grid 146 x 6, (4, 2) pool -> rows 144, 145 in no window: pathways 144 / 145 have no window
    owner, ptr, idx = S.player_tables(S.parse_players("pathway"), 2, 4, 2)
    assert owner.shape == (146 * 6,) and ptr.shape == (147,)
    assert int(ptr[145]) == int(ptr[146]) == int(ptr[144])
    assert all(int(ptr[p + 1] - ptr[p]) == 3 for p in range(144))
    assert int(idx.max()) < 36 * 3
    # lgg: grid 146 x 9, (4, 2) pool -> column 8 is in no window; "omic" players share the window of columns 2-3 and 4-5
    owner, ptr, idx = S.player_tables(S.parse_players("omic"), 3, 4, 2)
    wins = [set(idx[ptr[k]:ptr[k + 1]].tolist()) for k in range(3)]
    assert [len(w) for w in wins] == [72, 72, 36]
    assert all(w % 4 in (0, 1) for w in wins[0]) and all(w % 4 in (1, 2) for w in wins[1])
    assert all(w % 4 == 3 for w in wins[2])
    assert len(wins[0] & wins[1]) == 36 and not (wins[0] & wins[2]) and not (wins[1] & wins[2])
    cov = _cells_of_windows(ptr, torch.arange(36 * 4), 4, 2, 9)
    assert all((r, 8) not in cov for r in range(146)) and all((144, c) not in cov for c in range(9))
    assert owner.view(146, 9)[:, 8].eq(2).all()
    # with reorder_pathway, segment 3p + o sits at the row q with reorder[q] == p
    g = torch.Generator().manual_seed(0)
    reorder = torch.randperm(146, generator=g)
    owner, ptr, idx = S.player_tables(S.parse_players("segment"), 3, 1, 1, reorder)
    grid = owner.view(146, 9)
    for p in (0, 17, 145):
        q = int((reorder == p).nonzero())
        for o in range(3):
            assert grid[q, 3 * o:3 * o + 3].eq(3 * p + o).all()
            k = 3 * p + o
            assert idx[ptr[k]:ptr[k + 1]].tolist() == [q * 9 + 3 * o + c for c in range(3)]
    # a partial player list: segments in no player are owned by nobody
    owner, ptr, idx = S.player_tables(S.parse_players([[0, 1], [5]]), 2, 4, 2)
    assert int((owner >= 0).sum()) == 3 * 2 and ptr.tolist() == [0, 2, 3]


def test_bad_players_raise():
    for bad in ([[0, 1], [1, 2]], [[0, 438]], [[-1]], [], [[0], []], [[0.5]]):
        with pytest.raises(ValueError):
            S.parse_players(bad)
    with pytest.raises(ValueError):
        S.parse_players("gene")


@pytest.fixture(scope="module")
def gbm():
    args = mlg.configs.make_args("gbm")
    torch.manual_seed(0)
    return mlg.MultilevelGNN(args), args


def test_constructor_validation(gbm):
    model, args = gbm
    N = 3 * model.node_num
    bg = torch.zeros(3, N)
    S.PathwayShapley(model, args, bg)
    for kw in (dict(target=2), dict(background=torch.zeros(3, N - 1)), dict(background=torch.zeros(0, N)),
               dict(background=torch.full((2, N), float("nan"))), dict(samples=3), dict(samples=0), dict(samples="all"),
               dict(samples="exact"), dict(players="segment", samples="exact"), dict(players=[[0], [0]]),
               dict(batch_size=1)):
        args_kw = dict(background=bg)
        args_kw.update(kw)
        with pytest.raises(ValueError):
            S.PathwayShapley(model, args, **args_kw)
    S.PathwayShapley(model, args, bg, players="omic", samples="exact")
    S.PathwayShapley(model, args, bg, players=[[s] for s in range(8)], samples="exact")
    h = model.head[1].register_forward_hook(lambda *a: None)
    try:
        with pytest.raises(NotImplementedError):
            S.PathwayShapley(model, args, bg)
    finally:
        h.remove()
    args2 = mlg.configs.make_args("gbm", head_dim=100)
    with pytest.raises(NotImplementedError):
        S.PathwayShapley(mlg.MultilevelGNN(args2), args2, bg)


def _pre_reorder(grid, model, args):
    """Head-input grids [R, 32, 146, 3P] -> the pooled tensor [R, 32, 438, P] that post_pool reorders into them."""
    if args.reorder_pathway and model.reorder_idxs is not None:
        grid = grid[:, :, S.segment_row(model.reorder_idxs)]
    return grid.reshape(grid.shape[0], 32, 438, model.pca_dim)


def _restated_chain(model, args, x, bgr, age, perm, tables, kh, kw, target):
    """Float64 restatement of mlg_shap_chains for one chain: p after every prefix of ``perm`` (K + 1 values)."""
    cm, hd = model.conv_model, model.head
    Hg, Wg = x.shape[1], x.shape[2]
    Ho, Wo = Hg // kh, Wg // kw

    def cells(g):
        z = g.double().permute(1, 2, 0).reshape(-1, 32)
        z = torch.relu(z @ cm[0].weight.double().view(32, 32).T + cm[0].bias.double())
        return torch.relu(z @ cm[2].weight.double().view(64, 32).T + cm[2].bias.double())     # [cells, 64]

    cp, cb = cells(x), cells(bgr)
    owner, ptr, idx = tables
    W1 = hd[0].weight.double()
    H = W1.shape[0]
    w1p = W1[:, :64 * Ho * Wo].reshape(H, 64, Ho * Wo).permute(2, 1, 0)
    coal = set()

    def a0(w, extra=None):
        ho, wo = divmod(w, Wo)
        best = torch.zeros(64, dtype=torch.float64)
        for dh in range(kh):
            for dw in range(kw):
                c = (ho * kh + dh) * Wg + wo * kw + dw
                o = int(owner[c])
                src = cp if (o < 0 or o in coal or o == extra) else cb
                best = torch.maximum(best, src[c])
        return best

    h = hd[0].bias.double().clone()
    if args.use_age:
        h += W1[:, 64 * Ho * Wo] * age
    for w in range(Ho * Wo):
        h += w1p[w].T @ a0(w)
    d3 = hd[3].weight.double()[target] - hd[3].weight.double()[1 - target]
    db = hd[3].bias.double()[target] - hd[3].bias.double()[1 - target]
    prob = lambda: float(torch.sigmoid(d3 @ torch.relu(h) + db))
    out = [prob()]
    for k in perm.tolist():
        for w in idx[ptr[k]:ptr[k + 1]].tolist():
            h += w1p[w].T @ (a0(w, extra=k) - a0(w))
        coal.add(k)
        out.append(prob())
    return torch.tensor(out, dtype=torch.float64)


@pytest.mark.parametrize("cfg,players", [("gbm", "pathway"), ("kirc", "pathway"), ("lgg", "omic"), ("lgg", "segment")])
def test_restated_chain_matches_post_pool(cfg, players):
    args = mlg.configs.make_args(cfg)
    torch.manual_seed(3)
    model = mlg.MultilevelGNN(args)
    if args.reorder_pathway:
        model.set_reorder_idxs(torch.randperm(146, generator=torch.Generator().manual_seed(3)).tolist())
    model.eval()
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        for lin in (model.head[0], model.head[3]):
            lin.bias.normal_(0, 0.3, generator=g)
    kh, kw, Ho, Wo, H = S.head_geometry(model)
    Wg = 3 * model.pca_dim
    groups = S.parse_players(players)
    reorder = model.reorder_idxs if args.reorder_pathway else None
    tables = S.player_tables(groups, model.pca_dim, kh, kw, reorder)
    owner = tables[0].view(146, Wg)
    x = torch.randn(32, 146, Wg, generator=g) * 2
    bgr = torch.randn(32, 146, Wg, generator=g) * 2
    age = 0.7
    for m, target in ((0, 1), (1, 0)):
        perm = S.shapley_perms(9, 2, len(groups))[m]
        with torch.no_grad():
            got = _restated_chain(model, args, x, bgr, age, perm, tables, kh, kw, target)
        rank = torch.empty(len(groups), dtype=torch.int64)
        rank[perm] = torch.arange(len(groups))
        prefix = torch.arange(len(groups) + 1).view(-1, 1, 1)
        own_rank = torch.where(owner >= 0, rank[owner.clamp(min=0).long()], torch.full_like(owner, -1, dtype=torch.int64))
        from_pat = own_rank.unsqueeze(0) < prefix                                                    # [K + 1, 146, Wg]
        grids = torch.where(from_pat.unsqueeze(1), x.unsqueeze(0), bgr.unsqueeze(0))
        with torch.no_grad():
            pred, _ = model.post_pool(_pre_reorder(grids, model, args), torch.full((grids.shape[0],), age), require_grad=False)
        ref = pred[:, target].double()
        assert (got - ref).abs().max().item() < 2e-6, (cfg, players, (got - ref).abs().max().item())
        assert float((got[1:] != got[:-1]).double().mean()) > 0.5      # the players do move the prediction
