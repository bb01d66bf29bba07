"""CPU checks of expected gradients' host logic: the draws are a pure function of (seed, patient index, S, M) with alpha in
(0, 1) exact in fp32 and j covering [0, M); the sample pass holds S weighted slots per patient (and S zero-weight alpha = 0
slots with completeness) on top of slot_plan; the constructor validates background / samples / method."""
import pytest
import torch

import multilevel_gnn_b200 as mlg
from multilevel_gnn_b200 import attribution as A


@pytest.fixture(scope="module")
def model():
    args = mlg.configs.make_args("gbm")
    return mlg.MultilevelGNN(args), args


def test_draws_are_a_pure_function():
    S, M = 16, 7
    ref = [A.eg_draws(3, i, S, M) for i in range(12)]
    for i in (11, 0, 5):                                                  # call order and repeats
        j, al = A.eg_draws(3, i, S, M)
        assert torch.equal(j, ref[i][0]) and torch.equal(al, ref[i][1])
    # what a dataset of any length draws for its first patients (the plan takes eg_draws per index, nothing else)
    for n in (1, 6, 12):
        for B, comp in ((8, False), (32, True), (5, True)):
            J = torch.stack([A.eg_draws(3, i, S, M)[0] for i in range(n)])
            Al = torch.stack([A.eg_draws(3, i, S, M)[1] for i in range(n)])
            got = {}
            for slots, j, al, w, pos in A.eg_plan(J, Al, B, comp):
                for r in range(slots.shape[0]):
                    p, k = int(slots[r, 0]), int(slots[r, 1])
                    if k < S:
                        got[(p, k)] = (int(j[r]), float(al[r]))
            for p in range(n):
                for k in range(S):
                    assert got[(p, k)] == (int(ref[p][0][k]), float(ref[p][1][k])), (n, B, comp, p, k)
    # a longer draw extends a shorter one; another seed or index draws differently
    j32, al32 = A.eg_draws(3, 4, 32, M)
    assert torch.equal(j32[:S], ref[4][0]) and torch.equal(al32[:S], ref[4][1])
    assert not torch.equal(A.eg_draws(4, 4, S, M)[1], ref[4][1])
    assert not torch.equal(ref[5][1], ref[4][1])


def test_draw_ranges():
    M = 13
    J, Al = zip(*(A.eg_draws(11, i, 256, M) for i in range(8)))
    J, Al = torch.cat(J), torch.cat(Al)
    assert J.dtype == torch.int64 and int(J.min()) >= 0 and int(J.max()) < M
    assert torch.equal(torch.unique(J), torch.arange(M))                  # covers all of [0, M) at large S
    assert bool((Al > 0).all()) and bool((Al < 1).all())
    assert torch.equal(Al.float().double(), Al)                           # exact in fp32
    assert abs(float(Al.mean()) - 0.5) < 0.03
    j1, al1 = A.eg_draws(0, 0, 4, 1)
    assert torch.equal(j1, torch.zeros(4, dtype=torch.int64))
    with pytest.raises(ValueError):
        A.eg_draws(0, 0, 0, 3)
    with pytest.raises(ValueError):
        A.eg_draws(0, 0, 3, 0)


@pytest.mark.parametrize("n,B,S,comp", [(5, 32, 4, False), (5, 32, 4, True), (7, 8, 3, True), (3, 8, 12, True),
                                        (2, 5, 5, False), (4, 1, 2, True)])
def test_sample_plan(n, B, S, comp):
    J = torch.stack([A.eg_draws(1, i, S, 9)[0] for i in range(n)])
    Al = torch.stack([A.eg_draws(1, i, S, 9)[1] for i in range(n)])
    rows = A.eg_plan(J, Al, B, comp)
    per = 2 * S if comp else S
    want = A.slot_plan(n, B, per)
    assert len(rows) == len(want)
    wsum = torch.zeros(n, dtype=torch.float64)
    kept = []
    for (slots, j, al, w, pos), ws in zip(rows, want):
        assert torch.equal(slots, ws) and slots.shape[0] <= B
        p, k = slots[:, 0], slots[:, 1]
        sample = k < S
        assert torch.equal(j, J[p, k % S])
        assert torch.equal(al[sample], Al[p, k % S][sample]) and bool((al[~sample] == 0).all())
        assert bool((w[sample] == 1.0 / S).all()) and bool((w[~sample] == 0).all())
        assert bool((pos[sample] == -1).all()) and torch.equal(pos[~sample], p[~sample] * S + k[~sample] - S)
        wsum.index_add_(0, p, w)
        kept.append(pos[~sample])
    assert torch.allclose(wsum, torch.ones(n, dtype=torch.float64))       # weights sum to 1 per patient
    kept = torch.cat(kept)
    if comp:                                                              # S alpha = 0 slots per patient, each kept once
        assert torch.equal(kept.sort().values, torch.arange(n * S))
    else:
        assert kept.numel() == 0
    one = A.slot_plan(n, B, 1)                                            # the alpha = 1 pass: each patient once
    assert torch.equal(torch.cat(one)[:, 0], torch.arange(n)) and all(r.shape[0] <= B for r in one)


def test_constructor_validation(model):
    m, args = model
    N = 3 * mlg.MultilevelGNN.GENES
    bg = torch.randn(4, N)
    at = mlg.Attributor(m, args, method="expected_gradients", background=bg, samples=3, seed=5, completeness=True)
    assert at.background.shape == (4, N) and at.samples == 3 and at.seed == 5 and at.completeness
    assert torch.equal(at.background, bg) and at.background.data_ptr() != bg.data_ptr()      # a copy
    bad = [dict(background=None),                                         # missing
           dict(background=torch.randn(N)),                               # not [M, N]
           dict(background=torch.randn(0, N)),                            # M = 0
           dict(background=torch.randn(3, N - 3)),                        # N does not match
           dict(background=torch.full((2, N), float("nan"))),             # not finite
           dict(background=bg.clone().index_fill_(1, torch.tensor([17]), float("inf"))),
           dict(background=bg, samples=0),
           dict(background=bg, baseline=torch.zeros(N))]
    for kw in bad:
        with pytest.raises(ValueError):
            mlg.Attributor(m, args, method="expected_gradients", **kw)
    for method in ("saliency", "input_x_gradient", "integrated_gradients"):
        with pytest.raises(ValueError):
            mlg.Attributor(m, args, method=method, background=bg)
        mlg.Attributor(m, args, method=method)                            # the other methods are unchanged
    with pytest.raises(ValueError):
        mlg.Attributor(m, args, method="shap")
