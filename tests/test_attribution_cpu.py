"""CPU checks of the Attributor's host logic: interpolation points and trapezoid weights, the packing of patients and
interpolants into replays (tails and multi-replay patients included), and the node -> (gene, omic) and pooled ->
(pathway, omic) reductions with the model's pathway reordering undone, each against a direct torch expression."""
import pytest
import torch

from multilevel_gnn_b200 import attribution as A


def test_alphas_and_trapezoid_weights():
    for m in (2, 3, 8, 64):
        al, w = A.ig_alphas(m), A.trapezoid_weights(m)
        assert al[0] == 0 and al[-1] == 1 and torch.allclose(al, torch.linspace(0, 1, m, dtype=torch.float64))
        assert torch.allclose(w.sum(), torch.tensor(1.0, dtype=torch.float64))
        f = torch.sin(3 * al) + al ** 2                     # the rule against torch.trapezoid on the same grid
        assert torch.allclose((w * f).sum(), torch.trapezoid(f, al))
    with pytest.raises(ValueError):
        A.ig_alphas(1)


@pytest.mark.parametrize("n,B,m", [(1, 32, 1), (45, 32, 1), (5, 32, 8), (11, 8, 4), (3, 32, 64), (2, 16, 40), (7, 5, 5)])
def test_slot_plan(n, B, m):
    plan = A.slot_plan(n, B, m)
    seen = torch.cat(plan)
    want = torch.stack([torch.arange(n).repeat_interleave(m), torch.arange(m).repeat(n)], 1)
    assert torch.equal(seen, want)                                          # every (patient, k) once, in order
    assert all(1 <= p.shape[0] <= B for p in plan)
    if m <= B:
        per = B // m
        assert len(plan) == -(-n // per)
        assert all(p.shape[0] == per * m for p in plan[:-1])                # only the last replay is a tail
        assert all(torch.equal(p[:, 1], torch.arange(m).repeat(p.shape[0] // m)) for p in plan)
    else:
        assert len(plan) == n * -(-m // B)
        assert all(p[:, 0].unique().numel() == 1 for p in plan)             # a replay holds one patient's interpolants


def test_gene_view():
    nodes = torch.randn(4, 3 * 5135)
    g = A.gene_view(nodes)
    for gene in (0, 17, 5134):
        for omic in range(3):
            assert torch.equal(g[:, gene, omic], nodes[:, 3 * gene + omic])


@pytest.mark.parametrize("P", [2, 3])
@pytest.mark.parametrize("reorder", [False, True])
def test_pathway_reduce(P, reorder):
    g = torch.Generator().manual_seed(P)
    B, C = 3, 32
    contrib = torch.randn(B, C, 146, 3 * P, generator=g, dtype=torch.float64)
    idx = torch.randperm(146, generator=g) if reorder else None
    got = A.pathway_reduce(contrib, P, idx)
    want = torch.zeros(B, 146, 3, dtype=torch.float64)
    for r in range(146):
        src = r if idx is None else int((idx == r).nonzero())              # position of pathway r in the reordered axis
        for o in range(3):
            want[:, r, o] = contrib[:, :, src, o * P:(o + 1) * P].sum((1, 2))
    assert torch.allclose(got, want)
