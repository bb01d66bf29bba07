"""The fused data-parallel update (reduce-scatter -> Adam -> all-gather over peer memory, csrc/peer_adam.cu) against
torch.optim.Adam on the averaged gradient.  One GPU is enough to exercise the whole protocol: the ranks' arenas all live on
this device and ONE cooperative launch steps all of them (mlg_peer_adam_step_emulated: blockIdx.y = rank), so the blocks that
wait on one another's system-scope flags are guaranteed to be co-resident.  (Separate launches per rank on one GPU are not --
/opt/skills/guides/B200_PROFILING.md -- and the real multi-process path is bench.py --gpus N / tools/peer_check.py.)"""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


@pytest.fixture(scope="module")
def mlg():
    import multilevel_gnn_b200 as m
    m._cabi.lib()
    return m


def _virtual_ranks(mlg, shapes, world, seed, wd):
    from multilevel_gnn_b200.train import GradBucket, PeerAdam, PeerArena
    g = torch.Generator().manual_seed(seed)
    init = [torch.randn(s, generator=g) for s in shapes]
    align = 4 * world
    ranks = []
    for r in range(world):
        params = [torch.nn.Parameter(t.clone().to(DEV)) for t in init]
        arena = PeerArena(GradBucket.padded_size(params, align), world, r, DEV, exchange=False)
        ranks.append([params, arena])
    for params, arena in ranks:
        arena.peer_base = [a.base for _, a in ranks]
    out = []
    for params, arena in ranks:
        bucket = GradBucket(params, flat=arena.grad, align=align)
        opt = PeerAdam(bucket, arena, lr=1e-2, betas=(0.9, 0.999), weight_decay=wd, timeout_s=2.0)
        out.append((params, bucket, opt))
    return init, out, g


def _step_all(mlg, ranks, scratch):
    """All ranks' update kernels as one cooperative launch."""
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()
    opt0 = ranks[0][2]
    world = len(ranks)
    g, p, f = opt0.arena.pointer_tables()
    arr = ctypes.c_void_p * world
    m = arr(*[o.exp_avg.data_ptr() for _, _, o in ranks])
    v = arr(*[o.exp_avg_sq.data_ptr() for _, _, o in ranks])
    t = arr(*[o.step_dev.data_ptr() for _, _, o in ranks])
    _cabi.check(L.mlg_peer_adam_step_emulated(g, p, f, world, opt0.bucket.n, m, v, t, 1e-2, 0.9, 0.999, 1e-8, float(opt0.wd),
                                              2.0, ctypes.c_void_p(scratch.data_ptr()), _cabi.stream_ptr()),
                "mlg_peer_adam_step_emulated")


@pytest.mark.parametrize("world,wd", [(1, 0.0), (2, 0.0), (3, 0.0), (4, 1e-2)])
def test_peer_adam_matches_torch_adam(mlg, world, wd):
    from multilevel_gnn_b200 import _cabi
    shapes = [(257, 33), (1000,), (64, 64), (3,), (50001,)]
    init, ranks, g = _virtual_ranks(mlg, shapes, world, 7 + world, wd)
    ref = [torch.nn.Parameter(t.clone().double()) for t in init]
    ref_opt = torch.optim.Adam(ref, lr=1e-2, betas=(0.9, 0.999), weight_decay=wd)
    scratch = torch.empty(int(_cabi.lib().mlg_peer_emulated_bytes(world)), dtype=torch.uint8, device=DEV)
    for step in range(4):
        grads = [[torch.randn(t.shape, generator=g) for t in init] for _ in range(world)]
        for p, gs in zip(ref, zip(*grads)):
            p.grad = torch.stack([x.double() for x in gs]).sum(0) / world
        ref_opt.step()
        for (params, bucket, opt), gr in zip(ranks, grads):
            bucket.store([x.to(DEV) for x in gr])
        _step_all(mlg, ranks, scratch)
        torch.cuda.synchronize()
        assert all(o.arena.status() == 0 for _, _, o in ranks), "a rank timed out waiting for its peers"
    for params, bucket, opt in ranks:
        for p, q, p0 in zip(params, ref, ranks[0][0]):
            assert torch.equal(p.data, p0.data), "replicas must stay bitwise identical"
            torch.testing.assert_close(p.data.cpu().double(), q.data, rtol=2e-5, atol=2e-6)
        assert float(opt.step_dev.item()) == 4.0


def test_peer_adam_timeout_is_a_hard_failure(mlg):
    """One rank of two never shows up: the waiting rank must give up, leave parameters and optimizer state untouched, set the
    device status of BOTH arenas and the pinned host word, and refuse to run again."""
    init, ranks, g = _virtual_ranks(mlg, [(1000,), (77, 3)], 2, 3, 0.0)
    params, bucket, opt = ranks[0]
    opt.timeout_s = 0.05
    before = [p.data.clone() for p in params]
    bucket.store([torch.randn(t.shape, generator=g).to(DEV) for t in init])
    opt.step()                     # rank 1 never launches: rank 0 waits 50 ms and gives up (a lone kernel: nothing to deadlock)
    torch.cuda.synchronize()
    assert opt.failed() and opt.arena.status() == 1
    assert ranks[1][2].arena.status() == 1, "the failure must be visible in the peer's status word too"
    assert all(torch.equal(p.data, b) for p, b in zip(params, before)), "a failed step must not touch the parameters"
    assert float(opt.step_dev.item()) == 0.0 and float(opt.exp_avg.abs().sum()) == 0.0
    opt.step()                     # sticky: returns immediately
    torch.cuda.synchronize()
    assert all(torch.equal(p.data, b) for p, b in zip(params, before))


def test_peer_adam_in_cuda_graph(mlg):
    """The update kernel replays inside a CUDA graph (device-side step counter and epoch), world = 1."""
    init, ranks, g = _virtual_ranks(mlg, [(4096,), (31, 7)], 1, 3, 0.0)
    params, bucket, opt = ranks[0]
    ref = [torch.nn.Parameter(t.clone().double()) for t in init]
    ref_opt = torch.optim.Adam(ref, lr=1e-2, betas=(0.9, 0.999))
    static = [torch.zeros(t.shape, device=DEV) for t in init]
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        bucket.store(static)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        bucket.store(static)
        opt.step()
    # the capture itself does not run the kernel: three replays = three steps
    for step in range(3):
        gr = [torch.randn(t.shape, generator=g) for t in init]
        for p, x, st in zip(ref, gr, static):
            p.grad = x.double()
            st.copy_(x)
        ref_opt.step()
        graph.replay()
    torch.cuda.synchronize()
    assert opt.arena.status() == 0 and not opt.failed()
    for p, q in zip(params, ref):
        torch.testing.assert_close(p.data.cpu().double(), q.data, rtol=2e-5, atol=2e-6)
