#!/usr/bin/env python
"""bench.py -- train graphs/sec on the gbm.yaml shape (BASELINE.json metric), 1..8 B200.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 2 --warmup 1      # CPU port of the reference path
    python bench.py --steps 20 --warmup 5 --dump-outputs DIR   # also DIR/*.npy: loss, gradients, parameters of the last timed step

One step = one pass of the hot path over one batch of 32 synthetic patient graphs per GPU
(MultilevelGNN forward, BCE + feature loss, backward, gradient all-reduce, Adam), SURVEY.md section 8(d)
cfg1/cfg5.  `value` times it with the batch resident in HBM; `e2e` re-uploads the batch from pinned
host memory every step and reads the loss back, as train.py:42,62 do.  Prints ONE JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="gbm", choices=["gbm", "kirc", "lgg"])
    ap.add_argument("--batch", type=int, default=None, help="graphs per GPU per step (default: the config's batch_size)")
    ap.add_argument("--cpu-batch", type=int, default=None,
                    help="graphs per CPU step of the reference arm / cpu_baseline (default: the GPU arm's batch)")
    ap.add_argument("--windows", type=int, default=3, help="timed windows of --steps steps each; the median is reported")
    ap.add_argument("--no-diffpool", action="store_true", help="skip the DiffPool legs (reference size + tensor-core contractions)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (fixed global batch 256, SURVEY section 8d cfg5)")
    ap.add_argument("--strong-batch", type=int, default=256, help="global batch of the strong-scaling leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-genconv", action="store_true", help="skip the GENConv aggregation roofline microbench")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step as a CUDA graph")
    ap.add_argument("--nccl-update", action="store_true",
                    help="N>1: NCCL all-reduce + replicated Adam instead of the fused NVLink peer-memory update kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, every trained parameter's gradient and updated "
                         "value) as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 train step; it has no meaning with --impl %s" % a.impl)
    return a


# ----------------------------------------------------------------------------------------------------
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons of one GPU sampled DURING the timed region: an NVML polling thread (1 ms period; the
    timed region of a 20-step run is ~30 ms, shorter than `nvidia-smi`'s start-up), `nvidia-smi -lms` as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index=0):
        self.p = self.f = self.thread = None
        self.sm, self.reason_bits, self.mx = [], 0, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nv, self.h, self.reasons_fn = nv, h, reasons_fn
            self._stop = threading.Event()
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self._sample()
            self.sm, self.reason_bits = [], 0
        except Exception:
            self.thread = None
        self.index = index

    def start(self):
        """Begin polling.  Set-up (NVML import/init: milliseconds) happens in __init__, BEFORE the barrier that opens the
        timed region -- done inside it, rank 0 would enter the region late and every other rank would wait for it."""
        if self.thread is not None:
            self.thread.start()
            return self
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None
        return self

    def _sample(self):
        try:
            self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            self.reason_bits |= int(self.reasons_fn(self.h))
        except Exception:
            pass

    def _poll(self):
        while not self._stop.is_set():
            self._sample()
            time.sleep(0.001)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self._sample()          # at least one sample with the last steps still in flight
            self._stop.set()
            self.thread.join(timeout=2)
            if self.sm:
                out = {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.mx,
                       "reasons": sorted(k for k, b in self.BITS.items() if self.reason_bits & b), "samples": len(self.sm),
                       "source": "nvml"}
            return out
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                   "source": "nvidia-smi"}
        return out


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` table
    (profiles/ncu_traffic.json: kernel -> {"dram_bytes": ..., "source": "profiles/<summary>"}), or None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        return (json.load(f).get(kernel) or {}).get("dram_bytes")




# per timer tag: the ncu kernel names behind it (profiles/ncu_traffic.json) and the ALGORITHMIC bytes of one launch (DESIGN.md section 4)
KERNEL_INFO = {
    "SAGE mean aggregation fwd+bwd (gather_nm_kernel on node-major rows)": {
        "ncu": ["gather_nm_kernel", "gather_nm_kernel#2"],
        "alg": "8*C*B*N + 8*nnz per launch counted by the timer (rows read once + written once + idx/val per entry), C = 32: the "
               "second SAGE layer (64 -> 32) runs transform-first, so its forward and backward aggregations gather 32-wide rows "
               "(with the addend row U / the copied self row: 12*C*B*N = 190 MB); bounded by L2 -> SM row gathers (441 MB re-read "
               "per launch: every source row once per CSR entry), not by DRAM.  The backward launch reads a node-major gradient "
               "(one contiguous block per CSR entry, written that way by the pool backward)"},
    "sage_rank1_fwd": {"ncu": ["sage_rank1_fwd_rows_kernel<2, 1>"],
                       "alg": "4*C*B*N (output) + 4*B*N + 8*nnz + 8*C*N (tables), C = 64: 137 MB, write bound"},
    "pool_bwd": {"ncu": ["pool_bwd_c32_kernel<2, 2>"], "alg": "2 * 4*C*B*N + 4*B*C*S*P: x read, g_x written, pooled gradient read"},
}


DUMP_BUDGET = 64 * 10 ** 6      # bytes --dump-outputs may write, all files together
DUMP_SAMPLE = 1 << 20           # elements kept of a longer tensor (kirc's classifier head alone has 43 M)


def last_step_outputs(tr, loss):
    """What one Trainer.step hands its caller, as float32 numpy arrays: the loss it returns and, for every trained
    parameter, the gradient of that step (grad.<name>) and the value Adam left (param.<name>).  A tensor of more than
    DUMP_SAMPLE elements is reduced to the same seeded sample of its flattened elements in every run and every build."""
    names = {id(p): n for n, p in tr.model.named_parameters()}
    out = {"loss": loss.detach().float().cpu().numpy()}
    for p in tr.params:
        for kind, t in (("param", p.detach()), ("grad", p.grad)):
            if t.numel() > DUMP_SAMPLE:
                idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
                t = t.reshape(-1)[idx.to(t.device)]
            out["%s.%s" % (kind, names[id(p)])] = t.float().cpu().numpy()
    nbytes = sum(v.nbytes for v in out.values())
    assert nbytes <= DUMP_BUDGET, "--dump-outputs: %d bytes > %d; lower DUMP_SAMPLE" % (nbytes, DUMP_BUDGET)
    return out


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + ".npy"), v)


def max_over_ranks(ms, world, dev):
    if world == 1:
        return ms
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------------
def cpu_reference_run(cfg, cpu_batch, steps, warmup):
    """Times one reference training step (train.py:38-68) on the host cores: the reference's OWN modules (oracle/_ref staged
    by oracle/make_ref.py, or /root/reference in the build container; kind "reference") behind oracle/pyg_stub.py, else the
    oracle's port of the same step (kind "port").  Returns (graphs/s, ms/step, cores, kind)."""
    import multilevel_gnn_b200 as m
    from oracle import ref_train
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    args = m.configs.make_args(cfg)
    torch.manual_seed(0)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model)
    batch = m.synth.multilevel_batch(batch_size=cpu_batch, seed=0)
    weight = torch.tensor([[0.8, 1.3]]).repeat(cpu_batch, 1)
    if ref_train.available():
        tr = ref_train.RefTrainer(cfg, model.state_dict(), weight, model.pathway_indexs, model.info_mask.data)
        kind = "reference"
    else:
        from oracle.train_port import CpuTrainer
        tr = CpuTrainer(model.state_dict(), args, weight, model.pathway_indexs)
        kind = "port"
    for _ in range(warmup):
        tr.step(batch)
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.step(batch)
    dt = time.perf_counter() - t0
    return cpu_batch * steps / dt, dt / steps * 1e3, cores, kind


def genconv_microbench(dev, hbm_peak):
    """GENConv softmax aggregation (fwd, fused MsgNorm epilogue) at cfg4: N=100k, k=16, H=128."""
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import _cabi, functional as Fn, graph
    n, k, H = 100000, 16, 128
    g = torch.Generator().manual_seed(0)
    src = torch.randint(0, n, (n * k,), generator=g)
    dst = torch.arange(n).repeat_interleave(k)
    ei = torch.stack([src, dst]).to(dev)
    x = torch.randn(n, H, generator=g).to(dev)
    e = torch.randn(n * k, H, generator=g).to(dev)
    topo = graph.topology(ei, n)
    scale = torch.ones(1, device=dev)
    t = torch.ones(1, device=dev)

    def run():
        return Fn.GenAggregate.apply(x, e, t, 1.0, None, scale, topo, "softmax", 1e-7, Fn.EPI_MSGNORM, True)

    for _ in range(3):
        run()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        run()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    nbytes = 4 * H * (n * k + 2 * n) + 4 * n * k + 4 * (n + 1)
    gbs = nbytes / ms / 1e6
    # backward of the same call (edge + node + t + msg_scale gradients): forward + backward minus forward
    xg, eg, tg, sg = (v.clone().requires_grad_() for v in (x, e, t, scale))
    go = torch.randn(n, H, generator=g).to(dev)

    def run_fb():
        h = Fn.GenAggregate.apply(xg, eg, tg, 1.0, None, sg, topo, "softmax", 1e-7, Fn.EPI_MSGNORM, True)
        return torch.autograd.grad(h, [xg, eg, tg, sg], go)

    for _ in range(2):
        run_fb()
    torch.cuda.synchronize()
    a.record()
    for _ in range(10):
        run_fb()
    b.record()
    torch.cuda.synchronize()
    ms_b = a.elapsed_time(b) / 10 - ms
    bbytes = 4 * H * (2 * n * k + 3 * n) + 8 * n * k
    bwd = {"kernel": "gen_bwd_ring_kernel (source-side sum inside the kernel)", "ms": round(ms_b, 4), "bytes": bbytes,
           "achieved": round(bbytes / ms_b / 1e6, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(bbytes / ms_b / 1e6 / hbm_peak, 4),
           "traffic": ncu_traffic("gen_bwd_ring_kernel<1, 0, 1, 1, 1>"),
           "note": "4H(2E+3N)+8E bytes; (forward+backward) - forward, 10 back-to-back repetitions"}
    del xg, eg, go
    return {"backward": bwd,
            "kernel": "gen_fwd_ring_kernel<1> (GENConv softmax aggregation + MsgNorm + residual, N=100k, k=16, H=128)", "bound": "hbm",
            "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(gbs / hbm_peak, 4),
            "ms": round(ms, 4), "bytes": nbytes, "traffic": ncu_traffic("gen_fwd_ring_kernel<1>"),
            "note": "inputs 0.93 GB > L2; 20 back-to-back launches; training-mode forward (also writes m and the "
                    "log-sum-exp for backward); traffic = ncu dram bytes per launch (profiles/ncu_traffic.json)"}


def dominant_kernel_alone(batch, hbm_peak, reps=20):
    """The dominant kernel (SAGE mean aggregation over the replicated CSR as the step's second layer launches it:
    transform-first, so 32-wide rows V gathered from the right half of the [U | V] buffer, U added, LeakyReLU fused) timed
    alone: `reps` back-to-back launches on the bench's own topology, CUDA events on the launching stream.  Besides the HBM
    fraction it reports the L2 -> SM side, which is what actually bounds a gather over ~7-entry rows: every source row is
    re-read once per entry, and those reads are served by L2 (full-chip L2 throughput cap measured at ~6300 B/clk,
    /opt/skills/guides/B300_MICROARCH.md 'LTS throughput cap')."""
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import functional as Fn, graph
    n = batch.x.shape[0]
    C = 32
    topo = graph.topology(batch.edge_index, n, self_loops=True, edge_weight=batch.edge_attr,
                          static_key=getattr(batch, "topology_key", None), period=3 * m.MultilevelGNN.GENES)
    uv = torch.randn(n, 2 * C, device=batch.x.device)
    out = torch.empty(n, C, device=batch.x.device)
    csr = topo.fwd
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()

    def run_graph_major():       # rows of (graph b, node i) at b * N + i: gather_sum_rep_kernel
        Fn.gather_sum(uv[:, C:], csr.rowptr, csr.col, topo.n_single, val=topo.fwd_val, post_mode=1, out=out,
                      addend=uv[:, :C], replicas=topo.replicas, order=topo.fwd_order, tag="sage_aggr_alone", act_slope=0.2)

    def run_node_major():        # [U | V] rows at i * B + b (what the step's forward launches): gather_nm_kernel
        _cabi.check(L.mlg_gather_sum_nm_ex(Fn._vptr(uv[:, C:]), 2 * C, _cabi.iptr(csr.rowptr), _cabi.iptr(csr.col),
                                           _cabi.fptr(topo.fwd_val, True), None, _cabi.iptr(topo.fwd_order, True), topo.n_single,
                                           topo.replicas, 1, _cabi.fptr(uv), 2 * C, 1, 0.2, _cabi.fptr(out), C, None, 0, 0,
                                           _cabi.stream_ptr()), "mlg_gather_sum_nm_ex")

    def timed(run):
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms_gm = timed(run_graph_major)
    ms = timed(run_node_major)
    nnz = int(csr.col.numel())
    alg = 12 * C * n + 8 * nnz                                   # U and V read once, output written once, idx + val
    gathered = 4 * C * nnz * topo.replicas + 8 * C * n           # V rows re-read per entry + U rows read + rows written
    sm_mhz = 1965.0
    l2_cap = 6300.0 * sm_mhz / 1e3                               # GB/s
    return {"ms": round(ms, 4), "achieved": round(alg / ms / 1e6, 1), "frac": round(alg / ms / 1e6 / hbm_peak, 4),
            "l2_bytes": gathered, "l2_GBps": round(gathered / ms / 1e6, 1), "l2_cap_GBps": round(l2_cap, 0),
            "l2_frac": round(gathered / ms / 1e6 / l2_cap, 4), "graph_major_layout_ms": round(ms_gm, 4),
            "note": "%d launches back to back of the forward aggregation on node-major rows (gather_nm_kernel, what the step "
                    "launches; graph_major_layout_ms: gather_sum_rep_kernel on the reference's row order), [U | V] [%d,%d] fp32 "
                    "(126 MB) -> out [%d,%d], nnz=%d per graph x %d replicas; l2_cap = 6300 B/clk x 1965 MHz (guide-measured "
                    "full-chip LTS cap)" % (reps, n, 2 * C, n, C, nnz, topo.replicas)}


def diffpool_legs(dev):
    """DiffPool (SURVEY.md section 8d cfg3): (1) forward + backward at the reference's size through DiffPool.forward
    (x [576, 146, 32], shared adj [146, 146], 146 -> 37 -> 10: the fused one-CTA-per-sample kernels), latency; (2) the four
    contractions of the synthetic-large shape (N = 10 k, K = 2.5 k, C = 1024) on the tcgen05 bf16 GEMM against the measured
    dense bf16 peak; (3) one DiffPool.forward at that shape end to end (fp32 in / out, casts included)."""
    import ctypes
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import _cabi
    L = _cabi.lib()
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    bf16_peak = float(json.load(open(path))["bf16_tflops"]) if os.path.exists(path) else 1590.0

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a0.record()
        for _ in range(reps):
            fn()
        a1.record()
        torch.cuda.synchronize()
        return a0.elapsed_time(a1) / reps

    out = {}
    args = m.configs.make_args("lgg")
    torch.manual_seed(0)
    dp = m.DiffPool(32, 2, 146, 2, 32, 64, args).to(dev)
    x, adj = m.synth.diffpool_inputs(576, 146, 32)
    xg, ag = x.to(dev).requires_grad_(), adj.to(dev)
    params = list(dp.parameters())

    def fwd_bwd():
        o, l, e = dp(xg, ag)
        torch.autograd.grad((o.sum() + l + e), [xg] + params, allow_unused=True)

    with torch.no_grad():
        ms_f = timed(lambda: dp(xg, ag), 10)
    ms_fb = timed(fwd_bwd, 10)
    dims = [(146, 32, 37, 32), (37, 32, 10, 64)]
    flop_f = 2.0 * 576 * sum(n * n * c + 2 * n * c * (k + h) + n * k * h + 2 * n * n * k + n * k * k for n, c, k, h in dims)
    out["reference_size"] = {"shape": "b=576, 146 -> 37 -> 10 nodes, 32 -> 32 -> 64 channels", "fused_kernel": bool(dp._fused_plan(xg, ag, None)),
                             "fwd_ms": round(ms_f, 4), "fwd_bwd_ms": round(ms_fb, 4), "fwd_GFLOPs_fp32": round(flop_f / ms_f / 1e6, 1),
                             "bound": "fp32 FMA out of shared memory (146-wide problems: no tensor-core tile fits)"}
    legs = {}
    for (M, N, K, what) in [(2500, 10000, 10000, "S^T.A"), (2500, 2500, 10000, "(S^T.A).S"), (10000, 1024, 10000, "A.X"),
                            (2500, 1024, 10000, "S^T.X")]:
        A = torch.randn(M, K, device=dev).bfloat16()
        Bm = torch.randn(N, K, device=dev).bfloat16()
        C = torch.empty(M, N, device=dev)
        ws = torch.zeros(L.mlg_gemm_bf16_workspace_bytes(), dtype=torch.uint8, device=A.device)   # stream-K partials + flags
        run = lambda: _cabi.check(L.mlg_gemm_bf16_ws(ctypes.c_void_p(A.data_ptr()), K, 0, ctypes.c_void_p(Bm.data_ptr()), K, 0,
                                                     _cabi.fptr(C), N, 0, M, N, K, 1, 1.0, ctypes.c_void_p(ws.data_ptr()),
                                                     ws.numel(), _cabi.stream_ptr()), "mlg_gemm_bf16_ws")
        ms = timed(run, 10)
        tf = 2.0 * M * N * K / ms / 1e9
        legs[what] = {"M": M, "N": N, "K": K, "ms": round(ms, 4), "bound": "tensor", "achieved": round(tf, 1), "peak": bf16_peak,
                      "unit": "TFLOP/s", "frac": round(tf / bf16_peak, 4)}
        del A, Bm, C
    out["contractions_tcgen05_bf16"] = legs
    torch.manual_seed(0)
    big = m.DiffPool(1024, 2, 10000, 2, 1024, 1024, args).to(dev)
    xb = torch.randn(1, 10000, 1024, device=dev)
    ab = torch.rand(10000, 10000, device=dev)
    with torch.no_grad():
        ms_big = timed(lambda: big(xb, ab), 3, warm=1)
    out["large_forward"] = {"shape": "b=1, N=10000 -> 2500 -> 625, C=1024", "ms": round(ms_big, 3),
                            "note": "DiffPool.forward end to end, fp32 in/out: bf16 casts, softmax / normalise passes and the "
                                    "N x N link term included"}
    return out


# ----------------------------------------------------------------------------------------------------
def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multilevel_gnn_b200 as m
    B = a.cpu_batch or a.batch or m.configs.make_args(a.config).batch_size
    v, ms, cores, kind = cpu_reference_run(a.config, B, a.steps, a.warmup)
    sample = "%d train steps of %d synthetic %s-shaped graphs (N=15405, E=92430/graph), %d warm-up" % (
        a.steps, B, a.config, a.warmup)
    what = ("the reference's own modules (oracle/_ref) behind the pure-torch PyG stub" if kind == "reference"
            else "CPU port of the reference path (oracle/train_port.py)")
    print(json.dumps({
        "impl": "reference", "metric": "train graphs/sec (%s.yaml shape)" % a.config, "value": round(v, 3),
        "unit": "graphs/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config/%s.yaml MultilevelGNN train step (fwd+bwd+allreduce+Adam), %d graphs/GPU, "
                               "N=15405 nodes, E=92430 edges/graph, G=25015, P=%d" % (a.config, B, m.configs.make_args(a.config).pca_dim),
                   "graphs_per_gpu": B, "ran_on": "host cores: " + what},
        "cpu_baseline": {"value": round(v, 3), "unit": "graphs/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(v, 3), "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def strong_scaling_leg(a, args, world, rank, dev, steps):
    """SURVEY section 8(d) cfg5, second half: a FIXED global batch (256 graphs) split over the ranks -- per-GPU batch 256 / N --
    through the same Trainer (own model replica, captured graph, fused peer update).  Returns (graphs/s, ms/step, per-GPU batch)."""
    import types
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200.train import Trainer
    Bs = a.strong_batch // world
    torch.manual_seed(0)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model)
    model.to(dev)
    model.pathway_indexs = model.pathway_indexs.to(dev)
    raw = m.synth.multilevel_batch(batch_size=Bs, seed=300 + rank)
    n1 = 3 * m.MultilevelGNN.GENES
    E1 = raw.edge_index.shape[1] // Bs
    topo = m.data.FoldTopology(raw.edge_index[:, :E1], raw.edge_attr[:E1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    patients = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(Bs)]
    resident = m.data.to_device(m.data.collate(patients, topo, pin=False), topo, dev)
    weight = torch.tensor([[0.8, 1.3]]).repeat(Bs, 1).to(dev)
    tr = Trainer(model, args, weight, world_size=world, peer_update=False if a.nccl_update else None)
    for _ in range(3):
        tr.step(resident)
    if not a.no_graph:
        tr.capture(resident)
        tr.step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    e0.record()
    for _ in range(steps):
        tr.step(resident)
    e1.record()
    barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
    return Bs * world * steps / (ms / 1e3), ms / steps, Bs


def run_b200(a):
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import _cabi
    from multilevel_gnn_b200.train import Trainer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _cabi.lib()
    args = m.configs.make_args(a.config)
    B = a.batch or args.batch_size
    torch.manual_seed(0)
    model = m.MultilevelGNN(args)
    m.synth.multilevel_params(model)
    model.to(dev)
    model.pathway_indexs = model.pathway_indexs.to(dev)
    # batches come out of the loader replacement (data.collate): per-patient records + ONE FoldTopology
    raw = m.synth.multilevel_batch(batch_size=B, seed=100 + rank)
    n1 = 3 * m.MultilevelGNN.GENES
    E1 = raw.edge_index.shape[1] // B
    topo = m.data.FoldTopology(raw.edge_index[:, :E1], raw.edge_attr[:E1], raw.gene_pca_match[0], raw.raw_indice[0], n1)
    import types
    patients = [types.SimpleNamespace(x=raw.x[i * n1:(i + 1) * n1], age=raw.age[i], y=raw.y[2 * i:2 * i + 2]) for i in range(B)]
    host = m.data.collate(patients, topo, pin=True)
    weight = torch.tensor([[0.8, 1.3]]).repeat(B, 1).to(dev)
    tr = Trainer(model, args, weight, world_size=world, peer_update=False if a.nccl_update else None)
    resident = m.data.to_device(host, topo, dev)
    hbm_peak, peak_src = peaks()

    # ---- warm-up (builds the CSR / pool layouts), optional CUDA-graph capture of the whole step ----
    for _ in range(max(a.warmup, 3)):
        tr.step(resident)
    l0 = _cabi.LAUNCH_COUNT
    tr._step_eager(resident)
    launches_per_step = _cabi.LAUNCH_COUNT - l0
    if not a.no_graph:
        tr.capture(resident)
        for _ in range(2):
            tr.step()

    # ---- resident leg: `value` = median of `--windows` timed windows of EXACTLY --steps steps each ----
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    windows_ms = []
    barrier(world)
    if sampler:
        sampler.start()
    for _ in range(max(1, a.windows)):
        barrier(world)
        e0.record()
        for _ in range(a.steps):
            loss = tr.step(resident)
        e1.record()
        barrier(world)
        windows_ms.append(max_over_ranks(e0.elapsed_time(e1), world, dev))
    ms_total = statistics.median(windows_ms)
    clocks = sampler.stop() if sampler else None
    launches = launches_per_step * a.steps
    loss_value = float(loss.item())
    dumped = None
    if a.dump_outputs:          # read now: the legs below step the same trainer further
        dumped = last_step_outputs(tr, loss) if rank == 0 else None
        barrier(world)          # the other ranks wait here, not in a fused peer-update kernel that gives up after seconds

    # ---- end-to-end legs: pinned host batch -> device EVERY step (train.py:42), loss read back (train.py:62) ----
    # graph mode: the next batch's H2D runs on a copy stream while the current step's graph executes; the loss of EVERY step
    # reaches the host inside the timed region, step i's value being awaited while step i+1 runs (Trainer.loss_to_host).
    # (1) `e2e`: batches from data.collate (the loader replacement): the fold-constant topology travels once under its key,
    #     per step only node values / labels / age are uploaded.  (2) `e2e_full_upload`: keyless batches as the reference's
    #     PyG loader emits them -- all 78 MB re-sent every step and verified on the device against the captured topology.
    def e2e_leg(host_batch):
        pending = []

        def step(first=False):
            if tr.graph is None:
                return float(tr.step(host_batch.to(dev, non_blocking=True)).item())
            if first:
                tr.prefetch(host_batch)
            handle = tr.loss_to_host(tr.step_prefetched())
            tr.prefetch(host_batch)                # H2D of the following step's batch, overlapped with this replay
            pending.append(handle)
            return pending.pop(0).get() if len(pending) > 1 else None

        def drain():
            out = [h.get() for h in pending]
            pending.clear()
            return out

        step(first=True)
        step()
        drain()
        barrier(world)
        nbytes = tr.h2d_bytes(host_batch) if tr.graph is not None else host_batch.nbytes()
        losses = []
        e0.record()
        for _ in range(a.steps):
            losses.append(step())
        losses += drain()
        e1.record()
        barrier(world)
        losses = [x for x in losses if x is not None]
        assert len(losses) == a.steps and all(x == x for x in losses), "every step's loss must reach the host"
        if tr.graph is not None:
            torch.cuda.synchronize()      # the prefetch issued by the last step is still in flight: let it land
        return max_over_ranks(e0.elapsed_time(e1), world, dev), nbytes

    ms_e2e, h2d = e2e_leg(host)
    keyless = m.synth.GraphBatch(**{k: v for k, v in vars(host).items() if k != "topology_key"})
    ms_full, h2d_full = e2e_leg(keyless)
    if tr.graph is not None:
        tr.check_topology_flag()

    # ---- per-kernel device time (CUDA events around every launch of the same step, eager) ----
    timer = _cabi.KernelTimer()
    _cabi.TIMER = timer
    for _ in range(a.steps):
        # a device-side delay in front of every eager step: the host (a few ms of Python per eager step) enqueues the whole step
        # while the GPU spins, so a span measures its kernel and not the wait for a launch that had not been issued yet
        torch.cuda._sleep(16_000_000)
        tr._step_eager(resident)
    torch.cuda.synchronize()
    _cabi.TIMER = None
    ksum = timer.summary()
    barrier(world)

    strong = None
    strong_err = None
    if not a.no_strong and a.strong_batch % world == 0:
        try:
            strong = strong_scaling_leg(a, args, world, rank, dev, a.steps)
        except Exception as exc:          # an extra key must never take the headline line down with it
            if world > 1:
                raise                     # (a rank that stops here would leave its peers waiting in a collective)
            strong_err = "%s: %s" % (type(exc).__name__, exc)
    if tr.peer is not None and tr.peer.status() != 0:
        # a rank gave up waiting for a peer's flag inside the fused update kernel: the replicas are no longer in step
        raise SystemExit("bench.py: rank %d: a peer wait of the fused NVLink update kernel timed out; the measurement is void "
                         "(re-run with --nccl-update to take the library path)" % rank)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_step = ms_total / a.steps
    value = B * world * a.steps / (ms_total / 1e3)
    # the kernels of the step, by what bounds them (DESIGN.md section 4)
    bound_of = {"sage_aggr_fwd": "hbm", "sage_aggr_bwd": "hbm", "pool_fwd": "hbm", "pool_bwd_x": "hbm",
                "pool_bwd_w": "hbm", "pool_bwd": "hbm", "sage_update_gemm": "hbm (tensor 3xTF32)", "sage_dgrad_gemm": "hbm (tensor 3xTF32)", "sage_bias_act": "hbm", "embed_scale_bwd": "hbm", "sage_wgrad": "fp32-fma"}
    # sage_aggr_fwd / sage_aggr_bwd: the layer-2 aggregation on the CSR / its transpose, reported together
    merged = {}
    for tag, d in ksum.items():
        key = "SAGE mean aggregation fwd+bwd (gather_nm_kernel on node-major rows)" if tag.startswith("sage_aggr") else tag
        m = merged.setdefault(key, {"launches": 0, "ms": 0.0, "bytes": 0, "bound": bound_of.get(tag, "hbm")})
        for f in ("launches", "ms", "bytes"):
            m[f] += d[f]
    hbm_kernels = {k: v for k, v in merged.items() if v["bound"] == "hbm"}
    roof = None
    if hbm_kernels:
        tag, d = max(hbm_kernels.items(), key=lambda kv: kv[1]["ms"])
        gbs = d["bytes"] / d["ms"] / 1e6
        info = KERNEL_INFO.get(tag, {})
        tr_vals = [t for t in (ncu_traffic(k) for k in info.get("ncu", [])) if t]
        roof = {"kernel": tag, "bound": "hbm", "achieved": round(gbs, 1), "peak": hbm_peak, "unit": "GB/s",
                "frac": round(gbs / hbm_peak, 4), "traffic": (int(sum(tr_vals) / len(tr_vals)) if tr_vals else None),
                "traffic_source": ("profiles/ncu_traffic.json: mean of " + ", ".join(info.get("ncu", []))) if tr_vals else None,
                "peak_source": peak_src,
                "launches": d["launches"], "avg_us": round(d["ms"] / d["launches"] * 1e3, 2),
                "share_of_step": round(d["ms"] / ms_total, 4),
                "algorithmic_bytes": info.get("alg", "see DESIGN.md section 4"),
                "timed": "CUDA events around each launch in an eager pass of the same %d steps, each step queued behind an 8 ms device-side delay so that no span waits for the host (the timed region itself "
                         "is a CUDA-graph replay)" % a.steps,
                "back_to_back": dominant_kernel_alone(resident, hbm_peak),
                "all_kernels": {k: {"bound": v["bound"], "ms_per_step": round(v["ms"] / a.steps, 4),
                                    "share_of_step": round(v["ms"] / ms_total, 4),
                                    "GBps": round(v["bytes"] / v["ms"] / 1e6, 1) if v["ms"] > 0 and v["bytes"] else None}
                                for k, v in sorted(merged.items())}}
    line = {
        "metric": "train graphs/sec (%s.yaml shape)" % a.config, "value": round(value, 2), "unit": "graphs/s",
        "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": round(ms_step, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config/%s.yaml MultilevelGNN train step (fwd+bwd+allreduce+Adam), %d graphs/GPU, "
                               "N=15405 nodes, E=92430 edges/graph, G=25015, P=%d" % (a.config, B, args.pca_dim),
                   "graphs_per_gpu": B, "parallelism": "dp%d" % world, "step": ("eager" if tr.graph is None else "one CUDA graph (fwd+loss+bwd+Adam)" if world == 1 else
                            "one CUDA graph per rank (fwd+loss+bwd + ONE fused kernel: gradient reduce-scatter -> Adam on the "
                            "owned shard -> parameter all-gather over NVLink peer memory; no NCCL call in the step)"
                            if tr.peer is not None else
                            "CUDA graph (fwd+loss+bwd) -> NCCL all-reduce -> CUDA graph (Adam)"),
                   "l2": "no flush: per-step working set (~2 GB of activations) exceeds the 126 MB L2",
                   "timing": "median of %d windows of %d steps" % (len(windows_ms), a.steps),
                   "e2e_h2d": "batches from data.collate (the PyG-collate replacement): per-step node features, labels, age "
                              "from pinned memory; the edge list / pooling layout are fold constants (one gene network for "
                              "all patients, multiloader.py:687-698) uploaded once under the batch's topology_key; "
                              "e2e_full_upload re-sends everything"},
        "e2e": {"value": round(B * world * a.steps / (ms_e2e / 1e3), 2), "unit": "graphs/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / a.steps, 4),
                "loss_readback": "every step's loss is copied to pinned host memory and read by the host inside the timed "
                                 "region; step i's value is awaited while step i+1 runs"},
        "e2e_full_upload": {"value": round(B * world * a.steps / (ms_full / 1e3), 2), "unit": "graphs/s",
                            "h2d_bytes_per_step": h2d_full, "d2h_bytes_per_step": 8, "ms_per_step": round(ms_full / a.steps, 4),
                            "note": "keyless batches (the reference loader's layout: every batch re-sends edge list, edge "
                                    "weights and pooling tables); PCIe-bound; the re-sent topology is compared on the "
                                    "device with the captured one"},
        "windows_ms": [round(x, 4) for x in windows_ms],
        "strong_scaling": ({"error": strong_err} if strong_err else None if strong is None else
                           {"global_batch": a.strong_batch, "graphs_per_gpu": strong[2], "value": round(strong[0], 2),
                            "unit": "graphs/s", "ms_per_step": round(strong[1], 4),
                            "note": "SURVEY section 8(d) cfg5: fixed global batch, per-GPU batch = global / N; same trainer, resident batch"}),
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "loss": loss_value,
        "dp_update": (None if world == 1 else "nccl all-reduce + replicated Adam" if tr.peer is None else
                      {"kernel": "peer_adam_kernel (reduce-scatter -> Adam shard -> all-gather over NVLink peer memory)",
                       "status": tr.peer.status()}),
        "cuda_graph": tr.graph is not None,
    }
    if world == 1 and not a.no_genconv:
        line["genconv_agg"] = genconv_microbench(dev, hbm_peak)
    if world == 1 and not a.no_cpu_baseline:
        cb = a.cpu_batch or B
        v, ms, cores, kind = cpu_reference_run(a.config, cb, 2, 1)
        line["cpu_baseline"] = {"value": round(v, 3), "unit": "graphs/s", "cores": cores, "kind": kind,
                                "sample": "2 train steps of %d graphs (same shape), 1 warm-up, torch CPU threads=%d"
                                          % (cb, cores)}
    if world == 1 and not a.no_diffpool:
        line["diffpool"] = diffpool_legs(dev)
    if dumped is not None:
        write_outputs(a.dump_outputs, dumped)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
