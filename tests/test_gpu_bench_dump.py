"""bench.py --dump-outputs: the last timed step's loss, gradients and updated parameters as .npy files, within the size
budget, and the same from run to run (seeded inputs), so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--gpus", "1", "--warmup", "1", "--windows", "1", "--no-cpu-baseline", "--no-diffpool", "--no-genconv", "--no-strong"]


def _bench(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + ["--steps", str(steps), "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-len(".npy")]: np.load(os.path.join(out, f)) for f in os.listdir(out)}


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    import multilevel_gnn_b200 as m
    line, a = _bench(tmp_path / "a", 2)
    _, b = _bench(tmp_path / "b", 2)
    _, c = _bench(tmp_path / "c", 3)
    args = m.configs.make_args("gbm")
    model = m.MultilevelGNN(args)
    trained = {n: p for n, p in model.named_parameters() if p.requires_grad and not n.endswith("lin_l.weight")}
    assert sorted(a) == sorted(["loss"] + ["param." + n for n in trained] + ["grad." + n for n in trained])
    assert float(a["loss"]) == line["loss"]
    assert sum(v.nbytes for v in a.values()) <= 64 * 10 ** 6
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        n = k.split(".", 1)[-1]
        if n in trained:
            want = (1 << 20,) if trained[n].numel() > 1 << 20 else tuple(trained[n].shape)     # head.0.weight: a sample
            assert v.shape == want, k
    assert float(np.abs(a["grad.node_embedding"]).max()) > 0
    for k in a:
        np.testing.assert_allclose(b[k], a[k], rtol=1e-5, atol=1e-6 * max(1.0, float(np.abs(a[k]).max())), err_msg=k)
    # one more timed step (run c): its dump differs from run a's in every parameter, by no more than one Adam step can move
    # a parameter (lr (1 - beta1) / sqrt(1 - beta2) for these betas): run c's last timed step starts where run a's dump
    # stands (same seeded inputs, same sequence of steps up to there)
    bound = args.lr * (1 - args.beta1) / (1 - args.beta2) ** 0.5 * 1.001
    assert c["loss"] != a["loss"]
    for n in trained:
        d = np.abs(c["param." + n].astype(np.float64) - a["param." + n])
        assert d.max() > 0 and d.max() <= bound, (n, float(d.max()), bound)
