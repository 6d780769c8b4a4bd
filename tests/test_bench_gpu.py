"""bench.py --dump-outputs: the files hold what the timed step computed -- the gradient and sum r^2 of the seeded C2 batch --
and agree with the CPU oracle on the same seeded parameters and points."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import workloads
from helpers import build_fused, get_params, oracle_eval, assert_parity

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_timed_step(tmp_path):
    n, steps = 4096, 3
    out = tmp_path / "outputs"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--points", str(n), "--cpu-seconds", "0.1", "--fit-epochs", "0", "--no-gpu-comparator",
                          "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads([ln for ln in res.stdout.splitlines() if ln.strip()][-1])
    assert line["step_ms_stats"]["count"] == steps and line["config"]["points_per_gpu"] == n   # event pairs timed
    files = sorted(os.listdir(str(out)))
    assert files == ["grad.npy", "sumsq.npy"]
    assert sum(os.path.getsize(str(out / f)) for f in files) <= 64 << 20
    grad, sumsq = np.load(str(out / "grad.npy")), np.load(str(out / "sumsq.npy"))
    assert grad.dtype == np.float32 and sumsq.dtype == np.float32 and sumsq.shape == (1,)

    wl, nets, _, fp = build_fused("c2", seed=0)             # the parameters and points bench.py uses at rank 0
    ref = oracle_eval("c2", get_params(nets), workloads.sample_coords(wl, n, seed=1000))
    assert grad.size == fp.grad.numel()
    # split the flat gradient the way the engine packs it (FusedProblem.grads_as_list), whatever the workload's net order
    grads = [grad[o:o + p.numel()].reshape(tuple(p.shape)) for p, o in zip(fp.params, fp.offsets)]
    assert_parity(None, None, float(sumsq[0]) / (n * fp.n_eq), grads, ref, label="c2 bench --dump-outputs")
