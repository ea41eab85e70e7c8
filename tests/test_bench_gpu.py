"""GPU: bench.py --dump-outputs writes what the last timed step computed, and the same arguments give the same outputs
(seeded inputs), so two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("latents", "velocity_cond", "velocity_uncond")


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "tiny", "--steps", str(steps),
                        "--warmup", "0", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == steps
    return {n: np.load(os.path.join(out_dir, n + ".npy")) for n in NAMES}


def test_dump_outputs_is_the_last_timed_step_and_reproducible(tmp_path):
    from diffsynth.schedulers.flow_match import FlowMatchScheduler
    a = _bench(tmp_path / "a", 1)
    for n in NAMES:
        assert a[n].dtype == np.float32 and a[n].shape == (1, 16, 3, 16, 16) and np.isfinite(a[n]).all(), n
    # one step from the seeded latents: x1 = x0 + (sigma_1 - sigma_0) * (v_u + cfg * (v_c - v_u)), the fused CFG/Euler update
    sched = FlowMatchScheduler(shift=5, sigma_min=0.0, extra_one_step=True)
    sched.set_timesteps(50, shift=5.0)
    x0 = torch.randn(1, 16, 3, 16, 16, generator=torch.Generator().manual_seed(0)).numpy()
    v = a["velocity_uncond"] + 5.0 * (a["velocity_cond"] - a["velocity_uncond"])
    np.testing.assert_allclose(a["latents"], x0 + float(sched.sigmas[1] - sched.sigmas[0]) * v, rtol=1e-5, atol=1e-5)
    b = _bench(tmp_path / "b", 1)
    for n in NAMES:
        np.testing.assert_allclose(b[n], a[n], rtol=1e-2, atol=1e-3, err_msg=n)
    c = _bench(tmp_path / "c", 2)          # a second timed step moves the latents on
    assert np.abs(c["latents"] - a["latents"]).max() > 1e-3
