"""CPU: bench.py's reference arm (`--impl reference`, the CPU oracle on the host cores) prints ONE JSON line with the keys
the driver reads; run on the tiny workload so it finishes in seconds.  The native arm needs a GPU and must say so."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    for k in ("metric", "value", "unit", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["config"]["workload"] == "tiny" and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_rejects_arguments_it_cannot_honour(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                  ["--workload", "cfg5", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny"] + extra,
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, extra
    assert not os.listdir(tmp_path)


def test_native_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
