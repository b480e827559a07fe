"""CPU checks of bench.py's contract: the reference arm prints ONE JSON line with the agreed keys (and uses every schedulable core even
when OMP_NUM_THREADS=1 is exported, as torchrun does to its workers); non-zero ranks of that arm exit silently; the GPU arm refuses to
run without a CUDA device; the oracle is only reachable from the cpu_baseline / reference legs."""
import json
import os
import re
import subprocess
import sys

from conftest import ROOT


def _run(args, env_extra=None, timeout=300):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)


KEYS = ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
        "data", "config", "cpu_baseline", "e2e", "gpu_launches")


def _check_line(r):
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in KEYS:
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "path-steps/s" and d["n_gpus"] == 2 and d["gpu_launches"] == 0 and d["value"] > 1e6
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["value"] == d["value"]
    usable = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    assert d["cpu_baseline"]["cores"] == usable           # not the 1 that OMP_NUM_THREADS=1 would give
    return d


def test_reference_arm_port_fallback_json_line_and_core_count():
    """without the installed reference (or with numba disabled) the arm times the oracle's C port on every schedulable core"""
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"], {"OMP_NUM_THREADS": "1", "RANK": "0", "WORLD_SIZE": "2",
                                                                                         "B200SV_BENCH_CPU_BUDGET_S": "2", "B200SV_BENCH_NO_NUMBA": "1"})
    d = _check_line(r)
    assert d["cpu_baseline"]["kind"] == "port"


def test_reference_arm_runs_the_unmodified_numba_reference_when_installed():
    """oracle/_ref (oracle/install_reference.sh) present: the arm is the reference as shipped -- Numba, one process per core"""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "stochvolmodels")):
        import pytest
        pytest.skip("oracle/_ref not installed in this checkout")
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"], {"OMP_NUM_THREADS": "1", "RANK": "0", "WORLD_SIZE": "2",
                                                                                         "B200SV_BENCH_CPU_BUDGET_S": "1"}, timeout=600)
    d = _check_line(r)
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and "unmodified stochvolmodels" in cb["sample"]
    assert cb["one_core"] > 1e6 and cb["parallel_speedup"] > 0.5 and "effective" in cb["cpu"]


def test_reference_arm_other_ranks_stay_silent():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"], {"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(["--steps", "1", "--warmup", "0", "--no-cpu-baseline"])
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_oracle_confined_to_cpu_legs_in_bench_source():
    src = open(os.path.join(ROOT, "bench.py")).read()
    uses = [m.start() for m in re.finditer(r"from oracle|import oracle", src)]
    allowed = ("def cpu_port_rate", "def cpu_port_block", "def run_reference")     # the CPU timing helpers of cpu_baseline / --impl reference
    for u in uses:
        fn_start = src.rfind("\ndef ", 0, u)
        assert src[fn_start:].lstrip().startswith(allowed), src[fn_start:fn_start + 60]
    # the Numba reference runs in a subprocess (oracle/ref_arm.py) launched only from numba_reference_block
    assert src.count('"ref_arm.py"') == 1
