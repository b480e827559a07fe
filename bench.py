#!/usr/bin/env python
"""bench.py -- LogSV Monte Carlo path-steps/sec on B200 (BASELINE.json `metric`), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--paths P] [--precision fp64|fp32] [--gauss fp32|fp64]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" = one pass of the hot path over one batch of synthetic input: price the whole option chain by Monte Carlo once
(simulate every maturity slice with the fused kernel, re-centre, per-strike payoff moments, prices + std errors).

Workload (config.workload): LogSV MC, BTC-style option chain (4 maturities, 49 strikes, reference sample chain and
LOGSV_BTC_PARAMS), nb_steps_per_year=582 => 25+34+57+136 = 252 steps per path, 1e8 paths PER GPU (weak scaling: per-GPU work
is fixed, the two per-maturity exchange steps are fp64 messages of <= 360 bytes).

Keys of the JSON line (rank 0):
`value`   : device-resident arm -- chain inputs already in HBM, CUDA-event timed on the launching stream, max over ranks.  Arithmetic:
            fp64 state, Gaussians drawn by the float Box-Muller on the SFU ("f64 state / f32 draws", the API default).
`all_fp64`: the same arm and the same e2e call with `gauss="fp64"` (fp64 Box-Muller from 52-bit uniforms) -- like-for-like with the
            CPU arms, which draw fp64 normals.
`e2e`     : the public API call a user makes (LogSVPricer.model_mc_price_chain -> C ABI) with HOST buffers in and out, host<->device
            copies inside the timed region.
`roofline`: dominant kernel (mc_slice_kernel) -- algorithmic bytes = 64 B per path-step (SURVEY.md §8d: the reference's streaming
            dataflow, 2 fp64 normals read + 3 fp64 state read + 3 written per path-step) over its CUDA-event duration, against the
            measured HBM copy bandwidth in MEASURED_PEAKS.json.  `traffic` and `compute_bound` are read from the parsed ncu capture
            profiles/slice_kernel_metrics.json (tools/ncu_summary.py), never from literals here.
`checks`  : N>1 only -- prices of the p2p exchange vs the NCCL exchange vs ONE GPU running all the paths (SURVEY.md §8d C5: <= 1e-13).
`extras`  : driver-visible numbers for BASELINE.json configs[0..4] (ms, path-steps/s, error vs the Fourier route / goldens).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the headline arm's LAST timed step returned -- the chain's 49 MC prices
            and their standard errors in chain order (float64, DIR/prices.npy and DIR/stds.npy).  Seeds depend only on the step index,
            so two builds run with the same arguments can be compared output for output.
`cpu_baseline` / `--impl reference`: the reference AS SHIPPED (unmodified stochvolmodels 2.2.0 in oracle/_ref, Numba; 1 core =
            one call, all cores = one call per worker process) with the oracle's C/OpenMP port beside it, both with effective-core
            accounting (affinity, cgroup quota, measured 1-thread rate and parallel speed-up).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NB_STEPS_PER_YEAR = 582          # BTC chain maturity gaps -> 25 + 34 + 57 + 136 = 252 steps
STEPS_PER_PATH = 252
ALGO_BYTES_PER_PATH_STEP = 64.0  # SURVEY.md §8(d)
SEED = 10
WORKLOAD = ("LogSV MC, BTC chain 4 maturities x 49 strikes, 252 steps/path (nb_steps_per_year=582, slices 25+34+57+136), "
            "LOGSV_BTC_PARAMS")


def workload():
    from stochvolmodels_b200 import LOGSV_BTC_PARAMS, get_btc_test_chain_data
    from stochvolmodels_b200.utils.funcs import set_time_grid
    chain = get_btc_test_chain_data()
    steps, t0 = [], 0.0
    for ttm in chain.ttms:
        steps.append(set_time_grid(ttm - t0, NB_STEPS_PER_YEAR)[0])
        t0 = ttm
    return chain, LOGSV_BTC_PARAMS, steps


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def slice_kernel_profile():
    """parsed ncu capture of the dominant kernel (written by tools/ncu_summary.py from the .ncu-rep of the shipped build)."""
    try:
        with open(os.path.join(ROOT, "profiles", "slice_kernel_metrics.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        clocks = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        maxc = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        power = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(clocks) if clocks else None, "sm_max_mhz": max(maxc) if maxc else None,
                "power_w_max": max(power) if power else None, "samples": len(clocks), "reasons": reasons}


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------------------------------------------------------------
def cpu_port_rate(chain, params, budget_s: float, nthreads: int):
    """time the C port on `nthreads` threads on a bounded sample of the SAME workload; returns (path_steps/s, paths, seconds)."""
    from oracle import cport
    p6 = (params.sigma0, params.theta, params.kappa1, params.kappa2, params.beta, params.volvol)
    # the thread count is passed explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers
    run = lambda n: cport.mc_chain("logsv", p6, chain.ttms, chain.forwards, chain.discfactors, None, chain.strikes_ttms,
                                   chain.optiontypes_ttms, n, NB_STEPS_PER_YEAR, True, 1, SEED, "f64", nthreads=nthreads)
    n0 = 20_000 * nthreads
    run(n0 // 4)                                   # warm (page faults, thread pool)
    t = time.perf_counter(); run(n0); dt0 = time.perf_counter() - t
    n = int(min(max(n0 * budget_s / max(dt0, 1e-3), n0), 4e8))
    t = time.perf_counter(); run(n); dt = time.perf_counter() - t
    return n * STEPS_PER_PATH / dt, n, dt


def cpu_port_block(chain, params, budget_s: float):
    """C/OpenMP port: 1-thread rate, all-effective-threads rate, measured parallel speed-up (what `cores` really delivered)."""
    from oracle import ref_arm
    cpus = ref_arm.effective_cpus()
    r1, n1, s1 = cpu_port_rate(chain, params, min(3.0, budget_s), 1)
    rn, nn, sn = cpu_port_rate(chain, params, budget_s, cpus["effective"])
    return {"value": rn, "unit": "path-steps/s", "cores": cpus["effective"], "kind": "port",
            "one_thread": r1, "parallel_speedup": rn / r1, "per_effective_core": rn / cpus["effective"],
            "sample": f"{nn} paths x 252 steps of the same chain, oracle/csrc/oracle_mc.c (OpenMP, fp64 draws, Philox stream), {sn:.1f} s"}


def numba_reference_block(budget_s: float, repeat: int, fourier: bool = False, timeout_s: float = 600.0):
    """run oracle/ref_arm.py (the unmodified reference in oracle/_ref) in a clean subprocess; returns its JSON dict.  Numba's on-disk
    cache and Python's bytecode go to a temporary directory / nowhere: the tree may be read-only."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_arm.py"), "--budget-s", str(budget_s), "--repeat", str(repeat)]
    if fourier:
        cmd.append("--fourier")
    env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "NUMBA_NUM_THREADS")}
    try:
        with tempfile.TemporaryDirectory(prefix="b200sv_numba_") as cache:
            env.update(NUMBA_CACHE_DIR=cache, PYTHONDONTWRITEBYTECODE="1")
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env, cwd=ROOT)
        lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
        if out.returncode != 0 or not lines:
            return {"unavailable": f"ref_arm.py rc={out.returncode}: {out.stderr.strip()[-300:]}"}
        return json.loads(lines[-1])
    except Exception as exc:      # timeout, missing interpreter ...
        return {"unavailable": f"{type(exc).__name__}: {exc}"}


def reference_summary(ref: dict):
    """cpu_baseline-style dict of the Numba reference run (all-cores value = median of the repeats)."""
    allc = ref.get("all_cores") or []
    one = ref.get("one_core")
    cpus = ref.get("cpus", {})
    if allc:
        value = statistics.median(a["value"] for a in allc)
        a0 = allc[0]
        sample = (f"{a0['workers']} worker processes x {a0['paths'] // a0['workers']} paths x 252 steps of the same chain per run "
                  f"({a0['seconds']:.1f} s), unmodified stochvolmodels 2.2.0 LogSVPricer.model_mc_price_chain (Numba {ref.get('numba')})")
        cores = a0["workers"]
    elif one:
        value, cores = one["value"], 1
        sample = f"{one['paths']} paths x 252 steps, one process ({one['seconds']:.1f} s)"
    else:
        return None
    d = {"value": value, "unit": "path-steps/s", "cores": cores, "kind": "reference", "sample": sample,
         "cpu": {k: cpus.get(k) for k in ("model", "os_cpu_count", "affinity", "cgroup_quota_cpus", "effective")}}
    if one:
        d["one_core"] = one["value"]
        d["parallel_speedup"] = value / one["value"]
        d["per_effective_core"] = value / max(cores, 1)
    return d


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, same workload / metric / unit;
    rank 0 only.  Preferred: the UNMODIFIED reference (oracle/_ref, Numba) on all effective cores, one bounded sample per step;
    fallback (reference not installed / numba missing): the oracle's C port."""
    if rank != 0:
        return
    chain, params, steps = workload()
    total = max(1, args.steps + args.warmup)
    budget = min(12.0, 150.0 / total)
    budget = float(os.environ.get("B200SV_BENCH_CPU_BUDGET_S", budget))     # tests shorten the bounded sample
    ref = numba_reference_block(budget, total, timeout_s=900.0) if not os.environ.get("B200SV_BENCH_NO_NUMBA") else {"unavailable": "disabled"}
    base = {"impl": "reference", "metric": "LogSV MC path-steps/sec", "unit": "path-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "gpu_launches": 0}
    summary = None if "unavailable" in ref else reference_summary(ref)
    if summary is not None and ref.get("all_cores"):
        timed = ref["all_cores"][args.warmup:] or ref["all_cores"]
        value = statistics.median(a["value"] for a in timed)
        summary["value"] = value
        a0 = timed[0]
        line = dict(base, value=value, ms_per_step=1e3 * statistics.median(a["seconds"] for a in timed),
                    config={"workload": WORKLOAD.replace("LOGSV_BTC_PARAMS", "LOGSV_BTC_PARAMS; bounded sample of "
                                                         f"{a0['paths']} paths per step ({a0['workers']} processes x {a0['paths'] // a0['workers']})"),
                            "paths_per_step": a0["paths"]},
                    cpu_baseline=summary)
    else:
        # fallback: C port of the reference algorithm
        rates = []
        from oracle import ref_arm
        threads = ref_arm.effective_cpus()["effective"]
        for i in range(total):
            r, n, secs = cpu_port_rate(chain, params, budget, threads)
            if i >= args.warmup:
                rates.append(r)
        value = statistics.median(rates)
        line = dict(base, value=value, ms_per_step=1e3 * secs,
                    config={"workload": WORKLOAD + f"; bounded sample of {n} paths per step", "paths_per_step": n},
                    cpu_baseline={"value": value, "unit": "path-steps/s", "cores": threads, "kind": "port",
                                  "sample": f"{n} paths x 252 steps, oracle/csrc/oracle_mc.c (OpenMP, fp64, Philox stream), {secs:.1f} s",
                                  "numba_reference_unavailable": ref.get("unavailable")})
    line["e2e"] = {"value": line["value"], "unit": "path-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------------------
# extras: BASELINE.json configs[0..4] through the public API (driver-visible; never allowed to lose the headline line)
# ---------------------------------------------------------------------------------------------------------------------------------
def _timed(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter(); out = fn(); ts.append(time.perf_counter() - t)
    return statistics.median(ts), out


def extras_single_gpu():
    """configs[0..3] on one GPU: wall ms through the API (host buffers), path-steps/s, error against the Fourier route / goldens."""
    from stochvolmodels_b200 import (HestonParams, HestonPricer, LOGSV_BTC_PARAMS, LogSvParams, LogSVPricer, OptionChain,
                                     get_btc_test_chain_data)
    out = {}
    K5 = np.array([0.8, 0.9, 1.0, 1.1, 1.2]); T5 = np.array(["P", "P", "C", "C", "C"])
    q = LogSvParams(sigma0=1.0, theta=1.0, kappa1=5.0, kappa2=5.0, beta=0.2, volvol=2.0)
    lp, hp = LogSVPricer(), HestonPricer()
    try:    # configs[0]: quickstart 5-strike slice, 10k paths x 64 steps
        chain = OptionChain(ttms=np.array([0.25]), forwards=np.ones(1), strikes_ttms=[K5], optiontypes_ttms=[T5])
        four = lp.price_chain(chain, q)[0]
        secs, (p, e) = _timed(lambda: lp.model_mc_price_chain(chain, q, nb_path=10_000, nb_steps=252, seed=SEED), 5)
        out["config0_quickstart_10k_x_64"] = {"ms": 1e3 * secs, "path_steps_per_s": 10_000 * 64 / secs, "fourier_atm": float(four[2]),
                                              "reference_atm": 0.197331, "mc_atm": float(p[0][2]), "mc_atm_se": float(e[0][2]),
                                              "max_z_vs_fourier": float(np.max(np.abs(p[0] - four) / e[0]))}
    except Exception as exc:
        out["config0_quickstart_10k_x_64"] = {"error": repr(exc)}
    try:    # configs[1]: Heston MC 1e6 paths x 252 steps, single maturity (ttm 0.7 x 360/yr -> 252), reference scheme + opt-in QE
        h = HestonParams(v0=0.04, theta=0.04, kappa=4.0, rho=-0.5, volvol=0.4)
        chain = OptionChain(ttms=np.array([0.7]), forwards=np.ones(1), strikes_ttms=[K5], optiontypes_ttms=[T5])
        four = hp.price_chain(chain, h)[0]
        blk = {}
        for scheme in ("euler_floor", "qe"):
            secs, (p, e) = _timed(lambda: hp.model_mc_price_chain(chain, h, nb_path=1_000_000, seed=SEED, scheme=scheme), 3)
            blk[scheme] = {"ms": 1e3 * secs, "path_steps_per_s": 1e6 * 252 / secs, "max_z_vs_fourier": float(np.max(np.abs(p[0] - four) / e[0])),
                           "max_abs_err": float(np.max(np.abs(p[0] - four)))}
        out["config1_heston_1e6_x_252"] = blk
    except Exception as exc:
        out["config1_heston_1e6_x_252"] = {"error": repr(exc)}
    try:    # configs[2]: LogSV MGF Fourier quadrature 5 maturities x 21 strikes vs the reference's own prices (committed golden)
        g = np.load(os.path.join(ROOT, "tests", "golden", "logsv_fourier_c3_5x21.npz"))
        M = int(g["nslices"])
        strikes, types = [g[f"strikes_{m}"] for m in range(M)], [g[f"types_{m}"] for m in range(M)]
        chain = OptionChain(ttms=g["ttms"], forwards=g["forwards"], strikes_ttms=strikes, optiontypes_ttms=types, discfactors=g["discfactors"])
        secs, prices = _timed(lambda: lp.price_chain(chain, q), 5)
        ref = np.concatenate([g[f"prices_{m}"] for m in range(M)])
        out["config2_logsv_fourier_5x21"] = {"ms": 1e3 * secs, "max_rel_err_vs_reference_golden": float(np.max(np.abs(np.concatenate(prices) / ref - 1.0))),
                                             "reference_cpu_s": 7.6}
    except Exception as exc:
        out["config2_logsv_fourier_5x21"] = {"error": repr(exc)}
    try:    # configs[3]: LogSV MC 1e7 paths x 252 steps, full BTC chain
        chain = get_btc_test_chain_data()
        four = np.concatenate(lp.price_chain(chain, LOGSV_BTC_PARAMS))
        secs, (p, e) = _timed(lambda: lp.model_mc_price_chain(chain, LOGSV_BTC_PARAMS, nb_path=10_000_000, nb_steps=NB_STEPS_PER_YEAR, seed=SEED), 3)
        p, e = np.concatenate(p), np.concatenate(e)
        fwd = np.concatenate([np.full(len(k), f) for k, f in zip(chain.strikes_ttms, chain.forwards)])
        out["config3_logsv_btc_1e7_x_252"] = {"ms": 1e3 * secs, "path_steps_per_s": 1e7 * 252 / secs,
                                              "max_abs_err_over_forward_vs_fourier": float(np.max(np.abs(p - four) / fwd)),
                                              "max_z_vs_fourier": float(np.max(np.abs(p - four) / e)), "tolerance_abs_over_forward": 1e-3}
    except Exception as exc:
        out["config3_logsv_btc_1e7_x_252"] = {"error": repr(exc)}
    return out


def extra_config4(world, rank, barrier, reduce_max):
    """configs[4]: LogSV MC 1e8 paths x 1024 steps (quickstart parameters, ttm 1, 1023 steps/yr) in TOTAL, strong-scaled over the
    `world` GPUs of this run through the public API (host buffers); all ranks call it."""
    from stochvolmodels_b200 import LogSvParams, LogSVPricer, OptionChain
    K5 = np.array([0.8, 0.9, 1.0, 1.1, 1.2]); T5 = np.array(["P", "P", "C", "C", "C"])
    q = LogSvParams(sigma0=1.0, theta=1.0, kappa1=5.0, kappa2=5.0, beta=0.2, volvol=2.0)
    chain = OptionChain(ttms=np.array([1.0]), forwards=np.ones(1), strikes_ttms=[K5], optiontypes_ttms=[T5])
    lp = LogSVPricer()
    call = lambda s: lp.model_mc_price_chain(chain, q, nb_path=100_000_000, nb_steps=1023, seed=s)
    call(SEED)
    barrier()
    t = time.perf_counter()
    reps = 3
    for k in range(reps):
        p, e = call(SEED + 1 + k)
    barrier()
    secs = reduce_max(time.perf_counter() - t) / reps
    if rank != 0:
        return None
    four = lp.price_chain(chain, q)[0]
    return {"ms": 1e3 * secs, "path_steps_per_s": 1e8 * 1024 / secs, "n_gpus": world, "scaling": "strong (1e8 paths in total)",
            "max_abs_err_vs_fourier": float(np.max(np.abs(p[0] - four))), "max_z_vs_fourier": float(np.max(np.abs(p[0] - four) / e[0]))}


# ---------------------------------------------------------------------------------------------------------------------------------
def dump_outputs(path: str, prices: np.ndarray, stds: np.ndarray) -> None:
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "prices.npy"), np.ascontiguousarray(prices, dtype=np.float64))
    np.save(os.path.join(path, "stds.npy"), np.ascontiguousarray(stds, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--paths", type=float, default=1e8, help="paths per GPU")
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    ap.add_argument("--gauss", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "collective"],
                    help="N>1: per-maturity moment exchange through NVLink peer memory inside the kernels (p2p) or NCCL all-reduce (collective)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the prices and standard errors of the last timed step to DIR/prices.npy and DIR/stds.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from stochvolmodels_b200 import LogSVPricer, engine
    from stochvolmodels_b200 import _capi as C
    from stochvolmodels_b200 import multi_gpu
    from stochvolmodels_b200.multi_gpu import CudaMcEngine
    from stochvolmodels_b200.pricers.logsv_pricer import _params_c
    from stochvolmodels_b200.utils.funcs import set_time_grid

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: stochvolmodels_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = C.load_library()
    chain, params, steps = workload()
    n_local = int(args.paths)
    total_paths = n_local * world
    offsets, strikes, types = C.flatten_chain(chain.strikes_ttms, chain.optiontypes_ttms)
    sizes = np.diff(offsets)
    use_p2p = world > 1 and args.exchange == "p2p"     # the two per-maturity messages ride inside the kernels over NVLink peer memory
    grid = []
    t0 = 0.0
    for ttm in chain.ttms:
        s, dt, _ = set_time_grid(ttm - t0, NB_STEPS_PER_YEAR)
        grid.append((s, dt))
        t0 = ttm
    path_steps_per_gpu = n_local * sum(s for s, _ in grid)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def device_arm(gauss: str, nsteps: int, nwarm: int, sample_clocks: bool):
        """device-resident arm; returns dict(value, ms_per_step, launches, clocks, slice_ms, slice_path_steps, prices[2, J])."""
        nonlocal use_p2p
        flags = engine.mc_flags(args.precision, gauss)
        eng = CudaMcEngine("logsv", _params_c(params), n_local, rank * n_local, flags, int(sizes.max()))
        if use_p2p:
            from stochvolmodels_b200.multi_gpu import P2pUnavailable
            try:
                eng.enable_p2p()
            except P2pUnavailable as e:          # raised on every rank together; the NCCL exchange is the same arithmetic
                if rank == 0:
                    print(f"bench.py: peer-memory exchange unavailable ({e}); using NCCL all-reduces", file=sys.stderr)
                use_p2p = False
                args.exchange = "collective"
        strikes_dev = eng.to_device(strikes, torch.float64)
        types_dev = eng.to_device(types, torch.int8)
        out_dev = torch.zeros((2, strikes.shape[0]), dtype=torch.float64, device=eng.device)
        slice_events = []

        def one_chain(seed, record):
            for m, (S, dt) in enumerate(grid):
                if record:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                mom = eng.simulate_slice(m, m == 0, S, dt, 1.0, True, float(chain.forwards[m]), seed)
                if record:
                    e1.record()
                    slice_events.append((e0, e1, S))
                if world > 1 and not use_p2p:
                    dist.all_reduce(mom)
                J, jo = int(sizes[m]), int(offsets[m])
                sums = eng.payoff_sums(float(chain.ttms[m]), float(chain.forwards[m]), strikes_dev[jo: jo + J], types_dev[jo: jo + J], J, C.LOG_RETURN, 1)
                if world > 1 and not use_p2p:
                    dist.all_reduce(sums)
                eng.finalize(sums, J, float(chain.discfactors[m]), total_paths, out_dev[0, jo: jo + J], out_dev[1, jo: jo + J])

        for w in range(nwarm):
            one_chain(SEED + w, False)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0 and sample_clocks:
            sampler.start()
        lib.b200sv_reset_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for k in range(nsteps):
            one_chain(SEED + 100 + k, True)
        ev1.record()
        barrier()
        launches = int(lib.b200sv_launch_count())
        clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
        elapsed_s = reduce_max(ev0.elapsed_time(ev1)) / 1e3
        if use_p2p:
            eng.check_p2p()
        res = {"value": path_steps_per_gpu * world * nsteps / elapsed_s, "ms_per_step": 1e3 * elapsed_s / nsteps, "launches": launches,
               "clocks": clocks, "slice_ms": sum(a.elapsed_time(b) for a, b, _ in slice_events),
               "slice_path_steps": sum(n_local * S for _, _, S in slice_events), "n_slice_launches": len(slice_events),
               "elapsed_s": elapsed_s, "prices": out_dev.cpu().numpy()}
        del eng
        torch.cuda.empty_cache()
        return res

    pricer = LogSVPricer()

    def e2e_arm(gauss: str, nsteps: int, nwarm: int, exchange):
        api = lambda seed: pricer.model_mc_price_chain(chain, params, nb_path=total_paths, nb_steps=NB_STEPS_PER_YEAR, seed=seed,
                                                       precision=args.precision, gauss=gauss, exchange=exchange)
        for w in range(nwarm):
            api(SEED + w)
        barrier()
        t = time.perf_counter()
        for k in range(nsteps):
            prices_api, stds_api = api(SEED + 100 + k)
        barrier()
        secs = reduce_max(time.perf_counter() - t)
        return path_steps_per_gpu * world * nsteps / secs, np.concatenate(prices_api), np.concatenate(stds_api)

    # ---------------- headline: f64 state / f32 draws ----------------
    head = device_arm(args.gauss, args.steps, args.warmup, True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, head["prices"][0], head["prices"][1])
    e2e_value, prices_api, stds_api = e2e_arm(args.gauss, args.steps, min(args.warmup, 2), args.exchange if world > 1 else None)
    # ---------------- all-fp64 sub-line (fp64 Box-Muller) ----------------
    alt_gauss = "fp64" if args.gauss == "fp32" else "fp32"
    sub_steps = max(2, min(args.steps, 3))
    try:
        sub = device_arm(alt_gauss, sub_steps, 1, False)
        sub_e2e, sub_prices_api, _ = e2e_arm(alt_gauss, sub_steps, 1, args.exchange if world > 1 else None)
    except Exception as exc:
        sub, sub_e2e, sub_prices_api = {"error": repr(exc)}, None, None

    h2d = strikes.nbytes + types.nbytes + 6 * 8 + 4 * 8 * 4 + offsets.nbytes      # strikes, types, params, ttms/forwards/dfs/etas, offsets
    d2h = 2 * strikes.shape[0] * 8

    # ---------------- N>1: the sharded prices against the other exchange and against ONE GPU running every path ----------------
    checks = None
    if world > 1:
        try:
            other = "collective" if args.exchange == "p2p" else "p2p"
            api_seed = SEED + 100 + args.steps - 1                           # the seed of the last timed API call
            p_this, _ = pricer.model_mc_price_chain(chain, params, nb_path=total_paths, nb_steps=NB_STEPS_PER_YEAR, seed=api_seed,
                                                    precision=args.precision, gauss=args.gauss, exchange=args.exchange)
            p_other, _ = pricer.model_mc_price_chain(chain, params, nb_path=total_paths, nb_steps=NB_STEPS_PER_YEAR, seed=api_seed,
                                                     precision=args.precision, gauss=args.gauss, exchange=other)
            multi_gpu.release_engines()
            torch.cuda.empty_cache()
            barrier()
            single = None
            if rank == 0:      # one GPU, all N x 1e8 paths (24 B/path of state: 19 GB at N=8), same global path ids => same draws
                single, _ = pricer.model_mc_price_chain(chain, params, nb_path=total_paths, nb_steps=NB_STEPS_PER_YEAR, seed=api_seed,
                                                        precision=args.precision, gauss=args.gauss, distributed=False)
            barrier()
            if rank == 0:
                a, b, c = np.concatenate(p_this), np.concatenate(p_other), np.concatenate(single)
                checks = {f"{args.exchange}_vs_{other}_max_rel": float(np.max(np.abs(a / b - 1.0))),
                          "vs_single_gpu_max_rel": float(np.max(np.abs(a / c - 1.0))), "tolerance": 1e-13, "paths_total": total_paths,
                          "api_vs_last_timed_call_max_rel": float(np.max(np.abs(a / prices_api - 1.0)))}
                checks["pass"] = bool(max(v for k, v in checks.items() if k.endswith("max_rel")) <= 1e-13)
        except Exception as exc:
            checks = {"error": repr(exc)}

    # ---------------- extras: BASELINE configs ----------------
    extras = {}
    if not args.no_extras:
        multi_gpu.release_engines()
        torch.cuda.empty_cache()
        try:
            c4 = extra_config4(world, rank, barrier, reduce_max)
            if rank == 0:
                extras["config4_logsv_1e8_x_1024"] = c4
        except Exception as exc:
            extras["config4_logsv_1e8_x_1024"] = {"error": repr(exc)}
        multi_gpu.release_engines()
        if world == 1:
            extras.update(extras_single_gpu())

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        # per launch: algorithmic bytes = 64 B x (n_local x S_m); achieved = sum of bytes / sum of CUDA-event durations of the slice launches
        achieved = ALGO_BYTES_PER_PATH_STEP * head["slice_path_steps"] / (head["slice_ms"] / 1e3) / 1e9
        prof = slice_kernel_profile()
        traffic = None
        compute_bound = None
        if prof:
            # traffic per launch = measured DRAM bytes per path per launch (ncu) x paths of an average launch of this run
            traffic = prof["dram_bytes_per_path_per_launch"] * n_local
            compute_bound = {k: prof[k] for k in prof if k not in ("dram_bytes_per_path_per_launch",)}
        same = bool(np.allclose(prices_api, head["prices"][0], rtol=1e-12))
        draws = {"fp32": "f32 draws (float Box-Muller on the SFU, 32-bit uniforms)", "fp64": "f64 draws (fp64 Box-Muller, 52-bit uniforms)"}
        line = {"metric": "LogSV MC path-steps/sec", "value": head["value"], "unit": "path-steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64" if args.precision == "fp64" else "f32",
                "dtype_detail": f"{'f64' if args.precision == 'fp64' else 'f32'} state / {draws[args.gauss]}", "data": "synthetic",
                "config": {"workload": WORKLOAD, "paths_per_gpu": n_local, "paths_total": total_paths,
                           "state": args.precision, "gaussians": f"Philox4x32-10 + Box-Muller {args.gauss}",
                           "parallelism": f"paths sharded over {world} GPU(s); 2 fp64 exchanges (16 B, 24*J B) per maturity, "
                                          + ("none needed at N=1" if world == 1 else ("fused into the reduction/payoff kernels over NVLink peer memory"
                                                                                      if use_p2p else "NCCL all-reduce")),
                           "l2": "per-GPU state 3 x paths x 8 B >> 126 MB L2 (inputs larger than L2; no flush needed)"},
                "e2e": {"value": e2e_value, "unit": "path-steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "api": "LogSVPricer.model_mc_price_chain (host numpy in/out through the C ABI)", "same_prices_as_device_arm": same},
                "gpu_launches": head["launches"],
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic,
                             "traffic_source": (prof or {}).get("source", "no parsed ncu capture found (profiles/slice_kernel_metrics.json)"),
                             "kernel": "mc_slice_kernel<LogsvPath>", "peak_source": peak_src,
                             "algorithmic_bytes_per_path_step": ALGO_BYTES_PER_PATH_STEP,
                             "kernel_share_of_step": head["slice_ms"] / (1e3 * head["elapsed_s"]),
                             "kernel_path_steps_per_s": head["slice_path_steps"] / (head["slice_ms"] / 1e3),
                             "note": "effective bandwidth of the reference's streaming dataflow; the fused kernel keeps state in registers, so "
                                     "frac > 1 means the HBM roofline is not what binds it: see compute_bound (one ncu --set full capture "
                                     "per kernel change, parsed into profiles/slice_kernel_metrics.json; not measured in this run)",
                             "compute_bound": compute_bound},
                "clocks": head["clocks"]}
        if "error" in sub:
            line["all_fp64"] = sub
        else:
            key = "all_fp64" if alt_gauss == "fp64" else "f32_draws"
            line[key] = {"dtype_detail": f"{'f64' if args.precision == 'fp64' else 'f32'} state / {draws[alt_gauss]}", "value": sub["value"],
                         "ms_per_step": sub["ms_per_step"], "steps": sub_steps, "e2e": {"value": sub_e2e, "unit": "path-steps/s"},
                         "kernel_path_steps_per_s": sub["slice_path_steps"] / (sub["slice_ms"] / 1e3),
                         "same_prices_as_device_arm": bool(np.allclose(sub_prices_api, sub["prices"][0], rtol=1e-12)),
                         "max_abs_diff_vs_headline_in_se": float(np.max(np.abs(sub["prices"][0] - head["prices"][0]) / head["prices"][1]))}
        if world == 1 and args.gauss == "fp32" and args.precision == "fp64":
            # decomposition of the gap between the two draw modes: the fp64 Box-Muller ARITHMETIC on the default stream's 32-bit uniforms (one
            # Philox call per two steps, |z| <= 6.66 like the float draws) -- what remains to all_fp64 is the second Philox call per two steps
            try:
                mid = device_arm("fp64_paired", 3, 3, False)
                line["f64_box_muller_on_32bit_uniforms"] = {
                    "dtype_detail": "f64 state / f64 Box-Muller arithmetic on 32-bit Philox uniforms (the check mode gauss='fp64_paired')",
                    "value": mid["value"], "ms_per_step": mid["ms_per_step"], "steps": 3}
            except Exception as exc:
                line["f64_box_muller_on_32bit_uniforms"] = {"error": repr(exc)}
        if checks is not None:
            line["checks"] = checks
        # second half of BASELINE.json's metric: price error of the timed MC chain against the Fourier reference (our GPU Fourier route,
        # itself within 1e-10 of the reference CPU path, tests/test_gpu_mgf.py); every one of the 49 strikes
        try:
            fourier = np.concatenate(pricer.price_chain(chain, params))
            fwd = np.concatenate([np.full(int(sizes[m]), chain.forwards[m]) for m in range(len(sizes))])
            err = np.abs(head["prices"][0] - fourier)
            line["price_err_vs_fourier"] = {"max_abs_over_forward": float(np.max(err / fwd)), "max_in_se": float(np.max(err / head["prices"][1])),
                                            "note": "explicit-Euler bias at 25..136 steps per slice dominates at 1e8 paths (DESIGN.md §6): the reference's "
                                                    "own MC carries the same bias, see price_err_vs_reference_mc; north_star abs tolerance 1e-3"}
        except Exception as exc:      # never lose the throughput line over the accuracy annotation
            line["price_err_vs_fourier"] = {"error": str(exc)}
        if extras:
            line["extras"] = extras
        if not args.no_cpu_baseline and world == 1:
            # reference as shipped (Numba, unmodified, oracle/_ref) + the C port, both with effective-core accounting
            ref = numba_reference_block(float(os.environ.get("B200SV_BENCH_CPU_BUDGET_S", 8.0)), 1, fourier=True) \
                if not os.environ.get("B200SV_BENCH_NO_NUMBA") else {"unavailable": "disabled"}
            summary = None if "unavailable" in ref else reference_summary(ref)
            try:
                port = cpu_port_block(chain, params, float(os.environ.get("B200SV_BENCH_CPU_BUDGET_S", 8.0)))
            except Exception as exc:
                port = {"error": repr(exc)}
            if summary is not None:
                line["cpu_baseline"] = dict(summary, port=port)
                # MC vs the REFERENCE'S OWN MC on the same chain / step grid (same Euler bias): z-score per strike
                rp, rs = np.array(ref["mc_prices"]), np.array(ref["mc_stds"])
                z = (head["prices"][0] - rp) / np.sqrt(head["prices"][1] ** 2 + rs ** 2)
                line["price_err_vs_reference_mc"] = {"max_abs_z": float(np.max(np.abs(z))), "mean_z": float(np.mean(z)),
                                                     "frac_within_3_se": float(np.mean(np.abs(z) < 3.0)), "reference_mc_paths": ref["mc_paths"],
                                                     "note": "GPU 1e8-path prices vs the unmodified Numba reference MC pooled over the cpu_baseline run"}
                if "fourier_ms" in ref:
                    fm, fprices = _timed(lambda: np.concatenate(pricer.price_chain(chain, params)), 5)
                    line["fourier_btc_chain"] = {"reference_cpu_ms": ref["fourier_ms"], "b200_ms": 1e3 * fm,
                                                 "max_rel_err_vs_reference": float(np.max(np.abs(fprices / np.array(ref["fourier_prices"]) - 1.0)))}
            else:
                line["cpu_baseline"] = dict(port, numba_reference_unavailable=ref.get("unavailable"))
        print(json.dumps(line), flush=True)
    if world > 1:
        barrier()
        multi_gpu.release_p2p() if hasattr(multi_gpu, "release_p2p") else None
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
