"""Reference-as-shipped CPU arm: the UNMODIFIED stochvolmodels 2.2.0 (Python + Numba) from ``oracle/_ref``.

TEST / MEASUREMENT INFRASTRUCTURE -- imported only by ``bench.py`` (``--impl reference`` and the ``cpu_baseline`` leg) and by
``tests/``; never by the product.

``oracle/_ref`` is produced by the committed recipe ``oracle/install_reference.sh`` (``pip install --no-index --no-deps --target
oracle/_ref`` of a temporary copy of the upstream source tree, run by ``build()``; git-ignored -- nothing here reads the source tree at
run time).  The three third-party packages the reference imports for plotting / implied
vols (matplotlib, seaborn, vanilla_option_pricers) are absent from the image and replaced by ``MagicMock`` modules: none of them is
touched by the timed calls (``LogSVPricer.model_mc_price_chain`` logsv_pricer.py:369-427 -> ``logsv_mc_chain_pricer`` :806-867 ->
``simulate_logsv_x_vol_terminal`` :950-1047 + ``compute_mc_vars_payoff`` mc_payoffs.py:10-88; ``price_chain`` :345-366).

The reference's MC kernels are ``@njit`` without ``parallel=True``: one call = ONE core (SURVEY.md §8d(1)).  The all-cores figure
(§8d(2)) runs one such call per worker process (fork) on distinct ``set_seed`` seeds, nb_path paths each, all started together;
aggregate = workers * nb_path * steps / wall time of the slowest.
"""
from __future__ import annotations

import multiprocessing as mp
import os
import sys
import time
from unittest.mock import MagicMock

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
_STUBS = ("matplotlib", "matplotlib.pyplot", "matplotlib.backends", "matplotlib.backends.backend_pdf", "matplotlib.lines",
          "matplotlib.ticker", "matplotlib.figure", "matplotlib.axes", "matplotlib.dates", "matplotlib.colors", "seaborn",
          "vanilla_option_pricers", "vanilla_option_pricers.bsm", "vanilla_option_pricers.bachelier")


def available() -> str:
    """'' when the reference arm can run here, else the one-line reason."""
    if not os.path.isdir(os.path.join(REF_DIR, "stochvolmodels")):
        return "oracle/_ref/stochvolmodels missing (run oracle/install_reference.sh <StochVolModels source tree>)"
    try:
        import numba  # noqa: F401
    except Exception as e:          # pragma: no cover
        return f"numba not importable: {e}"
    return ""


def import_reference():
    """import the unmodified reference package from oracle/_ref (stubs for the absent plotting / implied-vol packages)."""
    for name in _STUBS:
        sys.modules.setdefault(name, MagicMock())
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import stochvolmodels  # noqa: F401
    mod_file = os.path.abspath(sys.modules["stochvolmodels"].__file__)
    if not mod_file.startswith(REF_DIR):
        raise RuntimeError(f"stochvolmodels resolved to {mod_file}, not to oracle/_ref")
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers import heston_pricer as hp
    from stochvolmodels.data.sample_option_chains import get_btc_test_chain_data
    from stochvolmodels.utils.funcs import set_seed
    return lp, hp, get_btc_test_chain_data, set_seed


def effective_cpus() -> dict:
    """what this process may actually use: affinity mask, cgroup v2/v1 CPU quota, and the min of both (the `cores` the arms report)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:          # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    model = ""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return {"os_cpu_count": os.cpu_count(), "affinity": aff, "cgroup_quota_cpus": quota, "effective": eff, "model": model}


def _mc_once(nb_path: int, nb_steps_per_year: int, seed: int, model: str = "logsv"):
    """one reference call on the BTC chain; returns (seconds, prices list, std errors list)."""
    lp, hp, get_chain, set_seed = import_reference()
    chain = get_chain()
    set_seed(seed)
    if model == "logsv":
        pricer, params = lp.LogSVPricer(), lp.LOGSV_BTC_PARAMS
        t = time.perf_counter()
        prices, stds = pricer.model_mc_price_chain(option_chain=chain, params=params, nb_path=nb_path, nb_steps=nb_steps_per_year)
    else:
        pricer, params = hp.HestonPricer(), hp.BTC_HESTON_PARAMS
        t = time.perf_counter()
        prices, stds = pricer.model_mc_price_chain(option_chain=chain, params=params, nb_path=nb_path)
    return time.perf_counter() - t, [np.asarray(p) for p in prices], [np.asarray(s) for s in stds]


def _worker(args):
    nb_path, nb_steps_per_year, seed, t_start = args
    while time.time() < t_start:            # all workers start together (the parent JIT-compiled before forking: nothing to warm)
        time.sleep(0.001)
    t0 = time.time()
    secs, prices, stds = _mc_once(nb_path, nb_steps_per_year, seed)
    return t0, t0 + secs, secs, np.concatenate(prices), np.concatenate(stds)


def numba_mc_rate(nb_path: int, nb_steps_per_year: int, steps_per_path: int, workers: int = 1, seed: int = 10, warm_paths: int = 2000):
    """time ``LogSVPricer.model_mc_price_chain`` of the reference (warm: called once before to JIT) on the BTC chain.

    workers == 1: in this process, one core (the reference as shipped: its njit kernels are not parallel).  workers > 1: that many
    forked processes (forked AFTER the JIT warm-up, so they inherit the compiled code) each running the same call on nb_path paths with
    distinct ``set_seed`` seeds, started together; aggregate rate = workers * nb_path * steps / (last end - first start).  Returns the
    rate, the pooled prices (mean over workers) and pooled standard errors."""
    _mc_once(warm_paths, nb_steps_per_year, seed)
    if workers <= 1:
        secs, prices, stds = _mc_once(nb_path, nb_steps_per_year, seed)
        return {"value": nb_path * steps_per_path / secs, "seconds": secs, "workers": 1, "paths": nb_path,
                "prices": np.concatenate(prices), "stds": np.concatenate(stds)}
    ctx = mp.get_context("fork")
    with ctx.Pool(workers) as pool:
        t_start = time.time() + 0.5 + 0.01 * workers
        res = pool.map(_worker, [(nb_path, nb_steps_per_year, seed + 1000 * (w + 1), t_start) for w in range(workers)], chunksize=1)
    start = min(r[0] for r in res)
    end = max(r[1] for r in res)
    prices = np.mean([r[3] for r in res], axis=0)
    stds = np.sqrt(np.mean([r[4] ** 2 for r in res], axis=0) / workers)
    return {"value": workers * nb_path * steps_per_path / (end - start), "seconds": end - start, "workers": workers,
            "paths": workers * nb_path, "per_worker_seconds_min_max": [min(r[2] for r in res), max(r[2] for r in res)],
            "prices": prices, "stds": stds}


def numba_fourier_ms(repeat: int = 1):
    """warm wall time (ms) of the reference ``LogSVPricer.price_chain`` on the BTC chain + its prices (SURVEY.md §8d(3))."""
    lp, hp, get_chain, _ = import_reference()
    chain = get_chain()
    pricer, params = lp.LogSVPricer(), lp.LOGSV_BTC_PARAMS
    pricer.price_chain(option_chain=chain, params=params)
    t = time.perf_counter()
    for _ in range(repeat):
        prices = pricer.price_chain(option_chain=chain, params=params)
    return 1e3 * (time.perf_counter() - t) / repeat, np.concatenate([np.asarray(p) for p in prices])


def main(argv=None):
    """CLI used by bench.py in a SUBPROCESS (a clean interpreter: no CUDA context, no torch threads to fork):
        python oracle/ref_arm.py --budget-s 8 --repeat 1 [--workers W] [--fourier]
    prints one JSON object: cpus, one_core {value, paths, seconds}, all_cores [ {value, workers, paths, seconds} x repeat ],
    pooled prices / std errors of everything simulated, optional fourier_ms."""
    import argparse
    import json
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget-s", type=float, default=8.0, help="target seconds per timed call")
    ap.add_argument("--repeat", type=int, default=1, help="number of all-cores runs")
    ap.add_argument("--workers", type=int, default=0, help="0 = effective cpus")
    ap.add_argument("--nb-steps-per-year", type=int, default=582)
    ap.add_argument("--steps-per-path", type=int, default=252)
    ap.add_argument("--fourier", action="store_true")
    ap.add_argument("--no-one-core", action="store_true")
    a = ap.parse_args(argv)
    why = available()
    if why:
        print(json.dumps({"unavailable": why}))
        return
    cpus = effective_cpus()
    workers = a.workers or cpus["effective"]
    out = {"cpus": cpus, "numba": __import__("numba").__version__}
    probe = numba_mc_rate(20_000, a.nb_steps_per_year, a.steps_per_path, 1)        # includes the JIT warm-up
    n1 = int(min(max(a.budget_s * probe["value"] / a.steps_per_path, 2e4), 2e6))
    pool_p, pool_w = [], []
    if not a.no_one_core:
        one = numba_mc_rate(n1, a.nb_steps_per_year, a.steps_per_path, 1)
        out["one_core"] = {k: one[k] for k in ("value", "paths", "seconds")}
        pool_p.append(one["prices"]); pool_w.append((one["stds"], one["paths"]))
    out["all_cores"] = []
    nw = int(min(max(0.6 * n1, 2e4), 1e6))          # per worker: memory-bandwidth contention roughly halves the per-core rate
    for r in range(a.repeat):
        if workers <= 1:
            break
        allc = numba_mc_rate(nw, a.nb_steps_per_year, a.steps_per_path, workers, seed=10 + 7919 * (r + 1))
        out["all_cores"].append({k: allc[k] for k in ("value", "workers", "paths", "seconds", "per_worker_seconds_min_max")})
        pool_p.append(allc["prices"]); pool_w.append((allc["stds"], allc["paths"]))
    # pool everything simulated into one reference-MC estimate (weights = path counts)
    if pool_p:
        w = np.array([n for _, n in pool_w], dtype=float)
        out["mc_prices"] = (np.sum([p * n for p, n in zip(pool_p, w)], axis=0) / w.sum()).tolist()
        out["mc_stds"] = (np.sqrt(np.sum([(s * n) ** 2 for (s, _), n in zip(pool_w, w)], axis=0)) / w.sum()).tolist()
        out["mc_paths"] = int(w.sum())
    if a.fourier:
        ms, prices = numba_fourier_ms()
        out["fourier_ms"] = ms
        out["fourier_prices"] = prices.tolist()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
