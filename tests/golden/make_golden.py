"""Generate the golden fixtures under tests/golden/ by RUNNING THE REFERENCE in this container.

Run (only where /root/reference exists; the GPU box never runs this):

    python tests/golden/make_golden.py

It imports the unmodified reference from /root/reference/src with the three absent
third-party packages (matplotlib, seaborn, vanilla_option_pricers) replaced by
``MagicMock`` modules (they are only touched by plotting / implied-vol code that is
outside the hot path) and stores inputs + outputs of every hot-path function of
SURVEY.md §8(a) as ``.npz`` files.  The fixtures pin ``oracle/`` (CPU restatement) and,
through it and directly, the CUDA path.

Nothing here is imported by the product or by the tests; the tests read only the
``.npz`` files this script wrote.
"""
from __future__ import annotations

import os
import sys
from unittest.mock import MagicMock

import numpy as np

REF_SRC = "/root/reference/src"
OUT = os.path.dirname(os.path.abspath(__file__))


def _import_reference():
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.backends",
                 "matplotlib.backends.backend_pdf", "matplotlib.lines", "matplotlib.ticker",
                 "matplotlib.figure", "matplotlib.axes", "matplotlib.dates", "matplotlib.colors",
                 "seaborn", "vanilla_option_pricers", "vanilla_option_pricers.bsm",
                 "vanilla_option_pricers.bachelier"):
        sys.modules.setdefault(name, MagicMock())
    sys.path.insert(0, REF_SRC)


def main() -> None:
    _import_reference()
    import scipy
    import numba
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers import heston_pricer as hp
    from stochvolmodels.pricers.logsv import affine_expansion as afe
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.utils import mgf_pricer as mgfp
    from stochvolmodels.utils import mc_payoffs as mcp
    from stochvolmodels.utils.funcs import set_time_grid
    from stochvolmodels.utils.config import VariableType
    from stochvolmodels.data.sample_option_chains import get_btc_test_chain_data

    versions = np.array([f"numpy={np.__version__}", f"scipy={scipy.__version__}", f"numba={numba.__version__}"])
    Q = LogSvParams(sigma0=1.0, theta=1.0, kappa1=5.0, kappa2=5.0, beta=0.2, volvol=2.0)
    K5 = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T5 = np.array(['P', 'P', 'C', 'C', 'C'])

    # ------------------------------------------------------------------ a7 set_time_grid
    cases = [(0.25, 252), (0.25, 360), (1.0, 1023), (0.7, 360), (1.0, 252), (0.04289242541152263, 252),
             (0.05833333333333334, 252), (0.0972222222222222, 582), (1.0 / 12.0, 360), (0.02, 360), (1e-3, 360)]
    tg = np.array([[ttm, n, *set_time_grid(ttm, n)[:2]] for ttm, n in cases])
    np.savez(os.path.join(OUT, "time_grid.npz"), cases=tg, versions=versions)

    # ------------------------------------------------------------------ a12 grids and weights
    grids = {}
    for name, vs, spot in (("mma", 0.2041241452319315, True), ("inv", 0.2041241452319315, False), ("dflt", 0.28, True)):
        phi, psi, theta = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, is_spot_measure=spot, vol_scaler=vs)
        grids[f"phi_{name}"] = phi
        grids[f"w_{name}"] = mgfp._compute_legacy_pricer_weights(phi, True)
    grids["vol_scaler_q_025"] = np.array(lp.set_vol_scaler(sigma0=1.0, ttm=0.25))
    grids["vol_scaler_btc"] = np.array(lp.set_vol_scaler(sigma0=0.8376, ttm=0.04289242541152263))
    np.savez(os.path.join(OUT, "grids.npz"), versions=versions, **grids)

    # ------------------------------------------------------------------ a8 M, L, H
    mlh = {}
    phis = np.array([-0.5 + 0.0j, -0.5 + 3.7j, 0.5 + 11.25j, -0.3 + 0.4j])
    psis = np.array([0.0j, 0.0j, 0.0j, -0.5 + 2.0j])
    k = 0
    for order in (afe.ExpansionOrder.FIRST, afe.ExpansionOrder.SECOND):
        for spot in (True, False):
            for eta in (1.0, 0.85):
                for phi, psi in zip(phis, psis):
                    M, L, H = afe.func_a_ode_quadratic_terms(theta=1.0413, kappa1=3.1844, kappa2=3.058, beta=0.1514,
                                                             volvol=1.8458, phi=phi, psi=psi, is_spot_measure=spot,
                                                             expansion_order=order, vol_backbone_eta=eta)
                    mlh[f"case{k}_in"] = np.array([order.value, float(spot), eta, phi.real, phi.imag, psi.real, psi.imag])
                    mlh[f"case{k}_M"], mlh[f"case{k}_L"], mlh[f"case{k}_H"] = M, L, H
                    # one RHS evaluation at a fixed complex state
                    A = (np.arange(1, M.shape[0] + 1) * (0.1 - 0.05j)).astype(np.complex128)
                    mlh[f"case{k}_rhs"] = afe.func_rhs(0.0, A, M, L, H)
                    k += 1
    mlh["ncases"] = np.array(k)
    mlh["params"] = np.array([1.0413, 3.1844, 3.058, 0.1514, 1.8458])
    np.savez(os.path.join(OUT, "mlh.npz"), versions=versions, **mlh)

    # ------------------------------------------------------------------ a9-a11, a13 LogSV Fourier chain
    def fourier_case(tag, params, ttms, forwards, discfactors, strikes_ttms, types_ttms, spot, order=afe.ExpansionOrder.SECOND,
                     backbone=None):
        """run logsv_chain_pricer and ALSO replay its loop to capture a_t1 / log_mgf per maturity."""
        if backbone is not None:
            params.set_vol_backbone(backbone)
        prices = lp.logsv_chain_pricer(params=params, ttms=ttms, forwards=forwards, discfactors=discfactors,
                                       strikes_ttms=strikes_ttms, optiontypes_ttms=types_ttms,
                                       is_spot_measure=spot, expansion_order=order)
        vol_scaler = lp.set_vol_scaler(sigma0=params.sigma0, ttm=np.min(ttms))
        phi, psi, theta = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, is_spot_measure=spot,
                                                      vol_scaler=vol_scaler)
        a_t0 = np.zeros((phi.shape[0], afe.get_expansion_n(order)), dtype=np.complex128)
        ttm0 = 0.0
        out = dict(params=np.array([params.sigma0, params.theta, params.kappa1, params.kappa2, params.beta, params.volvol]),
                   ttms=ttms, forwards=forwards, discfactors=discfactors, is_spot=np.array(spot), order=np.array(order.value),
                   vol_scaler=np.array(vol_scaler), phi=phi, nslices=np.array(len(ttms)))
        etas = []
        for m, ttm in enumerate(ttms):
            eta = params.get_vol_backbone_eta(tau=ttm)
            etas.append(eta)
            a_t0, log_mgf = afe.compute_logsv_a_mgf_grid(ttm=ttm - ttm0, phi_grid=phi, psi_grid=psi, theta_grid=theta,
                                                          a_t0=a_t0, expansion_order=order, is_spot_measure=spot,
                                                          **{kk: vv for kk, vv in params.to_dict().items()},
                                                          vol_backbone_eta=eta)
            out[f"a_t1_{m}"] = a_t0
            out[f"log_mgf_{m}"] = log_mgf
            out[f"strikes_{m}"] = np.asarray(strikes_ttms[m], dtype=float)
            out[f"types_{m}"] = np.asarray(types_ttms[m])
            out[f"prices_{m}"] = np.asarray(prices[m])
            ttm0 = ttm
        out["etas"] = np.array(etas, dtype=float)
        np.savez(os.path.join(OUT, f"logsv_fourier_{tag}.npz"), versions=versions, **out)
        print(tag, [np.asarray(p)[:3] for p in prices])

    # G1: quickstart 3m + 6m
    fourier_case("g1_quickstart", LogSvParams(1.0, 1.0, 5.0, 5.0, 0.2, 2.0), np.array([0.25, 0.5]), np.ones(2), np.ones(2),
                 (K5, K5), (T5, T5), True)
    # G2: inverse measure
    fourier_case("g2_inverse", LogSvParams(1.0, 1.0, 5.0, 5.0, 0.2, 2.0), np.array([0.25]), np.ones(1), np.ones(1),
                 (K5,), (np.array(['IP', 'IP', 'IC', 'IC', 'IC']),), False)
    # C3: 5 maturities x 21 strikes
    K21 = np.linspace(0.5, 1.5, 21)
    T21 = np.where(K21 >= 1.0, 'C', 'P')
    ttms5 = np.array([1.0 / 12.0, 0.25, 0.5, 0.75, 1.0])
    fourier_case("c3_5x21", LogSvParams(1.0, 1.0, 5.0, 5.0, 0.2, 2.0), ttms5, np.ones(5), np.ones(5),
                 tuple(K21 for _ in ttms5), tuple(T21 for _ in ttms5), True)
    # BTC chain with the reference's BTC parameters
    btc = get_btc_test_chain_data()
    fourier_case("btc", LogSvParams(sigma0=0.8376, theta=1.0413, kappa1=3.1844, kappa2=3.058, beta=0.1514, volvol=1.8458),
                 btc.ttms, btc.forwards, btc.discfactors, tuple(btc.strikes_ttms), tuple(btc.optiontypes_ttms), True)
    # FIRST order, discounting, forward != 1, negative beta
    fourier_case("first_order", LogSvParams(sigma0=0.35, theta=0.3, kappa1=2.0, kappa2=1.5, beta=-0.6, volvol=0.9),
                 np.array([0.1, 0.6]), np.array([100.0, 101.5]), np.array([0.995, 0.97]),
                 (np.array([80.0, 100.0, 125.0]), np.array([70.0, 95.0, 101.5, 140.0])),
                 (np.array(['P', 'C', 'C']), np.array(['P', 'P', 'C', 'C'])), True, order=afe.ExpansionOrder.FIRST)
    # vol backbone (eta != 1) under the inverse measure, SECOND order
    import pandas as pd
    fourier_case("backbone_inverse", LogSvParams(sigma0=0.8, theta=1.0, kappa1=3.0, kappa2=3.0, beta=0.15, volvol=1.5),
                 np.array([0.1, 0.3]), np.array([1.0, 1.0]), np.array([1.0, 1.0]),
                 (K5, K5), (np.array(['IP', 'IP', 'IC', 'C', 'P']), np.array(['IP', 'IP', 'IC', 'IC', 'IC'])), False,
                 backbone=pd.Series([0.9, 1.1], index=[0.1, 0.3]))

    # ------------------------------------------------------------------ a14 Heston Fourier
    def heston_case(tag, v0, theta, kappa, volvol, rho, ttms, forwards, discfactors, strikes_ttms, types_ttms):
        prices = hp.heston_chain_pricer(v0=v0, theta=theta, kappa=kappa, volvol=volvol, rho=rho, ttms=ttms, forwards=forwards,
                                        strikes_ttms=strikes_ttms, optiontypes_ttms=types_ttms, discfactors=discfactors)
        vol_scaler = np.minimum(0.3, np.sqrt(v0 * ttms[0]))
        phi, psi, _ = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, vol_scaler=vol_scaler)
        out = dict(params=np.array([v0, theta, kappa, rho, volvol]), ttms=ttms, forwards=forwards, discfactors=discfactors,
                   vol_scaler=np.array(vol_scaler), phi=phi, nslices=np.array(len(ttms)))
        a_t0 = np.zeros(phi.shape[0], dtype=np.complex128)
        b_t0 = np.zeros(phi.shape[0], dtype=np.complex128)
        ttm0 = 0.0
        for m, ttm in enumerate(ttms):
            log_mgf, a_t0, b_t0 = hp.compute_heston_mgf_grid(ttm=ttm - ttm0, v0=v0, theta=theta, kappa=kappa, volvol=volvol, rho=rho,
                                                             phi_grid=phi, psi_grid=psi, a_t0=a_t0, b_t0=b_t0)
            out[f"log_mgf_{m}"], out[f"a_t1_{m}"], out[f"b_t1_{m}"] = log_mgf, a_t0, b_t0
            out[f"strikes_{m}"] = np.asarray(strikes_ttms[m], dtype=float)
            out[f"types_{m}"] = np.asarray(types_ttms[m])
            out[f"prices_{m}"] = np.asarray(prices[m])
            ttm0 = ttm
        np.savez(os.path.join(OUT, f"heston_fourier_{tag}.npz"), versions=versions, **out)
        print("heston", tag, [np.asarray(p)[:3] for p in prices])

    heston_case("g4", 0.04, 0.04, 4.0, 0.4, -0.5, np.array([0.25, 1.0]), np.ones(2), np.ones(2), (K5, K5), (T5, T5))
    heston_case("c3_5x21", 0.04, 0.04, 4.0, 0.4, -0.5, ttms5, np.ones(5), np.ones(5),
                tuple(K21 for _ in ttms5), tuple(T21 for _ in ttms5))
    heston_case("btc", 0.8, 1.0, 2.0, 2.0, 0.0, btc.ttms, btc.forwards, np.array([0.999, 0.998, 0.996, 0.99]),
                tuple(btc.strikes_ttms), tuple(btc.optiontypes_ttms))

    # ------------------------------------------------------------------ a1-a3 LogSV MC with fixed randoms
    def mc_fixed_case(tag, params, ttms, forwards, discfactors, strikes_ttms, types_ttms, etas, spot, nb_path, n_per_year, seed,
                      variable_type=VariableType.LOG_RETURN):
        W0s, W1s, dts = lp.get_randoms_for_chain_valuation(ttms=ttms, nb_path=nb_path, nb_steps_per_year=n_per_year, seed=seed)
        prices, stds = lp.logsv_mc_chain_pricer_fixed_randoms(ttms=ttms, forwards=forwards, discfactors=discfactors,
                                                              strikes_ttms=strikes_ttms, optiontypes_ttms=types_ttms,
                                                              W0s=W0s, W1s=W1s, dts=dts, v0=params.sigma0, theta=params.theta,
                                                              kappa1=params.kappa1, kappa2=params.kappa2, beta=params.beta,
                                                              volvol=params.volvol, vol_backbone_etas=etas, is_spot_measure=spot,
                                                              variable_type=variable_type)
        out = dict(params=np.array([params.sigma0, params.theta, params.kappa1, params.kappa2, params.beta, params.volvol]),
                   ttms=ttms, forwards=forwards, discfactors=discfactors, etas=etas, is_spot=np.array(spot),
                   nb_path=np.array(nb_path), n_per_year=np.array(n_per_year), seed=np.array(seed),
                   variable_type=np.array(variable_type.value), nslices=np.array(len(ttms)),
                   dts=np.array(list(dts)), nsteps=np.array([w.shape[0] for w in W0s]), W0_head=np.asarray(W0s[0])[0, :3])
        # replay slice by slice for terminal states
        x0 = np.zeros(nb_path); q0 = np.zeros(nb_path); s0 = params.sigma0 * np.ones(nb_path); ttm0 = 0.0
        for m, ttm in enumerate(ttms):
            x0, s0, q0 = lp.simulate_logsv_x_vol_terminal(ttm=ttm - ttm0, x0=x0, sigma0=s0, qvar0=q0, theta=params.theta,
                                                           kappa1=params.kappa1, kappa2=params.kappa2, beta=params.beta,
                                                           volvol=params.volvol, vol_backbone_eta=etas[m], nb_path=nb_path,
                                                           dt=dts[m], is_spot_measure=spot, W0=W0s[m], W1=W1s[m])
            ttm0 = ttm
            out[f"x_{m}"], out[f"sigma_{m}"], out[f"qvar_{m}"] = x0.copy(), s0.copy(), q0.copy()
            out[f"strikes_{m}"] = np.asarray(strikes_ttms[m], dtype=float)
            out[f"types_{m}"] = np.asarray(types_ttms[m])
            out[f"prices_{m}"], out[f"stderr_{m}"] = np.asarray(prices[m]), np.asarray(stds[m])
        np.savez(os.path.join(OUT, f"logsv_mc_fixed_{tag}.npz"), versions=versions, **out)
        print("mc", tag, np.asarray(prices[0])[:3], np.asarray(stds[0])[:3])

    mc_fixed_case("g5_c1", Q, np.array([0.25]), np.ones(1), np.ones(1), (K5,), (T5,), np.ones(1), True, 10000, 252, 10)
    mc_fixed_case("inverse_eta", LogSvParams(0.8376, 1.0413, 3.1844, 3.058, 0.1514, 1.8458), np.array([0.1, 0.3]),
                  np.array([1.0, 1.02]), np.array([0.999, 0.99]), (K5, K5),
                  (np.array(['IP', 'IP', 'IC', 'IC', 'IC']), np.array(['IP', 'P', 'C', 'IC', 'IC'])),
                  np.array([0.9, 1.1]), False, 4000, 360, 3)
    mc_fixed_case("btc_small", LogSvParams(0.8376, 1.0413, 3.1844, 3.058, 0.1514, 1.8458), btc.ttms, btc.forwards, btc.discfactors,
                  tuple(btc.strikes_ttms), tuple(btc.optiontypes_ttms), np.ones(4), True, 5000, 252, 11)
    mc_fixed_case("qvar", Q, np.array([0.25, 0.5]), np.ones(2), np.ones(2),
                  (np.array([0.5, 1.0, 1.5]), np.array([0.5, 1.0, 1.5])), (np.array(['P', 'C', 'C']), np.array(['P', 'C', 'C'])),
                  np.ones(2), True, 3000, 252, 5, variable_type=VariableType.Q_VAR)

    # ------------------------------------------------------------------ a6 Heston MC stepper (py_func + numpy global seed)
    def heston_mc_case(tag, v0, theta, kappa, rho, volvol, ttm, nb_path, seed):
        np.random.seed(seed)
        x, v, q = hp.simulate_heston_x_vol_terminal.py_func(ttm=ttm, x0=np.zeros(nb_path), var0=v0 * np.ones(nb_path),
                                                            qvar0=np.zeros(nb_path), theta=theta, kappa=kappa, rho=rho,
                                                            volvol=volvol, nb_path=nb_path)
        S, dt, _ = set_time_grid(ttm, 360)
        prices, stds = mcp.compute_mc_vars_payoff(x0=x, sigma0=np.sqrt(v), qvar0=q, ttm=ttm, forward=1.0, strikes_ttm=K5,
                                                  optiontypes_ttm=T5, discfactor=0.98)
        np.savez(os.path.join(OUT, f"heston_mc_fixed_{tag}.npz"), versions=versions,
                 params=np.array([v0, theta, kappa, rho, volvol]), ttm=np.array(ttm), nb_path=np.array(nb_path),
                 seed=np.array(seed), nsteps=np.array(S), dt=np.array(dt), x=x, var=v, qvar=q, strikes=K5, types=T5,
                 forward=np.array(1.0), discfactor=np.array(0.98), prices=prices, stderr=stds)
        print("heston mc", tag, prices[:3], "min v", v.min())

    heston_mc_case("dflt", 0.04, 0.04, 4.0, -0.5, 0.4, 0.7, 5000, 7)
    heston_mc_case("floor", 0.01, 0.02, 1.0, -0.7, 1.0, 0.5, 4000, 8)   # Feller violated: the 1e-4 floor binds

    # ------------------------------------------------------------------ a5 payoffs: all four codes, Q_VAR, NaN paths
    # NaN-free inputs go through the COMPILED reference.  Inputs with NaN paths go through ``.py_func`` (the Python
    # source semantics: np.nanmean / np.nanstd skip NaN paths): the compiled function is ``fastmath=True`` (LLVM
    # assumes no NaNs) and returns NaN / garbage for such inputs, so only the source-level behaviour can be pinned.
    rng = np.random.RandomState(42)
    x = 0.3 * rng.normal(size=2000) - 0.05
    qv = 0.1 * np.abs(rng.normal(size=2000)) + 0.01
    strikes = np.array([0.7, 0.9, 1.0, 1.1, 1.3, 1.0, 0.95, 1.05])
    types = np.array(['P', 'P', 'C', 'C', 'C', 'IC', 'IP', 'IC'])
    qstrikes = np.array([0.1, 0.2, 0.3, 0.2])
    qtypes = np.array(['P', 'C', 'C', 'IC'])
    kw = dict(sigma0=np.ones_like(x), ttm=0.5, forward=1.03, discfactor=0.97)
    p1, s1 = mcp.compute_mc_vars_payoff(x0=x, qvar0=qv, strikes_ttm=strikes, optiontypes_ttm=types,
                                        variable_type=VariableType.LOG_RETURN, **kw)
    p2, s2 = mcp.compute_mc_vars_payoff(x0=x, qvar0=qv, strikes_ttm=qstrikes, optiontypes_ttm=qtypes,
                                        variable_type=VariableType.Q_VAR, **kw)
    xn = x.copy()
    xn[[3, 77, 500]] = np.nan
    p3, s3 = mcp.compute_mc_vars_payoff.py_func(x0=xn, qvar0=qv, strikes_ttm=strikes, optiontypes_ttm=types,
                                                variable_type=VariableType.LOG_RETURN, **kw)
    p4, s4 = mcp.compute_mc_vars_payoff.py_func(x0=xn, qvar0=qv, strikes_ttm=qstrikes, optiontypes_ttm=qtypes,
                                                variable_type=VariableType.Q_VAR, **kw)
    np.savez(os.path.join(OUT, "payoffs.npz"), versions=versions, x=x, x_nan=xn, qvar=qv, ttm=np.array(0.5), forward=np.array(1.03),
             discfactor=np.array(0.97), strikes=strikes, types=types, prices=p1, stderr=s1,
             qstrikes=qstrikes, qtypes=qtypes, qprices=p2, qstderr=s2,
             prices_nan=p3, stderr_nan=s3, qprices_nan=p4, qstderr_nan=s4)

    # ------------------------------------------------------------------ a13 Fourier sum on a closed-form (lognormal) MGF
    vol, ttm = 0.3, 0.4
    for spot, tag in ((True, "mma"), (False, "inv")):
        phi, _, _ = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, is_spot_measure=spot,
                                                vol_scaler=vol * np.sqrt(ttm))
        sgn = 1.0 if spot else -1.0
        log_mgf = 0.5 * vol * vol * ttm * (phi * phi + sgn * phi)
        types = np.array(['P', 'P', 'C', 'C', 'C']) if spot else np.array(['IP', 'P', 'C', 'IC', 'IC'])
        prices = mgfp.vanilla_slice_pricer_with_mgf_grid(log_mgf_grid=log_mgf, phi_grid=phi, forward=1.5, strikes=1.5 * K5,
                                                         optiontypes=types, discfactor=0.9, is_spot_measure=spot)
        np.savez(os.path.join(OUT, f"fourier_sum_{tag}.npz"), versions=versions, phi=phi, log_mgf=log_mgf, forward=np.array(1.5),
                 strikes=1.5 * K5, types=types, discfactor=np.array(0.9), is_spot=np.array(spot), prices=prices)

    print("golden fixtures written to", OUT)


def reference_mc():
    """Large-N Monte Carlo prices from the REFERENCE's own Numba stepper + payoff code (seeded through its ``set_seed``):
    the statistical anchor for the GPU Philox path ("within 3 MC standard errors of the reference Numba CPU path").
    The Euler scheme carries a discretisation bias against the Fourier price that is visible at these path counts
    (|z| ~ 4 at 2e6 paths with ANY generator), so MC-vs-MC is the meaningful 3-SE comparison.
    Paths are simulated in chunks (the reference materialises W0/W1[steps, paths]) and the payoffs are taken once on the
    concatenated terminal states, so the forward re-centring is global exactly as in one big call."""
    _import_reference()
    import scipy
    import numba
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers import heston_pricer as hp
    from stochvolmodels.utils import mc_payoffs as mcp
    from stochvolmodels.utils.funcs import set_seed
    from stochvolmodels.data.sample_option_chains import get_btc_test_chain_data
    versions = np.array([f"numpy={np.__version__}", f"scipy={scipy.__version__}", f"numba={numba.__version__}"])
    K5 = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T5 = np.array(['P', 'P', 'C', 'C', 'C'])

    def logsv_case(tag, p6, ttms, forwards, discfactors, strikes_ttms, types_ttms, n_per_year, nb_path, chunk, seed):
        set_seed(seed)
        M = len(ttms)
        xs = [[] for _ in range(M)]
        qs = [[] for _ in range(M)]
        for c in range(nb_path // chunk):
            x = np.zeros(chunk); q = np.zeros(chunk); s = p6[0] * np.ones(chunk); t0 = 0.0
            for m, ttm in enumerate(ttms):
                x, s, q = lp.simulate_logsv_x_vol_terminal(ttm=ttm - t0, x0=x, sigma0=s, qvar0=q, theta=p6[1], kappa1=p6[2], kappa2=p6[3],
                                                           beta=p6[4], volvol=p6[5], nb_path=chunk, nb_steps_per_year=n_per_year)
                t0 = ttm
                xs[m].append(x.copy()); qs[m].append(q.copy())
        out = dict(params=np.array(p6), ttms=ttms, forwards=forwards, discfactors=discfactors, n_per_year=np.array(n_per_year),
                   nb_path=np.array(nb_path), seed=np.array(seed), nslices=np.array(M))
        for m in range(M):
            x, q = np.concatenate(xs[m]), np.concatenate(qs[m])
            pr, se = mcp.compute_mc_vars_payoff(x0=x, sigma0=x, qvar0=q, ttm=ttms[m], forward=forwards[m], strikes_ttm=strikes_ttms[m],
                                                optiontypes_ttm=types_ttms[m], discfactor=discfactors[m])
            out[f"strikes_{m}"], out[f"types_{m}"], out[f"prices_{m}"], out[f"stderr_{m}"] = strikes_ttms[m], types_ttms[m], pr, se
            out[f"mean_exp_x_{m}"] = np.array(np.mean(np.exp(x)))
            out[f"mean_qvar_{m}"] = np.array(np.mean(q))
            print("refmc", tag, m, pr[:3], se[:3])
        np.savez(os.path.join(OUT, f"refmc_logsv_{tag}.npz"), versions=versions, **out)

    which = [a.split("=")[1] for a in sys.argv if a.startswith("--case=")]
    if not which or "quickstart" in which:
        logsv_case("quickstart", (1.0, 1.0, 5.0, 5.0, 0.2, 2.0), np.array([0.25, 0.5]), np.ones(2), np.ones(2), (K5, K5), (T5, T5),
                   252, 16_000_000, 500_000, 1234)
    if not which or "btc" in which:
        btc = get_btc_test_chain_data()
        logsv_case("btc", (0.8376, 1.0413, 3.1844, 3.058, 0.1514, 1.8458), btc.ttms, btc.forwards, btc.discfactors,
                   tuple(btc.strikes_ttms), tuple(btc.optiontypes_ttms), 252, 16_000_000, 500_000, 4321)
    if which and "heston" not in which:
        return

    # Heston: reference stepper is hard-wired to 360 steps/yr
    set_seed(99)
    ttms = np.array([0.25, 1.0])
    nb_path, chunk = 8_000_000, 250_000
    xs = [[], []]
    for c in range(nb_path // chunk):
        x = np.zeros(chunk); q = np.zeros(chunk); v = 0.04 * np.ones(chunk); t0 = 0.0
        for m, ttm in enumerate(ttms):
            x, v, q = hp.simulate_heston_x_vol_terminal(ttm=ttm - t0, x0=x, var0=v, qvar0=q, theta=0.04, kappa=4.0, rho=-0.5, volvol=0.4,
                                                        nb_path=chunk)
            t0 = ttm
            xs[m].append(x.copy())
    out = dict(params=np.array([0.04, 0.04, 4.0, -0.5, 0.4]), ttms=ttms, nb_path=np.array(nb_path), nslices=np.array(2))
    for m in range(2):
        x = np.concatenate(xs[m])
        pr, se = mcp.compute_mc_vars_payoff(x0=x, sigma0=x, qvar0=x, ttm=ttms[m], forward=1.0, strikes_ttm=K5, optiontypes_ttm=T5)
        out[f"strikes_{m}"], out[f"types_{m}"], out[f"prices_{m}"], out[f"stderr_{m}"] = K5, T5, pr, se
        print("refmc heston", m, pr, se)
    np.savez(os.path.join(OUT, "refmc_heston_g4.npz"), versions=versions, **out)


def next_rows():
    """SURVEY.md §8f #3: Q_VAR / density / digital Fourier routes (psi grid P = 40000, theta grid P = 5000)."""
    _import_reference()
    import scipy
    import numba
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers import heston_pricer as hp
    from stochvolmodels.pricers.logsv import affine_expansion as afe
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.utils import mgf_pricer as mgfp
    from stochvolmodels.utils.config import VariableType
    versions = np.array([f"numpy={np.__version__}", f"scipy={scipy.__version__}", f"numba={numba.__version__}"])
    Q = LogSvParams(sigma0=1.0, theta=1.0, kappa1=5.0, kappa2=5.0, beta=0.2, volvol=2.0)
    p6 = np.array([1.0, 1.0, 5.0, 5.0, 0.2, 2.0])

    # ---- LogSV options on quadratic variance, both measures (logsv_pricer.py:723-731 -> mgf_pricer.py:323-358)
    ttms = np.array([0.25, 0.5])
    kq = np.array([0.5, 0.8, 1.0, 1.2, 1.6])
    tq = np.array(['C'] * 5)
    for spot, tag in ((True, "mma"), (False, "inv")):
        prices = lp.logsv_chain_pricer(params=Q, ttms=ttms, forwards=np.ones(2), discfactors=np.array([1.0, 0.98]),
                                       strikes_ttms=(kq, kq), optiontypes_ttms=(tq, tq), is_spot_measure=spot,
                                       variable_type=VariableType.Q_VAR)
        phi, psi, theta = mgfp.get_transform_var_grid(variable_type=VariableType.Q_VAR, is_spot_measure=spot)
        out = dict(params=p6, ttms=ttms, discfactors=np.array([1.0, 0.98]), strikes=kq, is_spot=np.array(spot), psi_head=psi[:4],
                   psi_tail=psi[-2:], phi0=phi[0], npsi=np.array(psi.shape[0]))
        a = np.zeros((psi.shape[0], 5), dtype=np.complex128)
        t0 = 0.0
        for m, ttm in enumerate(ttms):
            a, lm = afe.compute_logsv_a_mgf_grid(ttm=ttm - t0, phi_grid=phi, psi_grid=psi, theta_grid=theta, a_t0=a,
                                                 is_spot_measure=spot, **Q.to_dict())
            t0 = ttm
            out[f"a_sub_{m}"], out[f"log_mgf_sub_{m}"], out[f"prices_{m}"] = a[::40].copy(), lm[::40].copy(), np.asarray(prices[m])
        np.savez(os.path.join(OUT, f"logsv_fourier_qvar_{tag}.npz"), versions=versions, **out)
        print("qvar", tag, [np.asarray(p_) for p_ in prices])

    # ---- densities (logsv_pricer.py:742-803 -> mgf_pricer.py:361-384)
    grids = {"LOG_RETURN": np.linspace(-2.0, 1.5, 71), "Q_VAR": np.linspace(0.02, 3.0, 60), "SIGMA": np.linspace(0.05, 3.0, 60)}
    out = dict(params=p6, ttm=np.array(0.25))
    for vt in (VariableType.LOG_RETURN, VariableType.Q_VAR, VariableType.SIGMA):
        pdf = lp.logsv_pdfs(params=Q, ttm=0.25, space_grid=grids[vt.name], variable_type=vt)
        out[f"grid_{vt.name}"], out[f"pdf_{vt.name}"] = grids[vt.name], pdf
        print("pdf", vt.name, pdf[:3], pdf.sum())
    np.savez(os.path.join(OUT, "logsv_pdfs.npz"), versions=versions, **out)

    # ---- Heston options on quadratic variance (heston_pricer.py:217-282 with Q_VAR)
    prices = hp.heston_chain_pricer(v0=0.04, theta=0.04, kappa=4.0, volvol=0.4, rho=-0.5, ttms=ttms, forwards=np.ones(2),
                                    strikes_ttms=(0.04 * kq, 0.04 * kq), optiontypes_ttms=(tq, tq), discfactors=np.array([1.0, 0.98]),
                                    variable_type=VariableType.Q_VAR)
    np.savez(os.path.join(OUT, "heston_fourier_qvar.npz"), versions=versions, params=np.array([0.04, 0.04, 4.0, -0.5, 0.4]), ttms=ttms,
             discfactors=np.array([1.0, 0.98]), strikes=0.04 * kq, prices_0=np.asarray(prices[0]), prices_1=np.asarray(prices[1]))
    print("heston qvar", [np.asarray(p_) for p_ in prices])

    # ---- digitals on a closed-form lognormal MGF (mgf_pricer.py:224-269), both signs of Re(phi)
    vol, ttm = 0.3, 0.4
    K5 = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T5 = np.array(['P', 'P', 'C', 'C', 'C'])
    for spot, tag in ((True, "neg"), (False, "pos")):
        phi, _, _ = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, is_spot_measure=spot, vol_scaler=vol * np.sqrt(ttm))
        log_mgf = 0.5 * vol * vol * ttm * (phi * phi + phi)
        prices = mgfp.digital_slice_pricer_with_mgf_grid(log_mgf_grid=log_mgf, phi_grid=phi, forward=1.5, strikes=1.5 * K5,
                                                         optiontypes=T5, discfactor=0.9)
        np.savez(os.path.join(OUT, f"fourier_digital_{tag}.npz"), versions=versions, phi=phi, log_mgf=log_mgf, forward=np.array(1.5),
                 strikes=1.5 * K5, types=T5, discfactor=np.array(0.9), prices=prices)
        print("digital", tag, prices)


def vol_paths():
    """SURVEY.md §8f #4a: simulate_vol_paths with caller-supplied scaled increments (pricers/logsv_pricer.py:870-947)."""
    _import_reference()
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.utils.funcs import set_time_grid
    out = {}
    for tag, spot in (("mma", True), ("inv", False)):
        S, dt, grid = set_time_grid(0.1, 360)
        W = np.sqrt(dt) * np.random.RandomState(5).normal(0, 1, size=(S, 500))
        sig, grid_t = lp.simulate_vol_paths(ttm=0.1, v0=0.8376, theta=1.0413, kappa1=3.1844, kappa2=3.058, beta=0.1514, volvol=1.8458,
                                            is_spot_measure=spot, nb_path=500, nb_steps_per_year=360, brownians=W)
        out[f"sigma_t_{tag}"], out[f"grid_t_{tag}"] = sig, grid_t
    out["params"] = np.array([0.8376, 1.0413, 3.1844, 3.058, 0.1514, 1.8458])
    # the class method: nb_steps=None -> per-year rate ceil(year_days*ttm) (logsv_pricer.py:574)
    sig, grid_t = lp.LogSVPricer().simulate_vol_paths(params=lp.LOGSV_BTC_PARAMS, ttm=0.02, nb_path=4)
    out["method_shape"] = np.array(sig.shape)
    out["method_grid"] = grid_t
    np.savez(os.path.join(OUT, "logsv_vol_paths.npz"), **out)
    print("vol paths", out["sigma_t_mma"].shape, out["method_shape"])


def calibration() -> None:
    """goldens for the calibration drivers (SURVEY.md §8f #2): the reference's own ``calibrate_model_params_to_chain`` (SLSQP, scipy
    finite differences, CPU pricer) on a synthetic market generated by the reference pricer.  The third-party Black helpers the
    reference imports (``vanilla_option_pricers.bsm``: implied vols, vegas) are absent from the reference tree; a shim built on
    ``oracle/bsm.py`` stands in for them, so these goldens pin the DRIVER + PRICER, not the third-party inversion.
    Run:  python tests/golden/make_golden.py --only-calib"""
    import types
    sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
    from oracle import bsm as obsm
    shim = types.ModuleType("vanilla_option_pricers.bsm")
    shim.infer_bsm_ivols_from_model_chain_prices = obsm.infer_bsm_ivols_from_model_chain_prices

    def compute_bsm_vegas_ttms(ttms, forwards, strikes_ttms, optiontypes_ttms, vols_ttms):
        out = []
        for ttm, forward, strikes, vols in zip(ttms, forwards, strikes_ttms, vols_ttms):
            sdev = vols * np.sqrt(ttm)
            d1 = np.log(forward / strikes) / sdev + 0.5 * sdev
            out.append(forward * np.exp(-0.5 * d1 * d1) / np.sqrt(2.0 * np.pi) * np.sqrt(ttm))
        return out
    shim.compute_bsm_vegas_ttms = compute_bsm_vegas_ttms

    def compute_bsm_vanilla_slice_prices(ttm, forward, strikes, vols, optiontypes, discfactor=1.0):
        return np.array([obsm.compute_bsm_vanilla_price(forward, k, ttm, v, str(t), discfactor) for k, v, t in zip(strikes, vols, optiontypes)])
    shim.compute_bsm_vanilla_slice_prices = compute_bsm_vanilla_slice_prices
    pkg = MagicMock()          # the reference does `import vanilla_option_pricers as bsm`: the two functions it needs live on the package
    pkg.infer_bsm_ivols_from_model_chain_prices = shim.infer_bsm_ivols_from_model_chain_prices
    pkg.compute_bsm_vegas_ttms = shim.compute_bsm_vegas_ttms
    pkg.compute_bsm_vanilla_slice_prices = shim.compute_bsm_vanilla_slice_prices
    sys.modules["vanilla_option_pricers"] = pkg
    sys.modules["vanilla_option_pricers.bsm"] = shim
    sys.modules["vanilla_option_pricers.bachelier"] = MagicMock()
    _import_reference()
    import time
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers import heston_pricer as hp
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.data.option_chain import OptionChain

    ttms = np.array([1.0 / 12.0, 0.25])
    forwards = np.array([1.0, 1.0])
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    types_ = np.array(["P", "P", "C", "C", "C"])

    def chain_with(vols):
        return OptionChain(ttms=ttms, ids=np.array(["1m", "3m"]), forwards=forwards, strikes_ttms=[K, K], optiontypes_ttms=[types_, types_],
                           bid_ivs=[v.copy() for v in vols], ask_ivs=[v.copy() for v in vols])

    flat = chain_with([0.8 * np.ones(5), 0.8 * np.ones(5)])
    # ---- LogSV, PARAMS4, analytic engine
    truth = LogSvParams(sigma0=0.9, theta=1.0, kappa1=4.0, kappa2=4.0, beta=0.3, volvol=1.5)
    pricer = lp.LogSVPricer()
    market = pricer.compute_model_ivols_for_chain(option_chain=flat, params=truth, vol_scaler=pricer.set_vol_scaler(option_chain=flat))
    chain = chain_with([np.asarray(v) for v in market])
    start = LogSvParams(sigma0=0.8, theta=0.9, kappa1=4.0, kappa2=4.0, beta=0.1, volvol=1.2)
    t = time.time()
    fit = pricer.calibrate_model_params_to_chain(option_chain=chain, params0=start,
                                                 model_calibration_type=lp.LogsvModelCalibrationType.PARAMS4,
                                                 constraints_type=lp.ConstraintsType.UNCONSTRAINT)
    secs = time.time() - t
    fit_vols = pricer.compute_model_ivols_for_chain(option_chain=chain, params=fit, vol_scaler=pricer.set_vol_scaler(option_chain=chain))
    print("logsv fit", fit, f"{secs:.1f}s")
    np.savez(os.path.join(OUT, "calib_logsv_params4.npz"), ttms=ttms, forwards=forwards, strikes=K, types=types_,
             market_vols=np.array(market), truth=np.array([truth.sigma0, truth.theta, truth.kappa1, truth.kappa2, truth.beta, truth.volvol]),
             start=np.array([start.sigma0, start.theta, start.kappa1, start.kappa2, start.beta, start.volvol]),
             fit=np.array([fit.sigma0, fit.theta, fit.kappa1, fit.kappa2, fit.beta, fit.volvol]), fit_vols=np.array(fit_vols),
             vol_scaler=np.array(pricer.set_vol_scaler(option_chain=chain)), ref_seconds=np.array(secs))
    # ---- LogSV, PARAMS_WITH_VARSWAP_FIT (beta, volvol; eta backbone re-fitted to the chain's var-swap strikes at every point)
    if "--skip-varswap" not in sys.argv:
        from stochvolmodels.pricers.logsv import vol_moments_ode as vmo
        K9 = np.linspace(0.6, 1.4, 9)
        T9 = np.where(K9 >= 1.0, "C", "P")
        ttms3 = np.array([0.04, 0.25, 0.5])

        def chain9(vols):
            return OptionChain(ttms=ttms3, ids=np.array(["2w", "3m", "6m"]), forwards=np.ones(3), strikes_ttms=[K9] * 3, optiontypes_ttms=[T9] * 3,
                               bid_ivs=[v.copy() for v in vols], ask_ivs=[v.copy() for v in vols])
        flat9 = chain9([0.8 * np.ones(9)] * 3)
        market9 = pricer.compute_model_ivols_for_chain(option_chain=flat9, params=truth, vol_scaler=pricer.set_vol_scaler(option_chain=flat9))
        c9 = chain9([np.asarray(v) * s for v, s in zip(market9, (1.05, 1.0, 0.97))])        # tilt the term structure so that eta != 1
        vs = c9.get_slice_varswap_strikes(floor_with_atm_vols=True)
        vs_raw = c9.get_slice_varswap_strikes(floor_with_atm_vols=False)
        start2 = LogSvParams(sigma0=0.9, theta=1.0, kappa1=4.0, kappa2=4.0, beta=0.1, volvol=1.2)
        eta0 = vmo.fit_model_vol_backbone_to_varswaps(log_sv_params=start2, varswap_strikes=vs)
        moments = np.array([vmo.compute_analytic_vol_moments(params=start2, t=t_, n_terms=4) for t_ in (0.0, 0.04, 0.5, 2.0)])
        int_moments = np.array([vmo.compute_analytic_vol_moments(params=start2, t=t_, n_terms=4, is_qvar=True) for t_ in (0.04, 0.5, 2.0)])
        qvars = np.array([vmo.compute_analytic_qvar(params=start2, ttm=t_) for t_ in (0.0, 0.04, 0.25, 0.5, 2.0)])
        t = time.time()
        fit2 = pricer.calibrate_model_params_to_chain(option_chain=c9, params0=start2,
                                                      model_calibration_type=lp.LogsvModelCalibrationType.PARAMS_WITH_VARSWAP_FIT)
        secs2 = time.time() - t
        fit2_vols = pricer.compute_model_ivols_for_chain(option_chain=c9, params=fit2, vol_scaler=pricer.set_vol_scaler(option_chain=c9))
        print("logsv varswap fit", fit2, f"{secs2:.1f}s")
        np.savez(os.path.join(OUT, "calib_logsv_varswap.npz"), ttms=ttms3, forwards=np.ones(3), strikes=K9, types=T9,
                 market_vols=np.array([np.asarray(v) for v in c9.get_mid_vols()]), start=np.array([0.9, 1.0, 4.0, 4.0, 0.1, 1.2]),
                 varswap_strikes=vs.to_numpy(), varswap_strikes_raw=vs_raw.to_numpy(), eta_start=eta0.to_numpy(),
                 lambda4=start2.get_vol_moments_lambda(n_terms=4), moments=moments, int_moments=int_moments, qvars=qvars,
                 fit=np.array([fit2.sigma0, fit2.theta, fit2.kappa1, fit2.kappa2, fit2.beta, fit2.volvol]),
                 fit_eta=fit2.vol_backbone.to_numpy(), fit_vols=np.array(fit2_vols), ref_seconds=np.array(secs2))
        if "--only-varswap" in sys.argv:
            return
    # ---- Heston
    htruth = hp.HestonParams(v0=0.7, theta=0.9, kappa=3.0, rho=-0.3, volvol=1.2)
    hpr = hp.HestonPricer()
    hmarket = hpr.compute_model_ivols_for_chain(option_chain=flat, params=htruth)
    hchain = chain_with([np.asarray(v) for v in hmarket])
    hstart = hp.HestonParams(v0=0.5, theta=0.7, kappa=2.0, rho=-0.1, volvol=1.0)
    t = time.time()
    hfit = hpr.calibrate_model_params_to_chain(option_chain=hchain, params0=hstart)
    hsecs = time.time() - t
    hfit_vols = hpr.compute_model_ivols_for_chain(option_chain=hchain, params=hfit)
    print("heston fit", hfit, f"{hsecs:.1f}s")
    np.savez(os.path.join(OUT, "calib_heston.npz"), ttms=ttms, forwards=forwards, strikes=K, types=types_, market_vols=np.array(hmarket),
             truth=np.array([htruth.v0, htruth.theta, htruth.kappa, htruth.rho, htruth.volvol]),
             start=np.array([hstart.v0, hstart.theta, hstart.kappa, hstart.rho, hstart.volvol]),
             fit=np.array([hfit.v0, hfit.theta, hfit.kappa, hfit.rho, hfit.volvol]), fit_vols=np.array(hfit_vols), ref_seconds=np.array(hsecs))



def rough_mc() -> None:
    """rough-LogSV multi-factor MC with caller-supplied normals (pricers/logsv_pricer.py:1164-1232 ->
    rough_logsv/split_simulation.py:466 log_spot_full_combined): per-maturity terminal states, prices and the route's 'std errors'."""
    _import_reference()
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.pricers.rough_logsv.split_simulation import log_spot_full_combined
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T = np.array(['P', 'P', 'C', 'C', 'C'])
    TI = np.array(['IP', 'IP', 'IC', 'IC', 'IC'])
    cases = {
        "h030_n3": dict(params=LogSvParams(sigma0=0.8, theta=1.0, kappa1=3.0, kappa2=3.0, beta=0.15, volvol=1.8, H=0.3), ttms=np.array([0.1, 0.25]),
                        forwards=np.array([1.0, 1.02]), discfactors=np.array([0.999, 0.99]), types=(T, T), npy=360, seed=3, nb_path=3000),
        "h045_n2": dict(params=LogSvParams(sigma0=1.0, theta=1.0, kappa1=5.0, kappa2=5.0, beta=0.2, volvol=2.0, H=0.45), ttms=np.array([1.0 / 12.0, 0.25, 0.5]),
                        forwards=np.ones(3), discfactors=np.ones(3), types=(T, TI, T), npy=252, seed=11, nb_path=2000),
        "h050_n1": dict(params=LogSvParams(sigma0=0.5, theta=0.6, kappa1=2.0, kappa2=0.0, beta=-0.4, volvol=0.9, H=0.5), ttms=np.array([0.25]),
                        forwards=np.array([100.0]), discfactors=np.array([0.97]), types=(T,), npy=360, seed=5, nb_path=2500),
    }
    for name, c in cases.items():
        p = c["params"]
        p.approximate_kernel(T=float(c["ttms"][-1]))
        Z0, Z1, grids = lp.get_randoms_for_rough_vol_chain_valuation(ttms=c["ttms"], nb_path=c["nb_path"], nb_steps_per_year=c["npy"], seed=c["seed"])
        M = len(c["ttms"])
        strikes = tuple(K * c["forwards"][m] for m in range(M))
        prices, stds = lp.rough_logsv_mc_chain_pricer_fixed_randoms(
            ttms=c["ttms"], forwards=c["forwards"], discfactors=c["discfactors"], strikes_ttms=strikes, optiontypes_ttms=c["types"], Z0=Z0, Z1=Z1,
            sigma0=p.sigma0, theta=p.theta, kappa1=p.kappa1, kappa2=p.kappa2, beta=p.beta, orthog_vol=p.volvol, weights=p.weights, nodes=p.nodes,
            timegrids=grids)
        out = dict(params=np.array([p.sigma0, p.theta, p.kappa1, p.kappa2, p.beta, p.volvol, p.H]), weights=p.weights, nodes=p.nodes, ttms=c["ttms"],
                   forwards=c["forwards"], discfactors=c["discfactors"], npy=np.array(c["npy"]), seed=np.array(c["seed"]), nb_path=np.array(c["nb_path"]),
                   nslices=np.array(M), Z0_head=Z0[:3, :5], Z1_head=Z1[:3, :5])
        # terminal states per maturity, exactly as the chain pricer computes them (restart from t = 0 with the prefix of the normals)
        N = p.nodes.size
        volvol = np.sqrt(p.beta ** 2 + p.volvol ** 2)
        rho = p.beta / volvol
        v0 = np.full((N,), p.sigma0 / np.sum(p.weights))
        v0_vec = np.repeat(v0[:, None], c["nb_path"], axis=1)
        w_vec = np.repeat(p.weights[:, None], c["nb_path"], axis=1)
        n_vec = np.repeat(p.nodes[:, None], c["nb_path"], axis=1)
        for m in range(M):
            S = grids[m].size - 1
            ls, vol, qv = log_spot_full_combined(n_vec, w_vec, v0_vec, p.theta, p.kappa1, p.kappa2, 0.0, v0_vec.copy(), rho, volvol, grids[m],
                                                 c["nb_path"], Z0[:S], Z1[:S])
            out[f"grid_{m}"] = np.asarray(grids[m])
            out[f"log_spot_{m}"], out[f"vol_{m}"], out[f"qv_{m}"] = ls, vol, qv
            out[f"strikes_{m}"], out[f"types_{m}"] = strikes[m], c["types"][m]
            out[f"prices_{m}"], out[f"stds_{m}"] = np.asarray(prices[m]), np.asarray(stds[m])
        np.savez(os.path.join(OUT, f"rough_mc_{name}.npz"), **out)
        print(name, "nodes", p.nodes, "weights", p.weights, "prices", [np.asarray(a) for a in prices][0])
    # the reference's OWN regression fixture for this path (tests/test_rough_logsv_pricer_regression.py: BTC chain, H = 0.1, 10000 paths,
    # seed 10, rtol 1e-7): expected prices copied from its .npz, plus the kernel nodes / weights its european_rule produces (the
    # quadrature optimiser is host set-up code outside the hot path and is not rebuilt in the B200 package)
    from stochvolmodels.data.sample_option_chains import get_btc_test_chain_data
    chain = get_btc_test_chain_data()
    p = LogSvParams(sigma0=0.377, theta=0.347, kappa1=1.29, kappa2=1.93, beta=2.45, volvol=1.81)
    p.H = 0.1
    p.approximate_kernel(T=chain.ttms[-1])
    ref = np.load(os.path.join(os.path.dirname(REF_SRC), "src", "stochvolmodels", "tests", "test_rough_logsv_pricer_regression",
                               "test_rough_logsv_pricer_pricing_regression.npz"))
    out = dict(params=np.array([p.sigma0, p.theta, p.kappa1, p.kappa2, p.beta, p.volvol, p.H]), weights=p.weights, nodes=p.nodes,
               nb_path=np.array(10000), npy=np.array(360), seed=np.array(10), nslices=np.array(len(chain.ttms)))
    for m in range(len(chain.ttms)):
        out[f"expected_prices_{m}"] = ref[f"option_prices_ttm_{m}"]
    np.savez(os.path.join(OUT, "rough_mc_reference_regression.npz"), **out)
    print("reference regression fixture: nodes", p.nodes, "weights", p.weights)


def analytic_branch() -> None:
    """semi-analytic ODE branch (is_analytic=True): solve_analytic_ode_grid_phi (pricers/logsv/affine_expansion.py:388-470) and the chain pricer on
    parameter sets where the reference's fixed-point iteration converges (it returns NaN prices for the quickstart / BTC sets at SECOND order)."""
    _import_reference()
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers.logsv import affine_expansion as afe
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.utils import mgf_pricer as mgfp
    from stochvolmodels.utils.config import VariableType
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T = np.array(['P', 'P', 'C', 'C', 'C'])
    TI = np.array(['IP', 'IP', 'IC', 'IC', 'IC'])
    cases = {"quick_first": (LogSvParams(1.0, 1.0, 5.0, 5.0, 0.2, 2.0), afe.ExpansionOrder.FIRST, True, T),
             "mild_second": (LogSvParams(0.2, 0.2, 1.0, 2.5, -0.3, 0.4), afe.ExpansionOrder.SECOND, True, T),
             "mild2_second_inverse": (LogSvParams(0.3, 0.25, 2.0, 4.0, -0.2, 0.6), afe.ExpansionOrder.SECOND, False, TI),
             "quick_second_nan": (LogSvParams(1.0, 1.0, 5.0, 5.0, 0.2, 2.0), afe.ExpansionOrder.SECOND, True, T)}
    ttms = np.array([0.1, 0.25, 0.5])
    out = {}
    for name, (p, order, spot, types) in cases.items():
        vol_scaler = lp.set_vol_scaler(sigma0=p.sigma0, ttm=np.min(ttms))
        phi, psi, theta_grid = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, is_spot_measure=spot, vol_scaler=vol_scaler)
        a_t0 = np.zeros((phi.shape[0], afe.get_expansion_n(order)), dtype=np.complex128)
        t0 = 0.0
        for m, ttm in enumerate(ttms):
            a_t0, lm = afe.compute_logsv_a_mgf_grid(ttm=ttm - t0, phi_grid=phi, psi_grid=psi, theta_grid=theta_grid, a_t0=a_t0, is_analytic=True,
                                                    expansion_order=order, is_spot_measure=spot, sigma0=p.sigma0, theta=p.theta, kappa1=p.kappa1,
                                                    kappa2=p.kappa2, beta=p.beta, volvol=p.volvol)
            # every 8th grid point (the prices pin the whole grid); COPIES: the reference updates a_t0 in place across maturities (:487-488)
            out[f"{name}_a_{m}"], out[f"{name}_lm_{m}"] = a_t0[::8].copy(), lm[::8].copy()
            t0 = ttm
        prices = lp.logsv_chain_pricer(params=p, ttms=ttms, forwards=np.ones(3), discfactors=np.array([0.999, 0.99, 0.98]), strikes_ttms=(K, K, K),
                                       optiontypes_ttms=(types, types, types), is_analytic=True, expansion_order=order, is_spot_measure=spot)
        out[f"{name}_prices"] = np.array([np.asarray(x) for x in prices])
        out[f"{name}_params"] = np.array([p.sigma0, p.theta, p.kappa1, p.kappa2, p.beta, p.volvol, order.value, float(spot)])
        out[f"{name}_types"] = types
        out[f"{name}_phi"] = phi
        print(name, out[f"{name}_prices"][1])
    np.savez_compressed(os.path.join(OUT, "logsv_analytic_branch.npz"), ttms=ttms, strikes=K, discfactors=np.array([0.999, 0.99, 0.98]), **out)


def bdf_branch() -> None:
    """stiff branch (is_stiff_solver=True): solve_ivp(method='BDF', jac=func_rhs_jac) per grid point (pricers/logsv/affine_expansion.py:229-303).
    a_t1 / log_mgf on every 8th grid point for three parameter sets (two carried maturities), full-grid chain prices for one."""
    _import_reference()
    from stochvolmodels.pricers import logsv_pricer as lp
    from stochvolmodels.pricers.logsv import affine_expansion as afe
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.utils import mgf_pricer as mgfp
    from stochvolmodels.utils.config import VariableType
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T = np.array(['P', 'P', 'C', 'C', 'C'])
    cases = {"quick_second": (LogSvParams(1.0, 1.0, 5.0, 5.0, 0.2, 2.0), afe.ExpansionOrder.SECOND, True, 1.0),
             "btc_second_inverse_eta": (LogSvParams(0.8376, 1.0413, 3.1844, 3.058, 0.1514, 1.8458), afe.ExpansionOrder.SECOND, False, 0.9),
             "mild_first": (LogSvParams(0.2, 0.2, 1.0, 2.5, -0.3, 0.4), afe.ExpansionOrder.FIRST, True, 1.0)}
    ttms = np.array([0.1, 0.35])
    out = {}
    for name, (p, order, spot, eta) in cases.items():
        vol_scaler = lp.set_vol_scaler(sigma0=p.sigma0, ttm=np.min(ttms))
        phi, psi, theta_grid = mgfp.get_transform_var_grid(variable_type=VariableType.LOG_RETURN, is_spot_measure=spot, vol_scaler=vol_scaler)
        phi, psi, theta_grid = phi[::8], psi[::8], theta_grid[::8]
        a_t0 = np.zeros((phi.shape[0], afe.get_expansion_n(order)), dtype=np.complex128)
        t0 = 0.0
        for m, ttm in enumerate(ttms):
            a_t0, lm = afe.compute_logsv_a_mgf_grid(ttm=ttm - t0, phi_grid=phi, psi_grid=psi, theta_grid=theta_grid, a_t0=a_t0, is_stiff_solver=True,
                                                    expansion_order=order, is_spot_measure=spot, sigma0=p.sigma0, theta=p.theta, kappa1=p.kappa1,
                                                    kappa2=p.kappa2, beta=p.beta, volvol=p.volvol, vol_backbone_eta=eta)
            out[f"{name}_a_{m}"], out[f"{name}_lm_{m}"] = a_t0.copy(), lm.copy()
            t0 = ttm
        out[f"{name}_params"] = np.array([p.sigma0, p.theta, p.kappa1, p.kappa2, p.beta, p.volvol, order.value, float(spot), eta])
        out[f"{name}_phi"] = phi
        print(name, "done", np.abs(a_t0).max())
    p = cases["quick_second"][0]
    prices = lp.logsv_chain_pricer(params=p, ttms=ttms, forwards=np.ones(2), discfactors=np.array([0.999, 0.99]), strikes_ttms=(K, K),
                                   optiontypes_ttms=(T, T), is_stiff_solver=True)
    out["quick_second_prices"] = np.array([np.asarray(x) for x in prices])
    print("prices", out["quick_second_prices"])
    np.savez_compressed(os.path.join(OUT, "logsv_bdf_branch.npz"), ttms=ttms, strikes=K, types=T, discfactors=np.array([0.999, 0.99]), **out)


def hawkes_mc() -> None:
    """Hawkes jump-diffusion MC (pricers/hawkes_jd_pricer.py:644-779).  The reference draws from numpy's GLOBAL legacy generator, so each case
    is run after np.random.seed(seed): RandomState(seed) re-draws the same arrays in the same order (W0 normal, U_P, U_M uniform(1e-16, 1),
    J_P, J_M exponential; one block of shape (S, N) each per simulate call)."""
    _import_reference()
    from stochvolmodels.pricers import hawkes_jd_pricer as hj
    from stochvolmodels.data.sample_option_chains import get_btc_test_chain_data
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T = np.array(['P', 'P', 'C', 'C', 'C'])
    out = {}
    # (a) terminal values, default (BTC-like) parameters and a second set with mu != 0 and per-path initial state
    for name, params, ttm, N, seed, init in (("dflt", hj.HawkesJDParams(), 0.1, 3000, 21, None),
                                             ("drift", hj.HawkesJDParams(mu=0.05, sigma=0.3, shift_p=0.04, mean_p=0.05, shift_m=-0.03, mean_m=-0.06, lambda_p=12.0,
                                                                         theta_p=9.0, kappa_p=15.0, beta1_p=40.0, beta2_p=-30.0, lambda_m=10.0, theta_m=11.0,
                                                                         kappa_m=20.0, beta1_m=50.0, beta2_m=-60.0), 0.05, 2000, 22, 5)):
        d = params.to_dict()
        d.pop("risk_premia_gamma", None)
        if init is None:
            x0, lp0, lm0 = np.zeros(N), params.lambda_p * np.ones(N), params.lambda_m * np.ones(N)
        else:
            rs = np.random.RandomState(init)
            x0, lp0, lm0 = rs.normal(0, 0.05, N), params.lambda_p * np.exp(rs.normal(0, 0.2, N)), params.lambda_m * np.exp(rs.normal(0, 0.2, N))
        np.random.seed(seed)
        kw = {k: v for k, v in d.items() if k not in ("lambda_p", "lambda_m")}
        x, lp, lm = hj.simulate_hawkesjd_terminal(ttm=ttm, x0=x0.copy(), lambda_p0=lp0.copy(), lambda_m0=lm0.copy(), nb_path=N, **kw)
        out.update({f"{name}_params": np.array([d[k] for k in HAWKES_KEYS]), f"{name}_ttm": np.array(ttm), f"{name}_N": np.array(N),
                    f"{name}_seed": np.array(seed), f"{name}_x0": x0, f"{name}_lp0": lp0, f"{name}_lm0": lm0, f"{name}_x": x, f"{name}_lp": lp,
                    f"{name}_lm": lm})
    # (b) chain pricer on two maturities
    params = hj.HawkesJDParams()
    ttms, fw, df = np.array([0.05, 0.12]), np.array([1.0, 1.01]), np.array([0.999, 0.995])
    np.random.seed(33)
    prices, stds = hj.HawkesJDPricer().model_mc_price_chain.__wrapped__(hj.HawkesJDPricer(), _chain(ttms, fw, df, K, T), params, nb_path=4000) \
        if hasattr(hj.HawkesJDPricer.model_mc_price_chain, "__wrapped__") else hj.HawkesJDPricer().model_mc_price_chain(_chain(ttms, fw, df, K, T), params, nb_path=4000)
    out.update(chain_ttms=ttms, chain_forwards=fw, chain_discfactors=df, chain_strikes=K, chain_types=T, chain_seed=np.array(33), chain_N=np.array(4000),
               chain_params=np.array([params.to_dict()[k] for k in HAWKES_KEYS]),
               chain_prices=np.array([np.asarray(p) for p in prices]), chain_stds=np.array([np.asarray(p) for p in stds]))
    np.savez(os.path.join(OUT, "hawkes_mc.npz"), keys=np.array(HAWKES_KEYS), **out)
    print("hawkes chain prices", out["chain_prices"])


HAWKES_KEYS = ("mu", "sigma", "shift_p", "mean_p", "shift_m", "mean_m", "lambda_p", "theta_p", "kappa_p", "beta1_p", "beta2_p", "lambda_m", "theta_m",
               "kappa_m", "beta1_m", "beta2_m")


def hawkes_fourier() -> None:
    """Hawkes jump-diffusion Fourier route (pricers/hawkes_jd_pricer.py:365-641): per-maturity ODE grids (500 transform points, SciPy RK45 per
    point), log-MGF and chain prices, without and with the risk-premium kernel -> hawkes_fourier.npz.
    python tests/golden/make_golden.py --only-hawkes-fourier"""
    _import_reference()
    from stochvolmodels.pricers import hawkes_jd_pricer as hj
    from stochvolmodels.utils import mgf_pricer as mgfp
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T = np.array(['P', 'P', 'C', 'C', 'C'])
    ttms, fw, df = np.array([0.05, 0.12, 0.3]), np.array([1.0, 1.01, 1.02]), np.array([0.999, 0.995, 0.99])
    sets = {"dflt": hj.HawkesJDParams(),
            "alt": hj.HawkesJDParams(mu=0.05, sigma=0.3, shift_p=0.04, mean_p=0.05, shift_m=-0.03, mean_m=-0.06, lambda_p=12.0, theta_p=9.0, kappa_p=15.0,
                                     beta1_p=40.0, beta2_p=-30.0, lambda_m=10.0, theta_m=11.0, kappa_m=20.0, beta1_m=50.0, beta2_m=-60.0)}
    out = dict(ttms=ttms, forwards=fw, discfactors=df, strikes=K, types=T, keys=np.array(HAWKES_KEYS))
    from numba.typed import List
    for name, params in sets.items():
        out[f"{name}_params"] = np.array([params.to_dict()[k] for k in HAWKES_KEYS])
        vol_scaler = hj.set_vol_scaler(sigma0=params.sigma, ttm=np.min(ttms))
        phi, psi, theta = mgfp.get_transform_var_grid(max_phi=hj.MAX_PHI, vol_scaler=vol_scaler)
        out[f"{name}_phi"] = phi
        a, t0 = np.zeros((phi.shape[0], 3), dtype=np.complex128), 0.0
        for m, ttm in enumerate(ttms):
            a, lm = hj.compute_hawkes_a_mgf_grid(ttm=ttm - t0, phi_grid=phi, psi_grid=psi, theta_grid=theta, a_t0=a, model_params=params)
            out[f"{name}_a_{m}"], out[f"{name}_lm_{m}"] = a.copy(), lm.copy()
            t0 = ttm
        prices = hj.hawkesjd_chain_pricer(model_params=params, ttms=ttms, forwards=fw, discfactors=df, strikes_ttms=List([K * f for f in fw]),
                                          optiontypes_ttms=List([T for _ in fw]))
        out[f"{name}_prices"] = np.array([np.asarray(p) for p in prices])
        print(name, out[f"{name}_prices"])
    # risk-premium kernel
    gamma = 0.4
    pg = hj.HawkesJDParams(risk_premia_gamma=gamma)
    normalizers, gamma_forwards = hj.hawkesjd_forwards_under_risk_kernel(model_params=pg, forwards=fw, risk_premia_gamma=gamma, ttms=ttms)
    prices = hj.hawkesjd_chain_pricer_with_risk_premia(model_params=pg, ttms=ttms, forwards=fw, discfactors=df, strikes_ttms=List([K * f for f in fw]),
                                                       optiontypes_ttms=List([T for _ in fw]))
    out.update(gamma=np.array(gamma), gamma_normalizers=normalizers, gamma_forwards=gamma_forwards, gamma_prices=np.array([np.asarray(p) for p in prices]))
    print("gamma", out["gamma_prices"], normalizers, gamma_forwards)
    np.savez(os.path.join(OUT, "hawkes_fourier.npz"), **out)
    print("wrote hawkes_fourier.npz")


def chain_transforms() -> None:
    """OptionChain slice views and strike transforms on the BTC sample chain -> option_chain_transforms.npz.
    python tests/golden/make_golden.py --only-chain"""
    _import_reference()
    from stochvolmodels.data.option_chain import OptionChain
    from stochvolmodels.data.sample_option_chains import get_btc_test_chain_data
    c = get_btc_test_chain_data()
    out = dict(ids=np.asarray(c.ids), ttms=c.ttms, forwards=c.forwards)
    for m in range(len(c.ttms)):
        out[f"bid_ivs_{m}"], out[f"ask_ivs_{m}"], out[f"strikes_{m}"] = c.bid_ivs[m], c.ask_ivs[m], c.strikes_ttms[m]
    n = OptionChain.to_forward_normalised_strikes(c)
    u = OptionChain.to_uniform_strikes(c, num_strikes=7)
    for m in range(len(c.ttms)):
        out[f"norm_strikes_{m}"] = n.strikes_ttms[m]
        out[f"uni_strikes_{m}"], out[f"uni_types_{m}"] = u.strikes_ttms[m], np.asarray(u.optiontypes_ttms[m])
    out["norm_forwards"], out["norm_forwards0"] = n.forwards, n.forwards0
    sub = OptionChain.get_slices_as_chain(c, ids=["3m", "1m"])
    out["sub_ttms"], out["sub_forwards"], out["sub_ids"] = sub.ttms, sub.forwards, np.asarray(sub.ids)
    out["sub_strikes_0"], out["sub_bid_1"] = sub.strikes_ttms[0], sub.bid_ivs[1]
    one = OptionChain.get_slices_as_chain(c, ids=["2m"])
    out["one_ttms"], out["one_strikes"] = one.ttms, one.strikes_ttms[0]
    sl = c.get_slice("2w")
    out["slice_scalars"] = np.array([sl.ttm, sl.forward, sl.discfactor, sl.discount_rate])
    out["slice_ask"] = sl.ask_ivs
    out["mid_vols_0"] = c.get_mid_vols()[0]
    np.savez(os.path.join(OUT, "option_chain_transforms.npz"), **out)
    print("wrote option_chain_transforms.npz")


def params_helpers() -> None:
    """LogSvParams helper methods (spatial grids, steady-state exponents, vol-moment generator) and the vol-moment / variance-swap functions of
    pricers/logsv/vol_moments_ode.py for three parameter sets -> logsv_params_helpers.npz.   python tests/golden/make_golden.py --only-helpers"""
    _import_reference()
    import pandas as pd
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.pricers.logsv import vol_moments_ode as vmo
    from stochvolmodels.utils.config import VariableType
    sets = np.array([[1.0, 1.0, 5.0, 5.0, 0.2, 2.0], [0.8376, 1.0413, 3.1844, 3.058, 0.1514, 1.8458], [0.35, 0.5, 2.0, 1.2, -0.6, 0.9]])
    ts = np.array([0.0, 0.05, 0.25, 1.0, 2.5])
    out = dict(sets=sets, ts=ts)
    for i, row in enumerate(sets):
        p = LogSvParams(*row)
        out[f"scalars_{i}"] = np.array([p.gamma, p.eta, p.kappa, p.theta2, p.vartheta2])
        for name, vt in (("x", VariableType.LOG_RETURN), ("sigma", VariableType.SIGMA), ("qvar", VariableType.Q_VAR)):
            out[f"grid_{name}_{i}"] = p.get_variable_space_grid(variable_type=vt, ttm=0.7, n_stdevs=2.5, n=37)
        out[f"grid_x_default_{i}"] = p.get_x_grid()
        out[f"lambda4_{i}"] = p.get_vol_moments_lambda(n_terms=4)
        out[f"lambda8_{i}"] = p.get_vol_moments_lambda(n_terms=8)
        out[f"moments_{i}"] = vmo.compute_vol_moments_t(params=p, ttm=ts, n_terms=4)
        out[f"moments8_{i}"] = vmo.compute_vol_moments_t(params=p, ttm=ts[1:], n_terms=8)
        out[f"int_moments_{i}"] = np.array([vmo.compute_analytic_vol_moments(params=p, t=t, n_terms=4, is_qvar=True) for t in ts[1:]])
        out[f"expected_vol_{i}"] = vmo.compute_expected_vol_t(params=p, t=ts, n_terms=4)
        out[f"sqrt_qvar_{i}"] = vmo.compute_sqrt_qvar_t(params=p, t=ts, n_terms=4)
        strikes = pd.Series(np.array([0.9, 0.95, 1.0, 1.05]) * row[0], index=np.array([0.04, 0.1, 0.5, 1.0]))
        out[f"varswap_strikes_{i}"] = np.stack([strikes.index.to_numpy(), strikes.to_numpy()])
        out[f"backbone_{i}"] = vmo.fit_model_vol_backbone_to_varswaps(log_sv_params=p, varswap_strikes=strikes).to_numpy()
    np.savez(os.path.join(OUT, "logsv_params_helpers.npz"), **out)
    print("wrote logsv_params_helpers.npz")


def reference_objects() -> None:
    """The state (``vars()`` after ``__post_init__``) of the reference's own OptionChain / LogSvParams / HestonParams / HawkesJDParams
    objects that tests/test_reference_ducktyping.py hands to the B200 pricers, and the members of its VariableType enum
    -> reference_objects.npz.  Key ``<obj>__fields`` lists the attributes in order; ``<obj>__<attr>`` holds a value, ``<obj>__<attr>__<i>``
    the i-th array of a list; an attribute with neither is None.  ``<obj>@<method>`` records what the reference's methods that the pricers
    call returned: get_vol_backbone_eta at the chain's maturities ([taus, etas]) and the keys of to_dict().
    python tests/golden/make_golden.py --only-objects"""
    _import_reference()
    from stochvolmodels.data.option_chain import OptionChain
    from stochvolmodels.pricers.hawkes_jd_pricer import HawkesJDParams
    from stochvolmodels.pricers.heston_pricer import HestonParams
    from stochvolmodels.pricers.logsv.logsv_params import LogSvParams
    from stochvolmodels.utils.config import VariableType
    hawkes = dict(sigma=0.4, mean_p=0.04, mean_m=-0.05, theta_p=6.0, lambda_p=7.0, kappa_p=20.0, beta1_p=30.0, beta2_p=-25.0)
    objects = dict(
        chain=OptionChain(ttms=np.array([0.1, 0.3]), forwards=np.array([1.0, 1.02]), discfactors=np.array([1.0, 0.99]), ids=np.array(["a", "b"]),
                          strikes_ttms=[np.array([0.9, 1.0, 1.1]), np.array([0.8, 1.2])],
                          optiontypes_ttms=[np.array(["P", "C", "C"]), np.array(["P", "C"])]),
        logsv=LogSvParams(sigma0=0.9, theta=1.0, kappa1=4.0, kappa2=3.0, beta=0.3, volvol=1.5),
        logsv_params5=LogSvParams(sigma0=0.9, theta=0.8, kappa1=4.0, kappa2=None, beta=0.3, volvol=1.5),
        heston=HestonParams(v0=0.05, theta=0.06, kappa=3.0, rho=-0.4, volvol=0.7),
        hawkes=HawkesJDParams(**hawkes),
        hawkes_gamma=HawkesJDParams(risk_premia_gamma=0.3, **hawkes))
    out = dict(variable_type_names=np.array([m.name for m in VariableType]), variable_type_values=np.array([m.value for m in VariableType]))
    for name, obj in objects.items():
        out[f"{name}__fields"] = np.array(list(vars(obj)))
        for attr, v in vars(obj).items():
            if isinstance(v, (list, tuple)):
                for i, a in enumerate(v):
                    out[f"{name}__{attr}__{i}"] = np.asarray(a)
            elif v is not None:
                out[f"{name}__{attr}"] = np.asarray(v)
        if isinstance(obj, LogSvParams):
            taus = objects["chain"].ttms
            etas = np.array([obj.get_vol_backbone_eta(tau=t) for t in taus], dtype=float)
            assert np.array_equal(etas, obj.get_vol_backbone_etas(ttms=taus))
            out[f"{name}@get_vol_backbone_eta"] = np.stack([taus, etas])
        if isinstance(obj, HawkesJDParams):
            out[f"{name}@to_dict"] = np.array(list(obj.to_dict()))
    np.savez(os.path.join(OUT, "reference_objects.npz"), **out)
    print("wrote reference_objects.npz")


def _chain(ttms, fw, df, K, T):
    from stochvolmodels.data.option_chain import OptionChain
    from numba.typed import List
    return OptionChain(ttms=ttms, forwards=fw, discfactors=df, strikes_ttms=List([K * f for f in fw]), optiontypes_ttms=List([T for _ in fw]),
                       ids=np.array([f"{t:0.2f}" for t in ttms]))


if __name__ == "__main__":
    if "--only-objects" in sys.argv:
        reference_objects()
        sys.exit(0)
    if "--only-hawkes-fourier" in sys.argv:
        hawkes_fourier()
        sys.exit(0)
    if "--only-chain" in sys.argv:
        chain_transforms()
        sys.exit(0)
    if "--only-helpers" in sys.argv:
        params_helpers()
        sys.exit(0)
    if "--only-bdf" in sys.argv:
        bdf_branch()
        sys.exit(0)
    if "--only-analytic" in sys.argv:
        analytic_branch()
        sys.exit(0)
    if "--only-hawkes" in sys.argv:
        hawkes_mc()
        sys.exit(0)
    if "--only-rough" in sys.argv:
        rough_mc()
        sys.exit(0)
    if "--only-calib" in sys.argv:
        calibration()
        sys.exit(0)
    if "--only-volpaths" in sys.argv:
        vol_paths()
        sys.exit(0)
    if "--only-next" in sys.argv:
        next_rows()
        sys.exit(0)
    if "--only-refmc" not in sys.argv:
        main()
    if "--skip-refmc" not in sys.argv:
        reference_mc()
