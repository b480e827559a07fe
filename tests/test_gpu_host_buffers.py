"""GPU: host-level library calls leave no device memory behind, on the error path as on the success path.

The library allocates its temporaries with cudaMallocAsync from the device's default memory pool; the pool's used bytes are read through
the CUDA runtime torch has loaded (the library links its own static copy, but the pool is per device, so both see the same one).
Only input the library rejects on the host is used: no device fault, no out-of-memory condition."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CUDA_MEMPOOL_ATTR_USED_MEM_CURRENT = 7      # cudaMemPoolAttrUsedMemCurrent (driver_types.h)


def _cudart():
    import torch
    torch.cuda.init()
    with open("/proc/self/maps") as f:
        paths = {line.split()[-1] for line in f if "libcudart.so" in line}
    assert paths, "torch has not loaded a shared CUDA runtime"
    return ctypes.CDLL(sorted(paths)[0])


def _pool_used_bytes(rt) -> int:
    import torch
    torch.cuda.synchronize()
    pool, used = ctypes.c_void_p(), ctypes.c_uint64()
    assert rt.cudaDeviceGetDefaultMemPool(ctypes.byref(pool), torch.cuda.current_device()) == 0
    assert rt.cudaMemPoolGetAttribute(pool, CUDA_MEMPOOL_ATTR_USED_MEM_CURRENT, ctypes.byref(used)) == 0
    return used.value


def test_rejected_call_frees_its_buffers(cuda_lib):
    """contradictory Gaussian flags are rejected with the same error, and nothing stays allocated"""
    from stochvolmodels_b200 import engine
    from stochvolmodels_b200 import _capi as C
    rt = _cudart()
    engine.device_normals(1, 0, 1000, 0, 4, C.GAUSS_F32)
    base = _pool_used_bytes(rt)
    with pytest.raises(C.B200svError, match="B200SV_GAUSS_F64 and B200SV_GAUSS_F64_PAIRED are mutually exclusive") as e:
        engine.device_normals(1, 0, 1000, 0, 4, C.GAUSS_F64 | C.GAUSS_F64_PAIRED)
    assert e.value.code == -1
    assert _pool_used_bytes(rt) == base


def test_host_level_calls_free_their_buffers(cuda_lib):
    """one small call of each host-level entry point family; the pool's used bytes are back at the baseline after each"""
    from stochvolmodels_b200 import HawkesJDParams, HawkesJDPricer, OptionChain, engine
    from stochvolmodels_b200 import _capi as C
    from stochvolmodels_b200.pricers.hawkes_jd_pricer import hawkesjd_chain_pricer_with_risk_premia, hawkesjd_device_draws
    from oracle.hawkes import KEYS
    rt = _cudart()
    lp = engine.logsv_params_c(0.4, 0.4, 2.21, 2.18, 0.15, 2.0)
    hp = engine.heston_params_c(0.04, 0.04, 4.0, -0.6, 0.8)
    ttms, fw, df = np.array([0.083, 0.25]), np.array([1.0, 1.01]), np.array([0.999, 0.99])
    K = np.array([0.8, 0.9, 1.0, 1.1, 1.2])
    T = np.array(["P", "P", "C", "C", "C"])
    strikes, types = [K, K], [T, T]
    N, seed = 10000, 7
    f64, f32 = engine.mc_flags("fp64"), engine.mc_flags("fp32")
    W = np.random.RandomState(0).normal(size=(2, 8, 1000))
    hawkes = HawkesJDParams(mu=0.02, sigma=0.4, lambda_p=9.0, lambda_m=11.0)
    chain = OptionChain(ttms=ttms, forwards=fw, discfactors=df, strikes_ttms=strikes, optiontypes_ttms=types)
    calls = {
        "logsv_mc_chain (cooperative)": lambda: engine.logsv_mc_chain(lp, ttms, fw, df, None, strikes, types, N, 360, True, 1, seed, f64),
        "logsv_mc_chain (multi-launch)": lambda: engine.logsv_mc_chain(lp, ttms, fw, df, None, strikes, types, N, 360, True, 1, seed, f32),
        "heston_mc_chain_batch": lambda: engine.heston_mc_chain_batch([hp, hp], ttms, fw, df, strikes, types, N, 360, seed, f32),
        "rough_logsv_mc_chain": lambda: engine.rough_logsv_mc_chain([lp], [0.5, 0.5], [0.1, 10.0], ttms, fw, df, strikes, types, N, [30, 90],
                                                                    [0.083 / 30, 0.25 / 90], seed=seed, with_ivols=True),
        "hawkesjd_mc_chain": lambda: HawkesJDPricer().model_mc_price_chain(chain, hawkes, nb_path=N, seed=seed),
        "logsv_terminal": lambda: engine.logsv_terminal(lp, 0.25, N, 360, True, 1.0, seed, f64),
        "logsv_terminal_from_state": lambda: engine.logsv_terminal_from_state(lp, np.zeros(N), np.full(N, 0.4), np.zeros(N), 0.25, 360, True, 1.0,
                                                                              seed, f64, slice_index=1),
        "heston_terminal": lambda: engine.heston_terminal(hp, 0.25, N, 360, seed, f64),
        "hawkesjd_terminal": lambda: HawkesJDPricer().simulate_terminal_values(hawkes, ttm=0.04, nb_path=N, seed=seed),
        "logsv_step_fixed": lambda: engine.logsv_step_fixed(0.0, 0.4, 0.0, W[0], W[1], 1 / 360, lp, 1.0, True),
        "mc_payoffs": lambda: engine.mc_payoffs(np.zeros(N), None, 0.25, 1.0, K, T),
        "device_normals": lambda: engine.device_normals(seed, 0, 1000, 0, 4, C.GAUSS_F64),
        "hawkesjd_device_draws": lambda: hawkesjd_device_draws(seed, 0, 1000, 0, 0.01, **{k: v for k, v in hawkes.to_dict().items() if k in KEYS}),
        "debug_exp_pair": lambda: engine.debug_exp_pair(np.linspace(-3, 3, 1000)),
        "logsv_vol_paths": lambda: engine.logsv_vol_paths(lp, 0.25, 1000, 360, True, seed),
        "logsv_price_chain": lambda: engine.logsv_price_chain(lp, ttms, fw, df, None, strikes, types),
        "heston_price_chain_batch": lambda: engine.heston_price_chain_batch([hp, hp], ttms, fw, df, strikes, types),
        "hawkesjd_price_chain (risk premia)": lambda: hawkesjd_chain_pricer_with_risk_premia(
            HawkesJDParams(**{**hawkes.to_dict(), "risk_premia_gamma": 0.5}), ttms, fw, df, strikes, types),
        "bsm_implied_vols": lambda: engine.bsm_implied_vols(ttms, fw, df, strikes, types, [np.full(5, 0.05), np.full(5, 0.08)]),
    }
    base = _pool_used_bytes(rt)
    for name, call in calls.items():
        call()
        assert _pool_used_bytes(rt) == base, name
