"""Run the REFERENCE'S OWN test files against this package as a drop-in (needs CUDA and oracle/_ref).

    python tools/run_reference_tests.py [test_file_stem ...]          # default: the files that touch SURVEY.md section 8's paths

The unmodified stochvolmodels 2.2.0 wheel that oracle/install_reference.sh puts into oracle/_ref ships its test-suite
(stochvolmodels/tests).  This tool aliases the module paths those tests import (``stochvolmodels.pricers.logsv_pricer`` ...) to the modules
of stochvolmodels_b200 in ``sys.modules`` -- no file of the reference is imported except its test files -- gives plain functions the
``py_func`` attribute the tests reach for on Numba dispatchers, and runs pytest on copies of the test files in a temporary directory.
Modules this package does not provide (fitters, HJM, rough-kernel quadrature, plotting, the third-party ``vanilla_option_pricers``) stay
unimportable, so the tests that need them error at import or fail: they are outside the hot-path scope and are reported as such.
It prints one line per test and a summary; the result is what profiles/r02_reference_tests.txt records.  Not part of the pytest suite."""
import importlib
import os
import shutil
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF_TESTS = os.path.join(ROOT, "oracle", "_ref", "stochvolmodels", "tests")

# reference module path -> module(s) of this package whose public names it exposes (later entries fill names the earlier ones lack)
ALIASES = {
    "stochvolmodels": ["stochvolmodels_b200"],
    "stochvolmodels.data": [],
    "stochvolmodels.data.option_chain": ["stochvolmodels_b200.data.option_chain"],
    "stochvolmodels.data.sample_option_chains": ["stochvolmodels_b200.data.option_chain"],
    "stochvolmodels.pricers": [],
    "stochvolmodels.pricers.model_pricer": ["stochvolmodels_b200.pricers.model_pricer", "stochvolmodels_b200.pricers.calibration"],
    "stochvolmodels.pricers.logsv_pricer": ["stochvolmodels_b200.pricers.logsv_pricer", "stochvolmodels_b200.pricers.calibration"],
    "stochvolmodels.pricers.heston_pricer": ["stochvolmodels_b200.pricers.heston_pricer"],
    "stochvolmodels.pricers.hawkes_jd_pricer": ["stochvolmodels_b200.pricers.hawkes_jd_pricer"],
    "stochvolmodels.pricers.logsv": [],
    "stochvolmodels.pricers.logsv.affine_expansion": ["stochvolmodels_b200.pricers.logsv.affine_expansion"],
    "stochvolmodels.pricers.logsv.logsv_params": ["stochvolmodels_b200.pricers.logsv_pricer"],
    "stochvolmodels.pricers.logsv.vol_moments_ode": ["stochvolmodels_b200.pricers.logsv.vol_moments"],
    "stochvolmodels.utils": [],
    "stochvolmodels.utils.config": ["stochvolmodels_b200.utils.config"],
    "stochvolmodels.utils.funcs": ["stochvolmodels_b200.utils.funcs"],
    "stochvolmodels.utils.mgf_pricer": ["stochvolmodels_b200.utils.mgf_pricer"],
    "stochvolmodels.utils.mc_payoffs": ["stochvolmodels_b200.utils.mc_payoffs"],
}
DEFAULT_FILES = ["test_heston_characterization", "test_numerical_utilities", "test_logsv_characterization", "test_model_calibration_contracts",
                 "test_option_chain_characterization", "test_mgf_pricer_identities", "test_rough_logsv_pricer_regression"]
# test_rough_logsv_characterization: 2 of 9 pass -- the other 7 exercise the rough kernel's quadrature optimiser (european_rule), not rebuilt


# modules of the reference this package does not rebuild: importable as empty placeholders so that the test MODULE can be collected and only the
# tests that use them fail
PLACEHOLDERS = ["stochvolmodels.fitters", "stochvolmodels.fitters.logsv_smile", "stochvolmodels.pricers.rough_logsv",
                "stochvolmodels.pricers.rough_logsv.rough_kernel"]


def black76_stand_in():
    """``vanilla_option_pricers`` is a third-party dependency of the reference that is absent from this image; its tests use three of its
    functions as the INDEPENDENT closed form they compare against.  Textbook Black-76 with the argument names the tests pass."""
    import numpy as np
    from scipy.special import ndtr
    mod = types.ModuleType("vanilla_option_pricers")

    def compute_bsm_vanilla_price(forward, strike, ttm, vol, optiontype="C", discfactor=1.0):
        sdev = vol * np.sqrt(ttm)
        d1 = np.log(forward / strike) / sdev + 0.5 * sdev
        d2 = d1 - sdev
        if optiontype in ("C", "IC"):
            price = forward * ndtr(d1) - strike * ndtr(d2)
        else:
            price = strike * ndtr(-d2) - forward * ndtr(-d1)
        return discfactor * (price / forward if optiontype in ("IC", "IP") else price)

    def compute_bsm_vanilla_slice_prices(ttm, forward, strikes, vols, optiontypes, discfactor=1.0):
        return np.array([compute_bsm_vanilla_price(forward, k, ttm, v, t, discfactor) for k, v, t in zip(strikes, vols, optiontypes)])

    def compute_bsm_digital_price(forward, strike, ttm, vol, optiontype="C", discfactor=1.0):
        sdev = vol * np.sqrt(ttm)
        d2 = np.log(forward / strike) / sdev - 0.5 * sdev
        return discfactor * (ndtr(d2) if optiontype == "C" else ndtr(-d2))

    mod.compute_bsm_vanilla_price = compute_bsm_vanilla_price
    mod.compute_bsm_vanilla_slice_prices = compute_bsm_vanilla_slice_prices
    mod.compute_bsm_digital_price = compute_bsm_digital_price
    mod.bsm = mod
    return mod


class _Missing:
    """stands in for a name the reference module has and this package does not: importing it works, using it fails the test that does"""

    def __init__(self, where, name):
        self.where, self.name = where, name

    def _fail(self, *a, **k):
        raise NotImplementedError(f"{self.where}.{self.name} is not provided by stochvolmodels_b200 (outside the hot-path scope)")

    __call__ = _fail

    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        return self._fail


class _LenientModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Missing(self.__name__, name)


def install_aliases():
    third = black76_stand_in()
    sys.modules.setdefault("vanilla_option_pricers", third)
    sys.modules.setdefault("vanilla_option_pricers.bsm", third)
    try:
        import matplotlib.pyplot  # noqa: F401
    except Exception:                           # plotting is out of scope; the calibration-contract tests only import it
        from unittest.mock import MagicMock
        for name in ("matplotlib", "matplotlib.pyplot"):
            sys.modules.setdefault(name, MagicMock())
    for name in PLACEHOLDERS:
        sys.modules[name] = _LenientModule(name)
        sys.modules[name].__path__ = []
    for ref_name, sources in ALIASES.items():
        mod = _LenientModule(ref_name)
        mod.__path__ = []                       # a package: submodule imports resolve through sys.modules only
        for src in sources:
            real = importlib.import_module(src)
            for name, value in vars(real).items():
                if not name.startswith("__") and name not in vars(mod):
                    setattr(mod, name, value)
                    if isinstance(value, types.FunctionType) and not hasattr(value, "py_func"):
                        value.py_func = value   # Numba dispatchers expose the Python function; here the function is its own
        sys.modules[ref_name] = mod
    sys.modules["stochvolmodels"].compute_bsm_vanilla_price = third.compute_bsm_vanilla_price     # re-exported by the reference
    for ref_name in list(ALIASES) + PLACEHOLDERS:      # parent.child attribute access (import a.b.c as x)
        parent, _, child = ref_name.rpartition(".")
        if parent:
            setattr(sys.modules[parent], child, sys.modules[ref_name])


def main(argv):
    import pytest
    if not os.path.isdir(REF_TESTS):
        print(f"{REF_TESTS} is missing: run oracle/install_reference.sh <StochVolModels source tree> first")
        return 2
    install_aliases()
    files = argv or DEFAULT_FILES
    work = tempfile.mkdtemp(prefix="b200sv_reftests_")
    try:
        shutil.copy(os.path.join(REF_TESTS, "conftest.py"), work)
        for stem in files:
            shutil.copy(os.path.join(REF_TESTS, stem + ".py"), work)
            if os.path.isdir(os.path.join(REF_TESTS, stem)):                      # data directory of the regression test
                shutil.copytree(os.path.join(REF_TESTS, stem), os.path.join(work, stem))
        return pytest.main(["-q", "-rA", "--tb=line", "-p", "no:cacheprovider", "--continue-on-collection-errors", "--rootdir", work, work])
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
