"""INTEGRATION.md claims that the reference's OWN objects (stochvolmodels.OptionChain, LogSvParams, HestonParams, HawkesJDParams, VariableType)
can be handed to the B200 pricers unchanged.  Checked here without a GPU: the C entry points are replaced by a recorder and the marshalled
arguments of calls made with reference objects must equal those made with this package's objects.  The reference objects are rebuilt from
tests/golden/reference_objects.npz (tests/golden/make_golden.py --only-objects): dataclasses of the reference's class names with exactly the
attributes, and the values after ``__post_init__``, that the reference's own constructors produced, and an Enum with its VariableType members."""
import dataclasses
import enum

import numpy as np
import pytest

from conftest import load_golden


def _rebuild(g, name, cls_name):
    """a dataclass instance with the attributes (same order, same values, None where absent) recorded for reference object `name`, and
    the reference methods the pricers call answering what the reference answered (any other argument is a KeyError)"""
    methods = {}
    if f"{name}@get_vol_backbone_eta" in g.files:
        table = dict(zip(*g[f"{name}@get_vol_backbone_eta"].tolist()))
        methods["get_vol_backbone_eta"] = lambda self, tau: table[float(tau)]
        methods["get_vol_backbone_etas"] = lambda self, ttms: np.array([table[float(t)] for t in ttms])
    if f"{name}@to_dict" in g.files:
        keys = [str(k) for k in g[f"{name}@to_dict"]]
        methods["to_dict"] = lambda self: {k: getattr(self, k) for k in keys}
    fields = [str(f) for f in g[f"{name}__fields"]]
    values = {}
    for f in fields:
        if f"{name}__{f}" in g.files:
            v = g[f"{name}__{f}"]
            values[f] = v.item() if v.ndim == 0 else v
        elif f"{name}__{f}__0" in g.files:
            values[f] = [g[f"{name}__{f}__{i}"] for i in range(sum(k.startswith(f"{name}__{f}__") for k in g.files))]
        else:
            values[f] = None
    return dataclasses.make_dataclass(cls_name, fields, namespace=methods)(**values)


@pytest.fixture(scope="module")
def ref():
    g = load_golden("reference_objects.npz")
    return dict(chain=_rebuild(g, "chain", "OptionChain"), logsv=_rebuild(g, "logsv", "LogSvParams"),
                logsv_params5=_rebuild(g, "logsv_params5", "LogSvParams"), heston=_rebuild(g, "heston", "HestonParams"),
                hawkes=_rebuild(g, "hawkes", "HawkesJDParams"), hawkes_gamma=_rebuild(g, "hawkes_gamma", "HawkesJDParams"),
                VariableType=enum.Enum("VariableType", {str(n): int(v) for n, v in zip(g["variable_type_names"], g["variable_type_values"])}))


class Recorder:
    """stands in for _capi.call: records (name, decoded args) and fills nothing (outputs stay uninitialised numpy buffers)."""
    def __init__(self):
        self.calls = []

    def __call__(self, name, *args):
        import ctypes
        decoded = []
        for a in args:
            if isinstance(a, (int, float, type(None))):
                decoded.append(a)
            elif isinstance(a, ctypes.Structure):
                decoded.append(tuple(getattr(a, f) for f, _ in a._fields_))
            elif hasattr(a, "_obj") and isinstance(a._obj, ctypes.Structure):          # byref(struct)
                decoded.append(tuple(getattr(a._obj, f) for f, _ in a._obj._fields_))
            else:
                decoded.append("ptr")
        self.calls.append((name, tuple(decoded)))


def _chains(ref):
    import stochvolmodels_b200 as svm
    kw = dict(ttms=np.array([0.1, 0.3]), forwards=np.array([1.0, 1.02]), discfactors=np.array([1.0, 0.99]), ids=np.array(["a", "b"]),
              strikes_ttms=[np.array([0.9, 1.0, 1.1]), np.array([0.8, 1.2])], optiontypes_ttms=[np.array(["P", "C", "C"]), np.array(["P", "C"])])
    return ref["chain"], svm.OptionChain(**kw)


def test_reference_objects_marshal_like_our_own(ref, monkeypatch):
    import stochvolmodels_b200 as svm
    from stochvolmodels_b200 import _capi as C, engine
    flat = []
    real_flatten = C.flatten_chain
    monkeypatch.setattr(C, "flatten_chain", lambda s, t: flat.append(real_flatten(s, t)) or flat[-1])
    rec = Recorder()
    monkeypatch.setattr(C, "call", rec)
    ref_chain, our_chain = _chains(ref)
    p6 = dict(sigma0=0.9, theta=1.0, kappa1=4.0, kappa2=3.0, beta=0.3, volvol=1.5)
    ref_params, our_params = ref["logsv"], svm.LogSvParams(**p6)
    pricer = svm.LogSVPricer()
    for chain, params, vt in ((ref_chain, ref_params, ref["VariableType"].LOG_RETURN), (our_chain, our_params, svm.VariableType.LOG_RETURN)):
        pricer.price_chain(chain, params)
        pricer.model_mc_price_chain(chain, params, nb_path=1000, nb_steps=360, seed=3, variable_type=vt, distributed=False)
    names = [c[0] for c in rec.calls]
    assert names == ["b200sv_logsv_price_chain", "b200sv_logsv_mc_chain"] * 2
    assert rec.calls[0] == rec.calls[2] and rec.calls[1] == rec.calls[3]            # identical scalars / structs for both object families
    assert rec.calls[0][1][0] == (0.9, 1.0, 4.0, 3.0, 0.3, 1.5)
    for a, b in zip(flat[:2], flat[2:]):                                            # identical flattened strikes / type codes / offsets
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)
    # kappa2=None of the reference's PARAMS5 convention and its vol backbone lookup go through unchanged as well
    q = ref["logsv_params5"]            # the reference's LogSvParams(sigma0=0.9, theta=0.8, kappa1=4.0, kappa2=None, beta=0.3, volvol=1.5)
    rec.calls.clear()
    pricer.price_chain(ref_chain, q)
    assert rec.calls[0][1][0][3] == 4.0 / 0.8


def test_reference_heston_params_and_enum_values(ref, monkeypatch):
    import stochvolmodels_b200 as svm
    from stochvolmodels_b200 import _capi as C, engine
    rec = Recorder()
    monkeypatch.setattr(C, "call", rec)
    ref_chain, _ = _chains(ref)
    hp = ref["heston"]                  # the reference's HestonParams(v0=0.05, theta=0.06, kappa=3.0, rho=-0.4, volvol=0.7)
    svm.HestonPricer().price_chain(ref_chain, hp)
    svm.HestonPricer().model_mc_price_chain(ref_chain, hp, nb_path=1000, seed=1, variable_type=ref["VariableType"].Q_VAR, distributed=False)
    assert rec.calls[0][0] == "b200sv_heston_price_chain" and rec.calls[0][1][0] == (0.05, 0.06, 3.0, -0.4, 0.7)
    assert rec.calls[1][0] == "b200sv_heston_mc_chain"
    assert engine.variable_code(ref["VariableType"].Q_VAR) == C.Q_VAR and engine.variable_code(ref["VariableType"].LOG_RETURN) == C.LOG_RETURN
    with pytest.raises(NotImplementedError):
        engine.variable_code(ref["VariableType"].SIGMA)


def test_reference_hawkes_params_marshal_like_our_own(ref, monkeypatch):
    """the reference's own HawkesJDParams (and OptionChain) through HawkesJDPricer: Monte Carlo and Fourier routes, with and without the risk
    kernel -- same C calls, same sixteen floats, same gamma"""
    import stochvolmodels_b200 as svm
    from stochvolmodels_b200 import _capi as C
    rec = Recorder()
    monkeypatch.setattr(C, "call", rec)
    ref_chain, our_chain = _chains(ref)
    kw = dict(sigma=0.4, mean_p=0.04, mean_m=-0.05, theta_p=6.0, lambda_p=7.0, kappa_p=20.0, beta1_p=30.0, beta2_p=-25.0)
    pricer = svm.HawkesJDPricer()
    for chain, plain, gamma in ((ref_chain, ref["hawkes"], ref["hawkes_gamma"]),
                                (our_chain, svm.HawkesJDParams(**kw), svm.HawkesJDParams(risk_premia_gamma=0.3, **kw))):
        pricer.model_mc_price_chain(chain, plain, nb_path=1000, seed=4, distributed=False)
        pricer.price_chain(chain, plain)
        pricer.price_chain(chain, gamma)
    names = [c[0] for c in rec.calls]
    assert names == ["b200sv_hawkesjd_mc_chain", "b200sv_hawkesjd_price_chain", "b200sv_hawkesjd_price_chain"] * 2
    for a, b in zip(rec.calls[:3], rec.calls[3:]):
        assert a == b or all(x == y or (x != x and y != y) for x, y in zip(a[1], b[1]))        # NaN = "no risk kernel" compares by identity
    sixteen = rec.calls[0][1][0]
    assert len(sixteen) == 16 and sixteen[1] == 0.4 and sixteen[6] == 7.0
    gammas = [c[1][11] for c in rec.calls if c[0] == "b200sv_hawkesjd_price_chain"]
    assert gammas[0] != gammas[0] and gammas[1] == 0.3 and gammas[3] == 0.3
