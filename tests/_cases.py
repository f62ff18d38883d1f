"""Shared helpers: load golden fixtures and regenerate their inputs (oracle-side, tests only)."""
import ast
import hashlib
import importlib.util
import os
import sys

import numpy as np
import pytest

from oracle import testsystems as ots

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PYMBAR_STAND_IN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_pymbar_stand_in")

SMALL = ["small_osc_8x40", "small_exp_6x50", "small_empty_state", "small_empty_first"]
MEDIUM = ["osc_50x100", "osc_100x100", "osc_200x50", "exp_200x50"]
C1 = ["c1_harmonic_5x1000"]     # BASELINE.json configs[0]: HarmonicOscillatorsTestCase() defaults, K=5, N=5000
ALL = ["golden_example"] + SMALL + MEDIUM + C1


def _regen(spec):
    kind = spec[0]
    if kind == "harmonic":
        _, O, K, N, seed = spec
        return ots.harmonic_u_kn(O, K, N, seed=seed)[1]
    if kind == "exponential":
        _, rates, N, seed = spec
        return ots.exponential_u_kn(rates, N, seed=seed)[1]
    if kind == "osc":
        return ots.oscillators(spec[1], spec[2], seed=spec[3])[0]
    if kind == "exp":
        return ots.exponentials(spec[1], spec[2], seed=spec[3])[0]
    raise ValueError(kind)


def load(name):
    z = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))
    if "u_kn" not in z:
        spec = ast.literal_eval(str(z["regen"]).replace("np.float64", ""))
        z["u_kn"] = _regen(spec)
    sha = hashlib.sha256(np.ascontiguousarray(z["u_kn"]).tobytes()).hexdigest()
    assert sha == str(z["u_sha"]), f"{name}: regenerated input differs from the fixture's input"
    z["N_k"] = z["N_k"].astype(np.int64)
    return z


def reference_suite_calls():
    """The `solve_mbar_for_all_states` calls pymbar.MBAR made while the reference's own test_mbar.py ran on the
    reference (oracle/record_reference_calls.py): inputs, the reference's f_k and sampled rows of its Log_W_nk."""
    z = np.load(os.path.join(GOLDEN_DIR, "reference_suite_calls.npz"), allow_pickle=False)
    calls = []
    for i in range(int(z["n_calls"])):
        c = {k: z[f"c{i}_{k}"] for k in ("u_kn", "N_k", "f_init", "sws", "f_k", "logW_rows", "logW")}
        c["test"] = str(z[f"c{i}_test"])
        c["protocol"] = ast.literal_eval(str(z[f"c{i}_protocol"]))
        assert hashlib.sha256(c["u_kn"].tobytes()).hexdigest() == str(z[f"c{i}_u_sha"]), c["test"]
        calls.append(c)
    return calls


def replay_reference_suite_call(ms, c):
    """One recorded call through the backend module `ms`, checked against the reference's answers and against the
    assertions of the reference's tests/test_mbar_solvers.py:35-41 (gradient zero, weights normalised, fixed point)."""
    u, N_k, sws = c["u_kn"], c["N_k"], c["sws"]
    proto = tuple(dict(s, options=dict(s.get("options") or {})) for s in c["protocol"])
    f = ms.solve_mbar_for_all_states(u.copy(), N_k.copy(), c["f_init"].copy(), sws.copy(), proto)
    np.testing.assert_allclose(f, c["f_k"], atol=1e-8, err_msg=c["test"])
    lw = ms.mbar_log_W_nk(u, N_k, f)
    np.testing.assert_allclose(lw[c["logW_rows"]], c["logW"], atol=1e-8, err_msg=c["test"])
    W = np.exp(lw)
    np.testing.assert_allclose(W[:, sws].sum(0), 1.0, atol=1e-10, err_msg=c["test"])
    np.testing.assert_allclose(W @ N_k, 1.0, atol=1e-10, err_msg=c["test"])
    s = N_k > 0
    np.testing.assert_allclose(ms.mbar_gradient(u[s], N_k[s], f[s]), 0.0, atol=1e-8, err_msg=c["test"])
    np.testing.assert_allclose(ms.self_consistent_update(u, N_k, f), f, atol=1e-10, err_msg=c["test"])


@pytest.fixture()
def pymbar_importable(monkeypatch):
    """`import pymbar` works inside the test: the installed package where there is one, else the stand-in in
    tests/_pymbar_stand_in (same module layout, calls the backend the way pymbar's MBAR does)."""
    if importlib.util.find_spec("pymbar") is not None:
        yield
        return
    monkeypatch.syspath_prepend(PYMBAR_STAND_IN)
    yield
    for name in [m for m in sys.modules if m == "pymbar" or m.startswith("pymbar.")]:
        del sys.modules[name]
