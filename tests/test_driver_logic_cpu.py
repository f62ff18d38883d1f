"""Host-side driver logic of the mirror (protocol chain, scipy closures, gauge handling, unsampled states,
warnings) exercised through the REAL pymbar.MBAR class on CPU.

The GPU is replaced by a test-only stand-in for DeviceProblem that answers every primitive with the
oracle, so what is tested is exactly the Python layer between pymbar.MBAR and the C ABI.  Where pymbar is not
installed, MBAR is the stand-in of tests/_pymbar_stand_in.  The DeviceProblem stand-in lives here, not in the
product: pymbar_b200 itself has no CPU path."""
import numpy as np
import pytest

from oracle import mbar_oracle as orc
from tests import _cases
from tests._cases import pymbar_importable  # noqa: F401  (fixture)


class OracleProblem:
    """DeviceProblem's interface, answered by oracle/mbar_oracle.py (test infrastructure)."""

    def __init__(self, u_kn, N_k, device=0, N_local=None):
        self.u = np.array(u_kn, dtype=np.float64)
        self.N_k = np.asarray(N_k, dtype=np.float64)
        self.K, self.N = self.u.shape
        self.s = self.N_k > 0

    def close(self):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        pass

    def weight_moments(self, f):
        W = orc.mbar_W_nk(self.u, self.N_k, np.asarray(f, float))
        return W.sum(0), W.T @ W

    def augmented(self, u_extra):
        u_extra = np.atleast_2d(np.asarray(u_extra, float))
        return OracleProblem(np.vstack([self.u, u_extra]), np.concatenate([self.N_k, np.zeros(len(u_extra))]))

    def _sub(self, f):
        return self.u[self.s], self.N_k[self.s], np.asarray(f, float)[self.s]

    def self_consistent_update(self, f):
        return orc.self_consistent_update(self.u, self.N_k, np.asarray(f, float))

    def gradient(self, f):
        g = np.zeros(self.K)
        g[self.s] = orc.mbar_gradient(*self._sub(f))
        return g

    def objective_and_gradient(self, f):
        o, gs = orc.mbar_objective_and_gradient(*self._sub(f))
        g = np.zeros(self.K)
        g[self.s] = gs
        return float(o), g

    def objective(self, f):
        return float(orc.mbar_objective(*self._sub(f)))

    def hessian(self, f):
        H = np.zeros((self.K, self.K))
        H[np.ix_(self.s, self.s)] = orc.mbar_hessian(*self._sub(f))
        return H

    def log_W_nk(self, f, exponentiate=False, out=None):
        lw = orc.mbar_log_W_nk(self.u, self.N_k, np.asarray(f, float))
        return np.exp(lw) if exponentiate else lw

    def log_denominator(self, f):
        return orc.log_denominator_n(*self._sub(f))

    def streaming_pass(self, f, want_G=False):
        S = np.zeros(self.K)
        Ss, L = orc.single_pass_sums(*self._sub(f))
        S[self.s] = Ss
        return S, float(L.sum()), None

    def solve_adaptive(self, f, tol=1e-12, maxiter=10000, min_sc_iter=2, gamma=1.0):
        u, N, fs = self._sub(f)
        r = orc.adaptive(u, N, fs - fs[0], tol=tol, options=dict(maxiter=maxiter, min_sc_iter=min_sc_iter, gamma=gamma))
        out = np.array(f, dtype=float)
        out[self.s] = r["x"]
        return out, dict(success=int(r["success"]), iterations=len(r["history"]), nr_iterations=r["nr_iter"],
                         sci_iterations=r["sci_iter"], passes=0, hessian_passes=0, max_delta=0.0, gnorm=0.0,
                         device_ms=0.0)


@pytest.fixture()
def patched_pymbar(monkeypatch, pymbar_importable):
    import pymbar

    import pymbar_b200
    from pymbar_b200 import mbar_solvers as ours

    monkeypatch.setattr(ours, "DeviceProblem", OracleProblem)
    monkeypatch.setenv("PYMBAR_B200_CACHE", "0")
    monkeypatch.setattr(pymbar_b200._lib, "load", lambda: None)
    pymbar_b200.install()
    yield pymbar
    pymbar_b200.uninstall()


@pytest.mark.parametrize("name", _cases.SMALL + ["golden_example"])
@pytest.mark.parametrize("protocol", ["default", "robust"])
def test_mbar_class_on_the_mirror(patched_pymbar, name, protocol):
    z = _cases.load(name)
    m = patched_pymbar.MBAR(z["u_kn"], z["N_k"], solver_protocol=protocol)
    assert np.max(np.abs(m.f_k - z[f"fk_{protocol}"])) < 1e-9
    np.testing.assert_allclose(np.exp(m.Log_W_nk) @ z["N_k"], 1.0, atol=1e-9)     # tests/test_mbar_solvers.py:38
    r = m.compute_free_energy_differences()
    if "est_dDelta_f" in z and protocol == "default":
        np.testing.assert_allclose(r["dDelta_f"], z["est_dDelta_f"], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("method", ["adaptive", "hybr", "lm", "L-BFGS-B", "BFGS", "Newton-CG", "trust-ncg", "SLSQP"])
def test_protocol_methods_of_the_reference_suite(patched_pymbar, method):
    """tests/test_mbar_solvers.py:57-91 drives these methods through MBAR(solver_protocol=({"method": m},))."""
    z = _cases.load("small_osc_8x40")
    m = patched_pymbar.MBAR(z["u_kn"], z["N_k"], solver_protocol=({"method": method},))
    m = patched_pymbar.MBAR(z["u_kn"], z["N_k"], initial_f_k=m.f_k, solver_protocol=({"method": method},))
    assert np.max(np.abs(m.f_k - z["fk_default"])) < 1e-6


def test_bootstrap_through_mbar_class(patched_pymbar):
    z = _cases.load("small_exp_6x50")
    m = patched_pymbar.MBAR(z["u_kn"], z["N_k"], n_bootstraps=4, rseed=11)
    np.testing.assert_array_equal(m.bootstrap_rints, z["boot_rints"])
    assert np.max(np.abs(m.f_k_boots - z["boot_f_k"])) < 1e-9


def test_three_dimensional_input_and_bad_method(patched_pymbar):
    from pymbar_b200.utils import ParameterError

    z = _cases.load("small_osc_8x40")
    K, N = z["u_kn"].shape
    n = N // K
    u_kln = np.zeros((K, K, n))
    for k in range(K):
        u_kln[k] = z["u_kn"][:, k * n:(k + 1) * n]
    m = patched_pymbar.MBAR(u_kln, z["N_k"])
    assert np.max(np.abs(m.f_k - z["fk_default"])) < 1e-9
    with pytest.raises(patched_pymbar.utils.ParameterError):          # pymbar's own class after install()
        patched_pymbar.MBAR(z["u_kn"], z["N_k"], solver_protocol=({"method": "no-such-method"},))
    del ParameterError


def test_facade_lazy_log_weights_and_device_moments(patched_pymbar):
    """SURVEY 8f N1 / N2 through the real MBAR class (pymbar_b200/facade.py): Log_W_nk is a ticket until somebody
    reads it; N_eff, overlap and dDelta_f come from the K x K moments; every number equals what the unmodified
    reference produced for the fixture (oracle/make_golden.py)."""
    from pymbar_b200 import facade

    z = _cases.load("small_osc_8x40")
    s0 = dict(facade.STATS)
    m = patched_pymbar.MBAR(z["u_kn"], z["N_k"])
    assert facade.STATS["tickets"] == s0["tickets"] + 1 and facade.STATS["redeemed"] == s0["redeemed"]
    assert isinstance(m.__dict__["_b200_logw"], facade.LogWeightTicket)          # nothing downloaded yet
    r = m.compute_free_energy_differences(return_theta=True)
    np.testing.assert_allclose(r["Delta_f"], z["est_Delta_f"], atol=1e-9)
    np.testing.assert_allclose(r["dDelta_f"], z["est_dDelta_f"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(r["Theta"], z["est_Theta"], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(m.compute_effective_sample_number(), z["est_N_eff"], rtol=1e-8)
    ov = m.compute_overlap()
    np.testing.assert_allclose(ov["matrix"], z["est_overlap_matrix"], rtol=1e-7, atol=1e-12)
    np.testing.assert_allclose(np.real(ov["scalar"]), z["est_overlap_scalar"], rtol=1e-7)
    assert facade.STATS["redeemed"] == s0["redeemed"] and facade.STATS["moments"] == s0["moments"] + 1
    # expectations / perturbed free energies: the routine behind them is served by the augmented problem
    x = z["x_n"]
    e = m.compute_expectations(x.copy())
    np.testing.assert_allclose(e["mu"], z["expt_avg_mu"], rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(e["sigma"], z["expt_avg_sigma"], rtol=1e-5, atol=1e-9)
    pf = m.compute_perturbed_free_energies(z["pert_u_ln"].copy())
    np.testing.assert_allclose(pf["Delta_f"], z["pert_Delta_f"], atol=1e-8)
    np.testing.assert_allclose(pf["dDelta_f"], z["pert_dDelta_f"], rtol=1e-5, atol=1e-9)
    assert facade.STATS["redeemed"] == s0["redeemed"] and facade.STATS["expectations"] >= s0["expectations"] + 2
    # the first read downloads the matrix: a plain writable ndarray, as in the reference
    lw = m.Log_W_nk
    assert isinstance(lw, np.ndarray) and lw.flags.writeable and lw.shape == (z["u_kn"].shape[1], z["u_kn"].shape[0])
    assert facade.STATS["redeemed"] == s0["redeemed"] + 1
    np.testing.assert_allclose(np.exp(lw) @ z["N_k"], 1.0, atol=1e-9)
    assert m.Log_W_nk is lw                                                        # cached after the first read
    # uncertainty methods outside the device path fall through to the original implementation
    r_svd = m.compute_free_energy_differences(uncertainty_method="svd")
    np.testing.assert_allclose(r_svd["dDelta_f"], r["dDelta_f"], rtol=1e-6, atol=1e-9)


def test_facade_bar_initialisation_and_uninstall(patched_pymbar):
    import pymbar_b200

    z = _cases.load("small_empty_state")
    m = patched_pymbar.MBAR(z["u_kn"], z["N_k"], initialize="BAR")
    assert np.max(np.abs(m.f_k - z["fk_default"])) < 1e-8                          # the start only seeds the solver
    cls = patched_pymbar.mbar.MBAR
    assert isinstance(cls.__dict__["Log_W_nk"], property)
    pymbar_b200.uninstall()
    assert "Log_W_nk" not in cls.__dict__ and cls.compute_overlap.__module__ == "pymbar.mbar"
    pymbar_b200.install()                                                          # (the fixture uninstalls again)
