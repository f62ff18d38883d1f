#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference — TEST INFRASTRUCTURE.

Runs only in the build container (needs /root/reference).  Imports pymbar from
/root/reference through the numexpr stub in oracle/ref_shim (SURVEY.md Appendix C), exercises
the solver path on seeded inputs and stores the outputs.  Small cases store their u_kn; larger
cases store only outputs plus a SHA-256 of the input bytes, and tests regenerate the input with
oracle/testsystems.py (this script asserts that regeneration is bit-exact).

    python oracle/make_golden.py
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "ref_shim"))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)
os.environ["PYMBAR_DISABLE_JAX"] = "1"

import pymbar  # noqa: E402  (the real reference)
from pymbar import mbar_solvers as ref  # noqa: E402
from pymbar import testsystems as ref_ts  # noqa: E402

from oracle import testsystems as ots  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


LAST_X = [None]   # positions of the most recently sampled test system (observable for expectations)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ref_harmonic(O_k, K_k, N_k, seed):
    tc = ref_ts.harmonic_oscillators.HarmonicOscillatorsTestCase(O_k=O_k, K_k=K_k)
    x_n, u_kn, N_out, _ = tc.sample(N_k, mode="u_kn", seed=seed)
    LAST_X[0] = np.array(x_n)
    return u_kn, np.asarray(N_out)


def ref_exponential(rates, N_k, seed):
    tc = ref_ts.exponential_distributions.ExponentialTestCase(rates)
    x_n, u_kn, N_out, _ = tc.sample(N_k, mode="u_kn", seed=seed)
    LAST_X[0] = np.array(x_n)
    return u_kn, np.asarray(N_out)


def primitives(u_kn, N_k, f):
    Nf = np.asarray(N_k, float)
    sampled = Nf > 0
    out = dict(
        sci=ref.self_consistent_update(u_kn, Nf, f),
        logW=ref.mbar_log_W_nk(u_kn, Nf, f),
    )
    # gradient / objective / hessian are only meaningful for sampled rows in the reference's solver
    us, Ns, fs = u_kn[sampled], Nf[sampled], f[sampled]
    out["grad"] = ref.mbar_gradient(us, Ns, fs)
    out["obj"] = np.float64(ref.mbar_objective(us, Ns, fs))
    out["hess"] = ref.mbar_hessian(us, Ns, fs)
    return out


def solve_all(u_kn, N_k):
    res = {}
    for name, proto in (
        ("default", "default"),
        ("robust", "robust"),
        ("adaptive", (dict(method="adaptive", options=dict(min_sc_iter=0)),)),
        ("adaptive_msi2", (dict(method="adaptive"),)),
    ):
        m = pymbar.MBAR(u_kn, N_k, solver_protocol=proto)
        res[name] = np.array(m.f_k)
    return res


def case(name, u_kn, N_k, store_u, regen, rng):
    K = u_kn.shape[0]
    N_k = np.asarray(N_k, np.int64)
    f_rand = rng.normal(scale=1.5, size=K)
    f_rand -= f_rand[0]
    data = dict(N_k=N_k, f_rand=f_rand, u_sha=np.array(sha(u_kn)), regen=np.array(repr(regen)))
    if store_u:
        data["u_kn"] = u_kn
    for tag, f in (("zero", np.zeros(K)), ("rand", f_rand)):
        for k, v in primitives(u_kn, N_k, f).items():
            if k in ("logW", "hess") and not store_u:
                # keep big fixtures out of git: store a few probes of the big outputs instead
                if k == "hess":
                    data[f"{tag}_hess_diag"] = np.diag(v).copy()
                    data[f"{tag}_hess_row1"] = v[min(1, v.shape[0] - 1)].copy()
                    data[f"{tag}_hess_fro"] = np.float64(np.linalg.norm(v))
                else:
                    data[f"{tag}_logW_colsum"] = v.sum(0)
                    data[f"{tag}_logW_head"] = v[:4].copy()
                continue
            data[f"{tag}_{k}"] = v
    for pname, fk in solve_all(u_kn, N_k).items():
        data[f"fk_{pname}"] = fk
    if K <= 64:
        # estimators of SURVEY 8f N1 at the converged default solution (mbar.py:620, :563, :496)
        m = pymbar.MBAR(u_kn, N_k)
        r = m.compute_free_energy_differences(uncertainty_method="svd-ew", return_theta=True)
        data["est_dDelta_f"] = np.array(r["dDelta_f"])
        data["est_Theta"] = np.array(r["Theta"])
        data["est_Delta_f"] = np.array(r["Delta_f"])
        ov = m.compute_overlap()
        data["est_overlap_matrix"] = np.array(ov["matrix"])
        data["est_overlap_scalar"] = np.float64(np.real(ov["scalar"]))
        data["est_N_eff"] = np.array(m.compute_effective_sample_number())
        W = np.exp(m.Log_W_nk)
        data["est_G"] = W.T @ W
    if store_u:
        # expectations / perturbed free energies (mbar.py:1124, :1442) at the default solution
        me = pymbar.MBAR(u_kn, N_k)
        x_n = LAST_X[0]
        data["x_n"] = x_n.copy()
        r = me.compute_expectations(x_n.copy())           # (the reference shifts A_n in place)
        data["expt_avg_mu"], data["expt_avg_sigma"] = np.array(r["mu"]), np.array(r["sigma"])
        r = me.compute_expectations(x_n.copy(), output="differences")
        data["expt_diff_mu"], data["expt_diff_sigma"] = np.array(r["mu"]), np.array(r["sigma"])
        r = me.compute_expectations(u_kn.copy(), state_dependent=True)
        data["expt_sd_mu"], data["expt_sd_sigma"] = np.array(r["mu"]), np.array(r["sigma"])
        u_ln = np.vstack([0.5 * (u_kn[0] + u_kn[1]), 1.3 * u_kn[-1], u_kn[0] + 0.2 * x_n])
        data["pert_u_ln"] = u_ln
        r = me.compute_perturbed_free_energies(u_ln.copy())
        data["pert_Delta_f"], data["pert_dDelta_f"] = np.array(r["Delta_f"]), np.array(r["dDelta_f"])
        # bootstrap replicates (mbar.py:417-449) with a fixed rseed: indices and the re-solved f_k
        mb = pymbar.MBAR(u_kn, N_k, n_bootstraps=4, rseed=11)
        data["boot_rints"] = np.array(mb.bootstrap_rints)
        data["boot_f_k"] = np.array(mb.f_k_boots)
        data["boot_f_k_start"] = np.array(mb.f_k)
    # adaptive trajectory from f=0 on sampled states (mbar_solvers.py:510-667), tol 1e-12
    sampled = N_k > 0
    us = ref.precondition_u_kn(u_kn[sampled], 1.0 * N_k[sampled], np.zeros(sampled.sum()))
    r = ref.adaptive(us, 1.0 * N_k[sampled], np.zeros(sampled.sum()), tol=1e-12,
                     options=dict(min_sc_iter=0))
    data["adaptive_x"] = np.array(r["x"])
    data["adaptive_success"] = np.array(bool(r["success"]))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **data)
    print(f"{name}: K={K} N={u_kn.shape[1]} stored_u={store_u} "
          f"fk_default[:4]={data['fk_default'][:4]}")


def c1_case():
    """BASELINE.json configs[0] (C1): HarmonicOscillatorsTestCase() defaults, K=5, N_k=[1000]*5, seed 0
    (SURVEY.md 8d).  Separate RNG stream so the older fixtures stay byte-identical; also pins
    precondition_u_kn (mbar_solvers.py:710-735, row a6) through probes of its output."""
    rng = np.random.RandomState(4321)
    O, Kk, Nk = [0.0, 1.0, 2.0, 3.0, 4.0], [1.0, 2.0, 4.0, 8.0, 16.0], [1000] * 5
    u, N = ref_harmonic(O, Kk, Nk, 0)
    _, u2, _ = ots.harmonic_u_kn(O, Kk, Nk, seed=0)
    assert np.array_equal(u, u2), "restated harmonic sampler is not bit-exact"
    case("c1_harmonic_5x1000", u, N, store_u=False, regen=("harmonic", O, Kk, Nk, 0), rng=rng)
    path = os.path.join(OUT, "c1_harmonic_5x1000.npz")
    data = dict(np.load(path, allow_pickle=False))
    Nf = 1.0 * np.asarray(N)
    for tag, f in (("zero", np.zeros(5)), ("rand", data["f_rand"])):
        pc = ref.precondition_u_kn(u, Nf, f)
        data[f"{tag}_precond_head"] = pc[:, :64].copy()
        data[f"{tag}_precond_rowsum"] = pc.sum(1)
        data[f"{tag}_precond_obj"] = np.float64(ref.mbar_objective(pc, Nf, f))
    np.savez_compressed(path, **data)


def bar_init_case():
    """MBAR._initialize_with_bar (mbar.py:1936-1988) on an empty-state harmonic sample: what tests/test_initialize.py
    compares pymbar_b200.initialize with."""
    tc = ref_ts.harmonic_oscillators.HarmonicOscillatorsTestCase(O_k=[0, 1, 2, 3, 4], K_k=[1, 2, 4, 8, 16])
    _, u, N, _ = tc.sample([300, 200, 0, 250, 100], mode="u_kn", seed=3)
    m = pymbar.MBAR(u, N, initialize="zeros")
    np.savez_compressed(os.path.join(OUT, "bar_init_5.npz"), u_kn=np.array(m.u_kn), N_k=np.array(m.N_k),
                        x_kindices=np.array(m.x_kindices), f_bar=np.array(m._initialize_with_bar(m.u_kn)))


def main():
    os.makedirs(OUT, exist_ok=True)
    if "--only-c1" in sys.argv:
        c1_case()
        return
    if "--only-bar-init" in sys.argv:
        bar_init_case()
        return
    rng = np.random.RandomState(1234)

    # --- the reference's literal golden vector ---------------------------------------------
    g = ots.GOLDEN_EXAMPLE
    u_ref, N_ref = ref_harmonic(g["O_k"], g["K_k"], g["N_k"], g["seed"])
    _, u_mine, _ = ots.harmonic_u_kn(g["O_k"], g["K_k"], g["N_k"], seed=g["seed"])
    assert np.array_equal(u_ref, u_mine), "restated harmonic sampler is not bit-exact"
    m = pymbar.MBAR(u_ref, N_ref, relative_tolerance=1.0e-10)
    printed = np.array(g["f_k_printed"])
    assert np.max(np.abs(m.f_k - printed)) < 5e-9, (m.f_k, printed)
    case("golden_example", u_ref, N_ref, store_u=False,
         regen=("harmonic", g["O_k"], g["K_k"], g["N_k"], g["seed"]), rng=rng)

    # --- small cases, inputs stored ----------------------------------------------------------
    O, Kk, Nk = np.linspace(1, 5, 8), np.linspace(1, 3, 8), [40] * 8
    u, N = ref_harmonic(O, Kk, Nk, 1)
    case("small_osc_8x40", u, N, True, ("harmonic", list(O), list(Kk), Nk, 1), rng)

    rates, Nk = np.linspace(1, 3, 6), [50] * 6
    u, N = ref_exponential(rates, Nk, 2)
    case("small_exp_6x50", u, N, True, ("exponential", list(rates), Nk, 2), rng)

    # tests/test_mbar.py:16 fixture shape: an empty state in the middle
    O, Kk, Nk = [0, 1, 2, 3], [1, 2, 4, 8], [100, 50, 0, 80]
    u, N = ref_harmonic(O, Kk, Nk, 3)
    case("small_empty_state", u, N, True, ("harmonic", O, Kk, Nk, 3), rng)

    # empty FIRST state (f_0 gauge applied after the all-state pass, mbar_solvers.py:1012-1015)
    O, Kk, Nk = [0, 1, 2, 3, 4], [4, 4, 2, 2, 1], [0, 60, 60, 0, 60]
    u, N = ref_harmonic(O, Kk, Nk, 4)
    case("small_empty_first", u, N, True, ("harmonic", O, Kk, Nk, 4), rng)

    # --- the shapes tests/test_mbar_solvers.py:25-41 uses; inputs regenerated -----------------
    for (ks, ns, kind, seed) in ((50, 100, "osc", 10), (100, 100, "osc", 11),
                                 (200, 50, "osc", 12), (200, 50, "exp", 13)):
        if kind == "osc":
            O, Kk = np.linspace(1, 5, ks), np.linspace(1, 3, ks)
            u, N = ref_harmonic(O, Kk, [ns] * ks, seed)
            u2, _ = ots.oscillators(ks, ns, seed=seed)
        else:
            rates = np.linspace(1, 3, ks)
            u, N = ref_exponential(rates, [ns] * ks, seed)
            u2, _ = ots.exponentials(ks, ns, seed=seed)
        assert np.array_equal(u, u2), "restated sampler is not bit-exact"
        case(f"{kind}_{ks}x{ns}", u, N, False, (kind, ks, ns, seed), rng)
    c1_case()


if __name__ == "__main__":
    main()
