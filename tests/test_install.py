"""pymbar_b200.install(): attribute rebinding on a pymbar.mbar_solvers-like module (mbar.py:413,437,455,910
resolve the solver through module attributes at call time)."""
import os
import sys
import types

import numpy as np
import pytest

from tests import _cases
from tests._cases import pymbar_importable  # noqa: F401  (fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_install_rebinds_real_pymbar_when_available(pymbar_importable):
    import pymbar.mbar_solvers as ref_ms

    import pymbar_b200
    from pymbar_b200 import mbar_solvers as ours

    orig = ref_ms.solve_mbar_for_all_states
    pymbar_b200.install()
    assert ref_ms.solve_mbar_for_all_states is ours.solve_mbar_for_all_states
    assert ref_ms.mbar_log_W_nk is ours.mbar_log_W_nk and ref_ms.jax_mbar_gradient is ours.mbar_gradient
    # (MBAR.__init__ mutates the reference's module-level protocol dicts in place, mbar.py:391-406:
    # compare the parts it never touches)
    assert [d["method"] for d in ref_ms.DEFAULT_SOLVER_PROTOCOL] == [d["method"] for d in ours.DEFAULT_SOLVER_PROTOCOL]
    import pymbar.mbar as mbar_mod
    from pymbar_b200 import utils as ours_utils

    assert mbar_mod.kln_to_kn is ours_utils.kln_to_kn
    pymbar_b200.uninstall()
    assert ref_ms.solve_mbar_for_all_states is orig
    assert mbar_mod.kln_to_kn is not ours_utils.kln_to_kn


@pytest.mark.gpu
def test_installed_backend_serves_an_mbar_like_caller():
    """What MBAR.__init__ does with the module (mbar.py:413-415, :455), against a stand-in module."""
    import pymbar_b200

    fake = types.ModuleType("fake_mbar_solvers")
    for name in ("solve_mbar_for_all_states", "mbar_log_W_nk", "self_consistent_update", "mbar_gradient"):
        setattr(fake, name, lambda *a, **k: (_ for _ in ()).throw(AssertionError("numpy path called")))
    pymbar_b200.install(fake)
    try:
        z = _cases.load("small_empty_state")
        u_kn = np.array(z["u_kn"], dtype=np.float64)
        N_k = z["N_k"]
        sws = np.where(N_k != 0)[0]
        proto = tuple(dict(s) for s in pymbar_b200.mbar_solvers.DEFAULT_SOLVER_PROTOCOL)
        f_k = fake.solve_mbar_for_all_states(u_kn, N_k, np.zeros(len(N_k)), sws, proto)
        assert np.max(np.abs(f_k - z["fk_default"])) < 1e-8
        logW = fake.mbar_log_W_nk(u_kn, N_k, f_k)
        assert logW.shape == (u_kn.shape[1], u_kn.shape[0]) and logW.flags.writeable
        np.testing.assert_allclose(np.exp(logW)[:, sws].sum(0), 1.0, atol=1e-9)   # tests/test_mbar_solvers.py:37
        np.testing.assert_allclose(np.exp(logW) @ N_k, 1.0, atol=1e-9)            # :38
    finally:
        pymbar_b200.uninstall()
        pymbar_b200.mbar_solvers.clear_cache()


def test_environment_switch_installs_at_import(pymbar_importable):
    """PYMBAR_B200=1: importing pymbar_b200 alone rebinds pymbar.mbar_solvers (SURVEY.md section 5)."""
    import subprocess

    env = dict(os.environ, PYMBAR_B200="1", PYMBAR_DISABLE_JAX="1",
               PYTHONPATH=os.pathsep.join([ROOT] + [p for p in sys.path if p]))
    code = ("import pymbar_b200, pymbar.mbar_solvers as m, pymbar.mbar as mb; "
            "from pymbar_b200 import mbar_solvers as o; "
            "assert m.solve_mbar_for_all_states is o.solve_mbar_for_all_states; "
            "assert isinstance(mb.MBAR.__dict__['Log_W_nk'], property); print('SWITCH_OK')")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert "SWITCH_OK" in out.stdout, out.stdout + out.stderr[-2000:]
