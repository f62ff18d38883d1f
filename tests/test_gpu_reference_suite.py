"""The calls `pymbar.MBAR` makes while the reference's own acceptance tests run (pymbar/tests/test_mbar.py), replayed
against the real kernels: every recorded `solve_mbar_for_all_states` call goes through pymbar_b200.mbar_solvers on
cuda:0 and must reproduce the reference's f_k and Log_W_nk and pass the checks of tests/test_mbar_solvers.py:35-41.
The calls and the reference's answers are stored in tests/golden/reference_suite_calls.npz
(oracle/record_reference_calls.py)."""
import pytest

from tests import _cases

pytestmark = pytest.mark.gpu


def test_reference_acceptance_suite_on_the_gpu_backend():
    import pymbar_b200
    from pymbar_b200 import mbar_solvers as ms

    pymbar_b200._lib.load()                      # fails loudly without the compiled library
    calls = _cases.reference_suite_calls()
    assert len(calls) >= 10
    try:
        for c in calls:
            _cases.replay_reference_suite_call(ms, c)
    finally:
        ms.clear_cache()
    loaded = [ln.split()[-1] for ln in open("/proc/self/maps") if "libmbar_b200.so" in ln]
    assert loaded, "the native library served no call"
