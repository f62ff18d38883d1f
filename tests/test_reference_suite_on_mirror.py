"""The calls `pymbar.MBAR` makes while the reference's own acceptance tests run (pymbar/tests/test_mbar.py), replayed
against the mirror's driver layer with the device replaced by the oracle stand-in: protocol chain, continuation,
unsampled states and gauge handling of pymbar_b200.mbar_solvers must reproduce the reference's f_k and Log_W_nk
(tests/golden/reference_suite_calls.npz, oracle/record_reference_calls.py)."""
import pymbar_b200
from pymbar_b200 import mbar_solvers as ms
from tests import _cases
from tests.test_driver_logic_cpu import OracleProblem


def test_reference_solver_tests_pass_on_the_mirror(monkeypatch):
    monkeypatch.setattr(ms, "DeviceProblem", OracleProblem)
    monkeypatch.setattr(pymbar_b200._lib, "load", lambda: None)
    monkeypatch.setenv("PYMBAR_B200_CACHE", "0")
    calls = _cases.reference_suite_calls()
    assert len(calls) >= 10
    for c in calls:
        _cases.replay_reference_suite_call(ms, c)
