#!/usr/bin/env python
"""Record the solver calls the reference's own acceptance tests make — TEST INFRASTRUCTURE.

Runs pymbar/tests/test_mbar_solvers.py and pymbar/tests/test_mbar.py of an unmodified pymbar checkout
(path in PYMBAR_REFERENCE, default ../reference next to the repository) on the reference's CPU solver,
with this module loaded as a pytest plugin.  Every `solve_mbar_for_all_states` call that `pymbar.MBAR`
makes is captured; a bounded selection (distinct inputs, at most two calls of each test,
small inputs only) is stored with the reference's answer and a seeded sample of rows of `mbar_log_W_nk`
at that answer in tests/golden/reference_suite_calls.npz.  tests/test_gpu_reference_suite.py and
tests/test_reference_suite_on_mirror.py replay those calls through pymbar_b200.mbar_solvers.

    python oracle/record_reference_calls.py
"""
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden", "reference_suite_calls.npz")
MAX_ENTRIES = 12_000          # u_kn entries per stored call (keeps the fixture well under 1 MB)
MAX_CALLS = 11
LOGW_ROWS = 64

_CALLS = []
_SEEN = set()


def pytest_configure(config):
    import pymbar.mbar_solvers as ms

    solve = ms.solve_mbar_for_all_states

    def recording_solve(u_kn, N_k, f_k, states_with_samples, solver_protocol):
        f_init = np.array(f_k, dtype=np.float64)
        out = solve(u_kn, N_k, f_k, states_with_samples, solver_protocol)
        test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0]
        u = np.asarray(u_kn, dtype=np.float64)
        key = (hashlib.sha256(u.tobytes()).hexdigest(), f_init.tobytes(), repr(solver_protocol))
        per_test = sum(c["test"] == test for c in _CALLS)
        if key not in _SEEN and per_test < 2 and u.size <= MAX_ENTRIES and len(_CALLS) < MAX_CALLS:
            _SEEN.add(key)
            _CALLS.append(dict(test=test, u_kn=u.copy(), N_k=np.asarray(N_k, dtype=np.int64).copy(), f_init=f_init,
                               sws=np.asarray(states_with_samples, dtype=np.int64).copy(),
                               protocol=repr(tuple(dict(s) for s in solver_protocol)),
                               f_k=np.array(out, dtype=np.float64)))
        return out

    ms.solve_mbar_for_all_states = recording_solve


def pytest_sessionfinish(session, exitstatus):
    import pymbar.mbar_solvers as ms

    data = {}
    rng = np.random.RandomState(2024)
    for i, c in enumerate(_CALLS):
        lw = ms.mbar_log_W_nk(c["u_kn"], c["N_k"], c["f_k"])
        rows = np.sort(rng.choice(lw.shape[0], size=min(LOGW_ROWS, lw.shape[0]), replace=False))
        for k in ("u_kn", "N_k", "f_init", "sws", "f_k"):
            data[f"c{i}_{k}"] = c[k]
        data[f"c{i}_test"] = np.array(c["test"])
        data[f"c{i}_protocol"] = np.array(c["protocol"])
        data[f"c{i}_logW_rows"] = rows
        data[f"c{i}_logW"] = lw[rows]
        data[f"c{i}_u_sha"] = np.array(hashlib.sha256(c["u_kn"].tobytes()).hexdigest())
    data["n_calls"] = np.int64(len(_CALLS))
    np.savez_compressed(OUT, **data)
    print(f"\nrecorded {len(_CALLS)} calls into {os.path.relpath(OUT, ROOT)} ({os.path.getsize(OUT)} bytes)")


def main():
    ref = os.path.abspath(os.environ.get("PYMBAR_REFERENCE", os.path.join(ROOT, "..", "reference")))
    tests = os.path.join(ref, "pymbar", "tests")
    if not os.path.isdir(tests):
        raise SystemExit(f"no pymbar checkout at {ref} (set PYMBAR_REFERENCE)")
    env = dict(os.environ, PYMBAR_DISABLE_JAX="1",
               PYTHONPATH=os.pathsep.join([ROOT, os.path.join(HERE, "ref_shim"), ref]))
    # fixed global seed: the reference's test systems draw from numpy's global RNG
    code = ("import numpy, sys, pytest; numpy.random.seed(7); "
            "sys.exit(pytest.main(sys.argv[1:]))")
    cmd = [sys.executable, "-c", code, "-q", "-p", "oracle.record_reference_calls", "-p", "no:cacheprovider",
           "-W", "ignore::pytest.PytestUnknownMarkWarning",
           os.path.join(tests, "test_mbar_solvers.py"), os.path.join(tests, "test_mbar.py")]
    raise SystemExit(subprocess.call(cmd, cwd=tempfile.gettempdir(), env=env))


if __name__ == "__main__":
    main()
