"""BAR initialisation (SURVEY.md 8f row N4, mbar.py:1936-1988): pymbar_b200.initialize vs the reference's
`MBAR._initialize_with_bar` (stored answer) and vs the identity BAR == two-state MBAR."""
import os

import numpy as np

from oracle import mbar_oracle as orc
from oracle import testsystems as ots
from pymbar_b200.initialize import bar_delta_f, initialize_with_bar

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bar_equals_two_state_mbar():
    _, u_kn, N_k = ots.harmonic_u_kn([0.0, 1.5], [1.0, 3.0], [400, 250], seed=5)
    f = orc.mbar_f_k(u_kn, N_k)
    w_F = u_kn[1, :400] - u_kn[0, :400]
    w_R = u_kn[0, 400:] - u_kn[1, 400:]
    dF = bar_delta_f(w_F, w_R, rtol=1e-12)
    assert abs(dF - (f[1] - f[0])) < 1e-9


def test_chain_with_an_empty_state_and_a_start_vector():
    _, u_kn, N_k = ots.harmonic_u_kn([0, 1, 2, 3], [1, 2, 4, 8], [100, 50, 0, 80], seed=3)
    x_k = np.repeat(np.arange(4), N_k)
    f = initialize_with_bar(u_kn, N_k, x_k)
    assert f[0] == 0 and f[2] == 0                      # unsampled states are left alone
    pair = np.concatenate([np.arange(0, 100), np.arange(100, 150)])
    f2 = orc.mbar_f_k(u_kn[:2][:, pair], np.array([100, 50]))
    assert abs(f[1] - f2[1]) < 1e-4
    g = initialize_with_bar(u_kn, N_k, x_k, f_k_init=np.array([5.0, 0, 0, 0]))
    s = N_k > 0
    np.testing.assert_allclose((g - g[0])[s], (f - f[0])[s], atol=1e-4)


def test_matches_the_reference_initialisation():
    # the reference's MBAR._initialize_with_bar on this sample (oracle/make_golden.py --only-bar-init)
    z = np.load(os.path.join(ROOT, "tests", "golden", "bar_init_5.npz"))
    mine = initialize_with_bar(z["u_kn"], z["N_k"], z["x_kindices"])
    assert np.max(np.abs(z["f_bar"] - mine)) < 1e-4          # both solve Bennett's equation to rtol 1e-5
