"""Stand-in for the pymbar package — TEST INFRASTRUCTURE, used only where pymbar itself is not installed.

pymbar_b200 plugs into pymbar: `pymbar_b200.install()` rebinds the entry points of `pymbar.mbar_solvers`, the
layout helpers `pymbar.mbar` imported from `pymbar.utils`, and methods of `pymbar.mbar.MBAR` (facade.py).  The
tests of that integration need a caller with the same module layout that calls the backend the way pymbar 4's
MBAR does: solver and log-weight entry points looked up as `mbar_solvers` attributes at call time, 3-D input
converted through the `kln_to_kn` name of its own module, estimators and expectations through the methods the
facade replaces.  This package is such a caller, written for the tests; every number the tests check comes from
pymbar_b200 and is compared with answers the unmodified pymbar produced (tests/golden/).
"""
from . import mbar, mbar_solvers, utils  # noqa: F401
from .mbar import MBAR  # noqa: F401
