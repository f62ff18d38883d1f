"""pymbar.mbar.MBAR for the stand-in (see the package docstring).

The constructor follows the order of pymbar 4's: 3-D input through `kln_to_kn`, the duplicate-state check that
spends one draw of the seeded generator, the initial f_k (given, zeros or BAR), the solver protocols completed
with `continuation` / `maxiter` / `verbose`, `mbar_solvers.solve_mbar_for_all_states`, the bootstrap replicates
drawn per state from the same generator, then `mbar_solvers.mbar_log_W_nk`.  Estimators the facade does not
serve on the device (`uncertainty_method="svd"`) are computed here from Log_W_nk.  Methods the facade provides
(`compute_expectations_inner`, `_initialize_with_bar`) have no stand-in implementation."""
import numpy as np

from pymbar import mbar_solvers
from pymbar.utils import ParameterError, kln_to_kn


def _complete_protocol(protocol, default, robust, maximum_iterations, verbose):
    if protocol is None or protocol == "default":
        protocol = default
    elif protocol == "robust":
        protocol = robust
    out = []
    for solver in protocol:
        s = dict(solver)
        s["options"] = dict(s.get("options") or {})
        s.setdefault("continuation", None)
        s["options"]["maxiter"] = max(s["options"].get("maxiter", maximum_iterations), maximum_iterations)
        s["options"].setdefault("verbose", verbose)
        out.append(s)
    return tuple(out)


class MBAR:
    def __init__(self, u_kn, N_k, maximum_iterations=10000, relative_tolerance=1.0e-7, verbose=False,
                 initial_f_k=None, solver_protocol=None, initialize="zeros", x_kindices=None, rseed=None,
                 n_bootstraps=0, bootstrap_solver_protocol=None):
        self.N_k = np.array(N_k, dtype=np.int64)
        if np.ndim(u_kn) == 3:
            u_kn = kln_to_kn(u_kn, N_k=self.N_k)
        self.u_kn = np.array(u_kn, dtype=np.float64)
        self.K, self.N = self.u_kn.shape
        if self.N_k.sum() != self.N:
            raise ParameterError("the sum of all N_k must equal the number of samples")
        self.x_kindices = (np.repeat(np.arange(self.K, dtype=np.int64), self.N_k) if x_kindices is None
                           else np.asarray(x_kindices))
        self.rng = np.random.default_rng(np.random.randint(np.iinfo(np.int32).max) if rseed is None else rseed)
        probe = self.rng.choice(np.arange(self.N), min(50, self.N))
        self.samestates = []
        for k in range(self.K):
            for l in range(k):
                d = self.u_kn[k, probe] - self.u_kn[l, probe]
                if d @ d < relative_tolerance:
                    self.samestates += [[k, l], [l, k]]
        self.states_with_samples = np.flatnonzero(self.N_k).astype(np.int64)
        if initial_f_k is not None:
            f_k = np.array(initial_f_k, dtype=np.float64)
            if f_k.shape != (self.K,):
                raise ParameterError(f"initial_f_k must be a {self.K}-dimensional array")
            f_k -= f_k[0]
        elif initialize == "zeros":
            f_k = np.zeros(self.K)
        elif initialize == "BAR":
            f_k = self._initialize_with_bar(self.u_kn)
        else:
            raise ParameterError(f"the stand-in implements initialize='zeros' and 'BAR', not {initialize!r}")
        solver_protocol = _complete_protocol(solver_protocol, mbar_solvers.DEFAULT_SOLVER_PROTOCOL,
                                             mbar_solvers.ROBUST_SOLVER_PROTOCOL, maximum_iterations, verbose)
        bootstrap_solver_protocol = _complete_protocol(
            bootstrap_solver_protocol, mbar_solvers.BOOTSTRAP_SOLVER_PROTOCOL, mbar_solvers.ROBUST_SOLVER_PROTOCOL,
            maximum_iterations, verbose)
        self.f_k = mbar_solvers.solve_mbar_for_all_states(self.u_kn, self.N_k, f_k, self.states_with_samples,
                                                          solver_protocol)
        if n_bootstraps > 0:
            self.n_bootstraps = n_bootstraps
            self.f_k_boots = np.zeros((n_bootstraps, self.K))
            self.bootstrap_rints = np.zeros((n_bootstraps, self.N), dtype=np.int64)
            for b in range(n_bootstraps):
                rints = np.zeros(self.N, dtype=np.int64)
                for k in range(self.K):
                    idx = np.flatnonzero(self.x_kindices == k)
                    rints[idx] = idx[self.rng.integers(int(self.N_k[k]), size=int(self.N_k[k]))]
                self.f_k_boots[b] = mbar_solvers.solve_mbar_for_all_states(
                    self.u_kn[:, rints], self.N_k, self.f_k.copy(), self.states_with_samples,
                    bootstrap_solver_protocol)
                self.bootstrap_rints[b] = rints
        self.Log_W_nk = mbar_solvers.mbar_log_W_nk(self.u_kn, self.N_k, self.f_k)

    def _zerosamestates(self, A):
        for k, l in self.samestates:
            A[k, l] = 0

    def compute_overlap(self):
        W = np.exp(self.Log_W_nk)
        O = self.N_k * (W.T @ W)
        eig = np.sort(np.linalg.eigvals(O))[::-1]
        return {"scalar": 1 - eig[1], "eigenvalues": eig, "matrix": O}

    def compute_free_energy_differences(self, compute_uncertainty=True, uncertainty_method=None,
                                        warning_cutoff=1.0e-10, return_theta=False):
        Delta = np.array(self.f_k - np.vstack(self.f_k))
        self._zerosamestates(Delta)
        out = {"Delta_f": Delta}
        if compute_uncertainty or return_theta:
            if uncertainty_method != "svd":
                raise ParameterError("the stand-in computes uncertainties with uncertainty_method='svd' only")
            # Shirts & Chodera, J. Chem. Phys. 129, 124105 (2008), appendix D, Eq. D4: W = U S V^T,
            # Theta = V S (I - S V^T diag(N) V S)^+ S V^T
            _, S, Vt = np.linalg.svd(np.exp(self.Log_W_nk), full_matrices=False)
            V, Sg = Vt.T, np.diag(S)
            inner = np.identity(self.K) - Sg @ V.T @ np.diag(self.N_k) @ V @ Sg
            Theta = V @ Sg @ np.linalg.pinv(inner, rcond=1e-10) @ Sg @ V.T
            if compute_uncertainty:
                d = np.diag(Theta)
                var = d[:, None] + d[None, :] - 2 * Theta
                d2 = np.sqrt(np.maximum(var, 0.0))
                self._zerosamestates(d2)
                out["dDelta_f"] = d2
            if return_theta:
                out["Theta"] = Theta
        return out

    def compute_expectations(self, A_n, output="averages", compute_uncertainty=True, uncertainty_method=None,
                             warning_cutoff=1.0e-10, state_dependent=False):
        A_n = np.asarray(A_n, dtype=np.float64)
        state_map = np.zeros((2, self.K), dtype=np.int64)
        state_map[0] = np.arange(self.K)
        state_map[1] = np.arange(self.K) if state_dependent else 0
        inner = self.compute_expectations_inner(A_n, self.u_kn, state_map, uncertainty_method=uncertainty_method,
                                                warning_cutoff=warning_cutoff, return_theta=compute_uncertainty)
        A = inner["observables"]
        out = {"mu": A if output == "averages" else A - np.vstack(A)}
        if compute_uncertainty:
            scale = np.concatenate([A - inner["Amin"]] * 2)
            Theta = scale[:, None] * inner["Theta"] * scale[None, :]
            K = self.K
            cov = Theta[:K, :K] + Theta[K:, K:] - Theta[:K, K:] - Theta[K:, :K]
            if output == "averages":
                out["sigma"] = np.sqrt(np.diag(cov))
            else:
                d = np.diag(cov)
                out["sigma"] = np.sqrt(np.maximum(d[:, None] + d[None, :] - 2 * cov, 0.0))
        return out

    def compute_perturbed_free_energies(self, u_ln, compute_uncertainty=True, uncertainty_method=None,
                                        warning_cutoff=1.0e-10):
        u_ln = np.atleast_2d(np.asarray(u_ln, dtype=np.float64))
        L = u_ln.shape[0]
        inner = self.compute_expectations_inner(np.array([0.0]), u_ln, np.arange(L),
                                                uncertainty_method=uncertainty_method,
                                                warning_cutoff=warning_cutoff, return_theta=compute_uncertainty)
        f = inner["f"]
        out = {"Delta_f": f - np.vstack(f)}
        if compute_uncertainty:
            d = np.diag(inner["Theta"])
            out["dDelta_f"] = np.sqrt(np.maximum(d[:, None] + d[None, :] - 2 * inner["Theta"], 0.0))
        return out
