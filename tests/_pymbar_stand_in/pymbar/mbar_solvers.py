"""pymbar.mbar_solvers for the stand-in: pymbar 4's protocol constants; the entry points exist only to be rebound by
pymbar_b200.install() (see the package docstring)."""

DEFAULT_SOLVER_PROTOCOL = (
    dict(method="hybr", continuation=True),
    dict(method="adaptive", options=dict(min_sc_iter=0)),
)
ROBUST_SOLVER_PROTOCOL = (
    dict(method="adaptive", options=dict(maxiter=1000)),
    dict(method="L-BFGS-B", options=dict(maxiter=1000)),
)
BOOTSTRAP_SOLVER_PROTOCOL = (dict(method="adaptive", options=dict(min_sc_iter=0)),)


def _not_installed(*args, **kwargs):
    raise NotImplementedError("the pymbar stand-in has no solver of its own: call pymbar_b200.install() first")


self_consistent_update = mbar_gradient = mbar_objective = mbar_objective_and_gradient = _not_installed
mbar_hessian = mbar_log_W_nk = mbar_W_nk = precondition_u_kn = adaptive = _not_installed
solve_mbar_once = solve_mbar = solve_mbar_for_all_states = _not_installed
jax_self_consistent_update = jax_mbar_gradient = jax_mbar_objective = jax_mbar_objective_and_gradient = _not_installed
jax_mbar_hessian = jax_mbar_log_W_nk = jax_mbar_W_nk = jax_precondition_u_kn = _not_installed
