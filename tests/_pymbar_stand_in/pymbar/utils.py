"""pymbar.utils names the stand-in needs (see the package docstring)."""
import numpy as np


class ParameterError(Exception):
    pass


def kln_to_kn(kln, N_k=None, cleanup=False):
    """[K, L, N_max] energies of the samples drawn from state k -> [L, N] in block order."""
    K, L, N_max = np.shape(kln)
    N_k = np.full(K, N_max, dtype=np.int64) if N_k is None else np.asarray(N_k, dtype=np.int64)
    return np.concatenate([np.asarray(kln)[k, :, :N_k[k]] for k in range(K)], axis=1)


def kn_to_n(kn, N_k=None, cleanup=False):
    """[K, N_max] values of the samples drawn from state k -> [N] in block order."""
    K, N_max = np.shape(kn)
    N_k = np.full(K, N_max, dtype=np.int64) if N_k is None else np.asarray(N_k, dtype=np.int64)
    return np.concatenate([np.asarray(kn)[k, :N_k[k]] for k in range(K)])
