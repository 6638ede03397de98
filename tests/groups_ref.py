"""Float64 numpy restatement of the cross terms of the joint score test of DESIGN §2.4 (the reference the kernel is
tested against)."""
import numpy as np

import wald_ref


def cross(Z_std_log, sigma_log, X, pairs, cell_mode=False):
    """A_gp = sum_c w_cg x_cj x_cj' for pair p = (j, j') of `pairs` (n_pairs, 2), (Ng, n_pairs); w the Louis weight
    of wald_ref.weights."""
    w = wald_ref.weights(Z_std_log, sigma_log, cell_mode)
    X = np.asarray(X, np.float64)
    pairs = np.asarray(pairs).reshape(-1, 2)
    return w.T @ (X[:, pairs[:, 0]] * X[:, pairs[:, 1]])


def engine_cross(eng, m, X, pairs):
    """cross() on FitEngine model m's own state."""
    n = eng.Nc if eng.cell_mode else eng.Ng
    return cross(eng.Z_std_log[m, :, :eng.Ng].cpu().numpy(), eng.sigma_log[m, :n].cpu().numpy(), X, pairs,
                 eng.cell_mode)
