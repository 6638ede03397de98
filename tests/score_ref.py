"""Float64 numpy restatement of the score-test parts of DESIGN §2.3 (the reference the kernel is tested against)."""
import numpy as np

import wald_ref


def parts(Z_loc, Z_std_log, sigma_log, prior_mean, Xt, X, cell_mode=False):
    """(U (Ng, J), A (Ng, J), B (Ng, J, K~), Ut (Ng, K~)) of candidates X (Nc, J) against design rows Xt (Nc, K~):
    r = (Z_loc - prior mean) / sigma^2, w the Louis weight of wald_ref.weights."""
    tau = np.asarray(sigma_log, np.float64).reshape(-1)
    tau = tau[:, None] if cell_mode else tau[None, :]
    r = (np.asarray(Z_loc, np.float64) - np.asarray(prior_mean, np.float64)) * np.exp(-2.0 * tau)
    w = wald_ref.weights(Z_std_log, sigma_log, cell_mode)
    X = np.asarray(X, np.float64)
    Xt = np.asarray(Xt, np.float64)
    return (r.T @ X, w.T @ (X * X), np.einsum('cg,cj,ck->gjk', w, X, Xt), r.T @ Xt)


def prior_mean(eng, m):
    """Float64 prior mean intercept + Xc Wc + Wg Xg^T of FitEngine model m, (Nc, Ng)."""
    Ng = eng.Ng
    f = lambda t: t.double().cpu().numpy()
    pm = f(eng.Xc[m]) @ f(eng.Wc[m, :, :Ng]) + f(eng.Wg[m]) @ f(eng.Xg[:Ng]).T
    b = f(eng.intercept[m])
    return pm + (b[:, None] if eng.cell_mode else b[None, :Ng])


def engine_reference(eng, m, X):
    """parts() on FitEngine model m's own state."""
    has_b = not eng.cell_mode and eng.intercept_const is None
    w = len(eng.masks[m])
    Xt = wald_ref.design_rows(eng.Xc[m, :, :w].cpu().numpy(), has_b)
    n = eng.Nc if eng.cell_mode else eng.Ng
    return parts(eng.Z_loc[m, :, :eng.Ng].cpu().numpy(), eng.Z_std_log[m, :, :eng.Ng].cpu().numpy(),
                 eng.sigma_log[m, :n].cpu().numpy(), prior_mean(eng, m), Xt, X, eng.cell_mode)
