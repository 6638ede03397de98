"""Float64 numpy restatement of the Wald information of DESIGN §2.2 (the reference the kernel is tested against)."""
import numpy as np


def design_rows(Xc_model, has_b):
    """x~_c: the model's Xc columns in mask order, then a 1 when the intercept is per-event and trained."""
    Xc_model = np.asarray(Xc_model, np.float64)
    if has_b:
        return np.concatenate([Xc_model, np.ones((Xc_model.shape[0], 1))], axis=1)
    return Xc_model


def weights(Z_std_log, sigma_log, cell_mode):
    """w_cg = max(sigma^2 - s_cg^2, 0) / sigma^4 = max(-expm1(2 (lambda - tau)), 0) exp(-2 tau), (Nc, Ng)."""
    lam = np.asarray(Z_std_log, np.float64)
    tau = np.asarray(sigma_log, np.float64).reshape(-1)
    tau = tau[:, None] if cell_mode else tau[None, :]
    return np.maximum(-np.expm1(2.0 * (lam - tau)), 0.0) * np.exp(-2.0 * tau)


def info(Z_std_log, sigma_log, Xt, cell_mode=False):
    """I_g = sum_c w_cg x~_c x~_c^T, (Ng, K~, K~)."""
    w = weights(Z_std_log, sigma_log, cell_mode)
    Xt = np.asarray(Xt, np.float64)
    return np.einsum('cg,ck,cl->gkl', w, Xt, Xt)


def naive_info(sigma_log, Xt, n_events, cell_mode=False):
    """The complete-data information sum_c x~_c x~_c^T / sigma^2 alone, without the missing-information term."""
    tau = np.asarray(sigma_log, np.float64).reshape(-1)
    Xt = np.asarray(Xt, np.float64)
    if cell_mode:
        return np.broadcast_to(np.einsum('c,ck,cl->kl', np.exp(-2 * tau), Xt, Xt), (n_events,) + (Xt.shape[1],) * 2)
    return np.exp(-2 * tau)[:n_events, None, None] * (Xt.T @ Xt)[None]


def engine_reference(eng, m):
    """info() on FitEngine model m's own state (Z_std_log, sigma_log, design)."""
    has_b = not eng.cell_mode and eng.intercept_const is None
    w = len(eng.masks[m])
    Xt = design_rows(eng.Xc[m, :, :w].cpu().numpy(), has_b)
    n = eng.Nc if eng.cell_mode else eng.Ng
    return info(eng.Z_std_log[m, :, :eng.Ng].cpu().numpy(), eng.sigma_log[m, :n].cpu().numpy(), Xt, eng.cell_mode)
