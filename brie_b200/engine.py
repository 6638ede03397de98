"""Batched BRIE2 fit engine: the thin Python layer over the C ABI.

One `FitEngine` holds the device state of M models (the base/full model and the
LRT refits of brie/models/model_wrap.py:155-187) over one event shard on one GPU
and drives the reference's optimisation schedule (brie/models/model_TFProb.py:
214-273) with every (model, reference-batch) pair converging independently, as
the reference's sequential per-batch fits do (model_wrap.py:241-260).

torch is used for device memory, streams and (optionally) torch.distributed --
all arithmetic on the path happens in libbrie_b200.so.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib

LEARNING_RATES = [0.001, 0.005, 0.01, 0.02, 0.01, 0.005]   # model_TFProb.py:234
KC_SUPPORTED = (0, 1, 2, 4, 8, 16)
KG_SUPPORTED = (0, 4, 8)


K_WIDE_MAX = 4096
SCORE_BLOCK_BYTES = 1 << 30     # device scratch + outputs of one block of score candidates (FitEngine.score_parts)


def _pad_to(k, allowed, what):
    """Width of the device arrays for a design of k columns: the next register-resident instantiation, or k itself
    when the design is wide (covariate contractions as GEMMs around the fused kernel, any width)."""
    for a in allowed:
        if k <= a:
            return a
    if k > K_WIDE_MAX:
        raise ValueError("brie_b200: %s = %d exceeds the supported maximum %d" % (what, k, K_WIDE_MAX))
    return k


def _round_up(x, m):
    return (x + m - 1) // m * m


def encode_counts(lib, counts, device):
    """Packed count codes of padded (Nc, ld) float32 tiles (brie_encode_counts): (codes (Nc, ld) int32, dict (3, 256)
    float32), or None when a layer has more than 255 distinct non-zero values (or a value that is negative or NaN).
    Synchronises once, to read the number of values per layer."""
    Nc, ld = counts[0].shape
    codes = torch.empty((Nc, ld), dtype=torch.int32, device=device)
    dct = torch.empty((3, 256), dtype=torch.float32, device=device)
    n_values = torch.empty(3, dtype=torch.int32, device=device)
    scratch = torch.empty(int(lib.brie_encode_counts_scratch_bytes()), dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    with torch.cuda.device(device):
        _lib.check(lib.brie_encode_counts(Nc, ld, counts[0].data_ptr(), counts[1].data_ptr(),
                                          counts[2].data_ptr() if len(counts) > 2 else None, codes.data_ptr(),
                                          dct.data_ptr(), n_values.data_ptr(), scratch.data_ptr(), st))
    if int(n_values.max()) > 255:
        return None
    return codes, dct


def gathered_round_is_cheaper(cols, n_events, n_cells, n_layers, n_steps, count_bytes=None):
    """Extension round on gathered sub-fits or in place?  cols[m]: local event indices still active in model m.

    Bytes per cell and step.  In place, every 8-event block (one 32-byte sector of each 4-byte array) that
    holds an active event moves whole: 48 B of state per model, and the counts once for the models
    co-resident on the tile.  Gathered, only active events move, but each model reads its own copy of the
    counts; add the gather and scatter passes (about 3 step-equivalents) and ~15 ms of set-up per round,
    expressed in the same unit.  Gathered must win by 10 % to be chosen.  count_bytes: bytes of counts per
    element the step kernel reads, 4 * n_layers for float32 tiles (default), 4 for packed codes."""
    cb = 4 * n_layers if count_bytes is None else count_bytes
    M = len(cols)
    n_act = sum(len(c) for c in cols)
    ev = np.zeros((M, _round_up(max(n_events, 1), 8)), bool)
    for m in range(M):
        ev[m, cols[m]] = True
    blk = ev.reshape(M, -1, 8).any(axis=2)
    in_place = 8.0 * (48 * blk.sum() + cb * blk.any(axis=0).sum())
    gathered = n_act * (48 + cb) * (1.0 + 3.0 / max(n_steps, 1)) + 1e11 / max(n_cells * n_steps, 1)
    return gathered <= 0.9 * in_place


def pair_index(kt):
    """(rows, cols) of the packed pairs k <= l of a kt x kt symmetric matrix, row-major over the upper triangle
    (the order of brie_fit_wald_info's output)."""
    return np.triu_indices(kt)


def unpack_pairs(packed, kt):
    """(..., kt (kt + 1) / 2) packed upper triangles -> (..., kt, kt) symmetric matrices."""
    packed = np.asarray(packed)
    k, l = pair_index(kt)
    out = np.zeros(packed.shape[:-1] + (kt, kt), packed.dtype)
    out[..., k, l] = packed
    out[..., l, k] = packed
    return out


WALD_RCOND = 1e-12


def _pd_factor(info):
    """The positive-definiteness checks of wald_from_info on a batch of informations (Ng, K, K), and the Cholesky
    factor of the accepted ones after rescaling to a unit diagonal: (ok (Ng,) bool, d (Ng, K) = sqrt(diag(info)),
    idx = flatnonzero(ok), L (len(idx), K, K) with L L^T = info[idx] / d d^T)."""
    Ng, K = info.shape[:2]
    with np.errstate(invalid='ignore'):
        d = np.sqrt(np.diagonal(info, axis1=1, axis2=2))         # rescale to a unit diagonal first
    ok = np.all(np.isfinite(info), axis=(1, 2)) & np.all(d > 0, axis=1)
    dd = np.where(ok[:, None], d, 1.0)
    with np.errstate(invalid='ignore'):
        R = np.where(ok[:, None, None], info / dd[:, :, None] / dd[:, None, :], np.eye(K))
    ev = np.linalg.eigvalsh(R)
    ok &= ev[:, 0] > WALD_RCOND * ev[:, -1]
    idx = np.flatnonzero(ok)
    L = np.linalg.cholesky(R[idx]) if idx.size else np.zeros((0, K, K))   # batched; PD after the checks above
    return ok, d, idx, L


def wald_from_info(coef, info):
    """Wald standard errors and p-values of per-event coefficients `coef` (Ng, K) from their observed information
    `info` (Ng, K, K): se = sqrt(diag(info^-1)), pval = chi2.sf((coef / se)^2, 1).  An event whose information is
    not positive definite -- Cholesky fails, or the reciprocal condition number of the unit-diagonal rescaling is
    below WALD_RCOND (e.g. too few cells with reads) -- gets se NaN and pval 1.0, so BH still works.
    Returns (se, pval), both (Ng, K) float64."""
    from scipy.stats import chi2
    coef = np.asarray(coef, np.float64)
    info = np.asarray(info, np.float64)
    Ng, K = coef.shape
    se = np.full((Ng, K), np.nan)
    if K > 0 and Ng > 0:
        _, d, idx, L = _pd_factor(info)
        if idx.size:
            Linv = np.linalg.solve(L, np.broadcast_to(np.eye(K), L.shape))
            diag_inv = (Linv ** 2).sum(axis=1)                        # diag(R^-1) = column sums of Linv^2
            se[idx] = np.sqrt(diag_inv) / d[idx]
    with np.errstate(invalid='ignore', divide='ignore'):
        pval = chi2.sf((coef / se) ** 2, df=1)
    pval[~np.isfinite(se)] = 1.0
    return se, pval


SCORE_VTOL = 1e-10


def score_from_parts(parts, info):
    """Score tests of candidates from their parts (FitEngine.score_parts: U, A (Ng, J), B (Ng, J, K~), Ut (Ng, K~))
    and the null model's information `info` (Ng, K~, K~) (DESIGN §2.3):
        V = A - B I^-1 B^T   (efficient information),   Ue = U - B I^-1 Ut   (efficient score),
        score_z = Ue / sqrt(V),   pval = chi2.sf(score_z^2, 1),   effect = Ue / V   (one-step estimate, logit scale).
    An event whose information fails wald_from_info's checks, and a candidate with A <= 0 or V <= SCORE_VTOL * A
    (collinear with the fitted columns, or zero on every cell), get score_z and effect NaN and pval 1.0.
    Returns (score_z, effect, pval), each (Ng, J) float64."""
    from scipy.stats import chi2
    U, A, B, Ut = (np.asarray(x, np.float64) for x in parts)
    info = np.asarray(info, np.float64)
    Ng, J = U.shape
    K = info.shape[1] if info.ndim == 3 else 0
    V, Ue = A.copy(), U.copy()
    ok = np.ones(Ng, bool)
    if K > 0 and Ng > 0:
        ok, d, idx, L = _pd_factor(info)
        if idx.size:                                                  # B I^-1 B^T = (L^-1 Bs^T)^T (L^-1 Bs^T), Bs = B / d
            dd = d[idx]
            Y = np.linalg.solve(L, np.swapaxes(B[idx] / dd[:, None, :], 1, 2))      # (n, K, J)
            y = np.linalg.solve(L, (Ut[idx] / dd)[:, :, None])                     # (n, K, 1)
            V[idx] -= (Y ** 2).sum(axis=1)
            Ue[idx] -= (Y * y).sum(axis=1)
    good = ok[:, None] & (A > 0) & (V > SCORE_VTOL * A)
    z, eff = np.full((Ng, J), np.nan), np.full((Ng, J), np.nan)
    with np.errstate(invalid='ignore', divide='ignore'):
        z[good] = Ue[good] / np.sqrt(V[good])
        eff[good] = Ue[good] / V[good]
    pval = np.ones((Ng, J))
    pval[good] = chi2.sf(z[good] ** 2, df=1)
    return z, eff, pval


def _quad_form(M, v, tol):
    """v^T M^-1 v per event for a batch of symmetric k x k matrices M (n, k, k) and vectors v (n, k), or NaN where M
    is not positive definite after rescaling to a unit diagonal with reciprocal condition number above `tol`."""
    n, k = v.shape
    out = np.full(n, np.nan)
    with np.errstate(invalid='ignore'):
        d = np.sqrt(np.diagonal(M, axis1=1, axis2=2))
    ok = np.all(np.isfinite(M), axis=(1, 2)) & np.all(d > 0, axis=1) & np.all(np.isfinite(v), axis=1)
    idx = np.flatnonzero(ok)
    if idx.size:
        dd = d[idx]
        R = M[idx] / dd[:, :, None] / dd[:, None, :]
        ev = np.linalg.eigvalsh(R)
        good = ev[:, 0] > tol * ev[:, -1]
        idx, R, dd = idx[good], R[good], dd[good]
        if idx.size:
            y = np.linalg.solve(np.linalg.cholesky(R), (v[idx] / dd)[:, :, None])[:, :, 0]
            out[idx] = (y ** 2).sum(axis=1)
    return out


def wald_groups_from_info(coef, info, groups):
    """Joint Wald tests that all coefficients of a group are 0 (DESIGN §2.4): per event and group G of columns of
    `coef` (Ng, K), stat = beta_G^T ((I^-1)_GG)^-1 beta_G with `info` (Ng, K, K), df = |G|.  An event whose
    information fails wald_from_info's checks gets stat NaN and pval 1.  Returns (stat, pval), each (Ng, H) float64."""
    from scipy.stats import chi2
    coef = np.asarray(coef, np.float64)
    info = np.asarray(info, np.float64)
    Ng, K = coef.shape
    stat, pval = np.full((Ng, len(groups)), np.nan), np.ones((Ng, len(groups)))
    if Ng == 0 or K == 0:
        return stat, pval
    _, d, idx, L = _pd_factor(info)
    if idx.size:
        Linv = np.linalg.solve(L, np.broadcast_to(np.eye(K), L.shape))   # R^-1 = Linv^T Linv, R = info / d d^T
        for h, G in enumerate(groups):
            G = list(G)
            S = np.einsum('nki,nkj->nij', Linv[:, :, G], Linv[:, :, G])   # (R^-1)_GG
            stat[idx, h] = _quad_form(S, coef[idx][:, G] * d[idx][:, G], 0.0)
    for h, G in enumerate(groups):
        ok = np.isfinite(stat[:, h])
        pval[ok, h] = chi2.sf(stat[ok, h], df=len(G))
    return stat, pval


def group_pairs(groups):
    """(n_pairs, 2) int32 table of the distinct off-diagonal candidate pairs (j < j') of the groups, sorted: the pairs
    whose cross terms FitEngine.score_cross computes."""
    pairs = sorted({(min(a, b), max(a, b)) for G in groups for i, a in enumerate(G) for b in G[i + 1:]})
    return np.array(pairs, np.int32).reshape(-1, 2)


def score_groups_from_parts(parts, cross, pairs, info, groups):
    """Joint score tests of groups of candidates (DESIGN §2.4) from their parts (FitEngine.score_parts: U, A, B, Ut),
    the cross terms `cross` (Ng, n_pairs) of the pairs `pairs` (FitEngine.score_cross, group_pairs) and the null
    model's information `info`: per group G of k candidates
        V_GG = A_GG - B_G I^-1 B_G^T,   Ue_G = U_G - B_G I^-1 Ut,   stat = Ue_G^T V_GG^-1 Ue_G,   df = k.
    An event whose information fails wald_from_info's checks, a member that fails score_from_parts' rule (A <= 0 or
    V <= SCORE_VTOL * A: collinear with the fitted columns, or zero on every cell), and a V_GG whose unit-diagonal
    rescaling has reciprocal condition number <= SCORE_VTOL (members collinear with each other) give stat NaN and
    pval 1.  Returns (stat, pval), each (Ng, H) float64."""
    from scipy.stats import chi2
    U, A, B, Ut = (np.asarray(x, np.float64) for x in parts)
    cross = np.asarray(cross, np.float64)
    info = np.asarray(info, np.float64)
    Ng = U.shape[0]
    K = info.shape[1] if info.ndim == 3 else 0
    col = {(int(a), int(b)): p for p, (a, b) in enumerate(np.asarray(pairs).reshape(-1, 2))}
    ok = np.ones(Ng, bool)
    Y = y = None
    if K > 0 and Ng > 0:
        ok, d, idx, L = _pd_factor(info)
        dfull = np.where(ok[:, None], d, 1.0)
        Lfull = np.broadcast_to(np.eye(K), (Ng, K, K)).copy()
        Lfull[idx] = L
        Y = np.linalg.solve(Lfull, np.swapaxes(B / dfull[:, None, :], 1, 2))    # (Ng, K, J): L^-1 (B / d)^T
        y = np.linalg.solve(Lfull, (Ut / dfull)[:, :, None])[:, :, 0]           # (Ng, K)
    stat, pval = np.full((Ng, len(groups)), np.nan), np.ones((Ng, len(groups)))
    for h, G in enumerate(groups):
        G = [int(j) for j in G]
        k = len(G)
        V = np.empty((Ng, k, k))
        for a, ja in enumerate(G):
            V[:, a, a] = A[:, ja]
            for b in range(a + 1, k):
                V[:, a, b] = V[:, b, a] = cross[:, col[(min(ja, G[b]), max(ja, G[b]))]]
        Ue = U[:, G].copy()
        if Y is not None:
            V -= np.einsum('nki,nkj->nij', Y[:, :, G], Y[:, :, G])
            Ue -= np.einsum('nki,nk->ni', Y[:, :, G], y)
        Ad, Vd = A[:, G], np.diagonal(V, axis1=1, axis2=2)
        good = ok & np.all((Ad > 0) & (Vd > SCORE_VTOL * Ad), axis=1)
        s = np.full(Ng, np.nan)
        s[good] = _quad_form(V[good], Ue[good], SCORE_VTOL)
        stat[:, h] = s
        fin = np.isfinite(s)
        pval[fin, h] = chi2.sf(s[fin], df=k)
    return stat, pval


class FitEngine:
    """Device-resident batched fit.

    Parameters
    ----------
    counts : list of 2 or 3 (Nc, Ng) float32 arrays (numpy or torch, host or device),
        pseudo-count already applied.
    effLen : (Ng, 6) array or None -- columns 0, 4, 5 are used (model_TFProb.py:176).
    Xc : (Nc, Kc) cell covariates (all columns any batched model uses).
    Xg : (Ng, Kg) gene features.
    masks : list (one per model) of the Xc column indices that model uses, in the order of
        that model's own design matrix (np.delete / np.append of model_wrap.py:161, 167).
        The device gets one compact (Nc, K) design matrix per model, K = the widest model --
        a 15-covariate one-vs-rest LRT with --testBase null is 15 models of width <= 2.
    model_ids : RNG model word per model (default 0..M-1).
    intercept, sigma : None (trainable) or constants (model_TFProb.py:67-78).
    group_size : events per reference batch, ceil(batch_size / Nc) (model_wrap.py:242);
        None = one group (un-batched branch, model_wrap.py:261-269).
    event_offset : global index of this shard's first event.
    target : "ELBO" (default) or "marginLik" (model_TFProb.py:156-157, 188-189, 202-205).
    dist_group : torch.distributed process group for event-sharded fits with shared
        per-cell parameters (Kg > 0 or intercept_mode 'cell'); None = single GPU.
    count_format : None (default) lets the fused step kernel read the counts as packed 8-bit
        dictionary codes (4 B per element instead of 4 B per layer, bit-identical results) whenever
        every layer has at most 255 distinct non-zero values; 'f32' keeps it on the float32 tiles.
        The chosen form is `self.count_format` ('code8' or 'f32').
    count_codes : `count_codes` of another engine over the same count tiles, reused instead of
        encoding them again (the engines of one fit_BRIE_matrix chunk share one code tile).
    """

    def __init__(self, counts, effLen=None, Xc=None, Xg=None, masks=None, model_ids=None,
                 intercept=None, intercept_mode='gene', sigma=None, MC_size=1, seed=0,
                 group_size=None, event_offset=0, n_events_total=None, device=None,
                 trace_cap=None, dist_group=None, n_events=None, target="ELBO", count_format=None,
                 count_codes=None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("brie_b200: no CUDA device (there is no CPU fallback)")
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        Nc, Ng = counts[0].shape
        if n_events is not None:          # device tensors already padded to (Nc, ld), e.g. from the simulator
            Ng = int(n_events)
        self.Nc, self.Ng = int(Nc), int(Ng)
        self.ld = _lib.leading_dim(self.Ng)
        self.event_offset = int(event_offset)
        self.n_events_total = int(n_events_total) if n_events_total is not None else self.event_offset + self.Ng
        self.n_layers = len(counts)
        self.cell_mode = intercept_mode.upper() == 'CELL'
        self.intercept_const, self.sigma_const = intercept, sigma
        self.S = int(MC_size)
        self.seed = int(seed)
        self.dist_group = dist_group
        if target not in _lib.TARGETS:
            raise ValueError("brie_b200: target must be 'ELBO' or 'marginLik', got %r" % (target,))
        self.target = target
        Xc = np.zeros((Nc, 0), np.float32) if Xc is None else np.asarray(Xc, np.float32)
        Xg = np.zeros((Ng, 0), np.float32) if Xg is None else np.asarray(Xg, np.float32)
        self.Kc_real, self.Kg_real = Xc.shape[1], Xg.shape[1]
        if masks is None:
            masks = [list(range(self.Kc_real))]
        self.masks = [[int(k) for k in mk] for mk in masks]   # ordered: compact Wc row kk <-> column masks[m][kk]
        self.M = len(self.masks)
        self.Kc = _pad_to(max(len(mk) for mk in self.masks), KC_SUPPORTED, "Kc (widest batched model)")
        self.Kg = _pad_to(self.Kg_real, KG_SUPPORTED, "Kg")
        # wide design: one of the widths is beyond the register-resident instantiations; then BOTH contractions run
        # as GEMMs and neither width is padded
        self.wide = self.Kc > KC_SUPPORTED[-1] or self.Kg > KG_SUPPORTED[-1]
        if self.wide:
            self.Kc, self.Kg = max(len(mk) for mk in self.masks), self.Kg_real
            if target != "ELBO":
                raise ValueError("brie_b200: target 'marginLik' supports at most %d cell covariates and %d gene features"
                                 % (KC_SUPPORTED[-1], KG_SUPPORTED[-1]))
        self.model_ids = list(range(self.M)) if model_ids is None else [int(i) for i in model_ids]
        self.shared = self.cell_mode or self.Kg_real > 0       # parameters shared across events
        if group_size is None or self.shared:
            group_size = max(self.n_events_total, 1)
        self.group_size = int(group_size)
        self.first_group = self.event_offset // self.group_size
        last_group = (self.event_offset + self.Ng - 1) // self.group_size
        self.n_groups = last_group - self.first_group + 1
        self.trace_cap = int(trace_cap) if trace_cap is not None else 1024

        dev, f32 = self.device, torch.float32
        ld = self.ld

        def padded(x):
            if (torch.is_tensor(x) and x.device == dev and x.dtype == f32 and tuple(x.shape) == (self.Nc, ld)
                    and x.is_contiguous()):
                return x                  # zero-copy: caller guarantees zero counts in the padding
            t = torch.zeros((self.Nc, ld), dtype=f32, device=dev)
            src = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
            t[:, :self.Ng].copy_(src, non_blocking=True)
            return t

        self.counts = [padded(c) for c in counts]
        # read counts are non-negative; the step kernel relies on it (an element whose counts sum to zero has
        # zeros in every layer, brie_kernels.cuh phase B)
        if float(torch.stack([c.min() for c in self.counts]).min()) < 0:      # one device sync for all layers
            raise ValueError("brie_b200: count layers must be non-negative")
        if count_format not in (None, 'f32'):
            raise ValueError("brie_b200: count_format must be None or 'f32', got %r" % (count_format,))
        # Only the ELBO step kernel reads codes (marginLik streams the float32 tiles itself).
        if count_format is None and target == "ELBO":
            self.count_codes = count_codes if count_codes is not None else encode_counts(self.lib, self.counts, dev)
        else:
            self.count_codes = None
        self.count_format = 'f32' if self.count_codes is None else 'code8'
        self.h2d_bytes = sum(int(np.prod(c.shape)) * 4 for c in counts)
        if effLen is not None:
            eff = np.ones((3, ld), np.float32)
            eff[:, :self.Ng] = np.asarray(effLen, np.float32)[:, [0, 4, 5]].T
            self.eff = torch.from_numpy(eff).to(dev)
        else:
            self.eff = None
        xc = np.zeros((self.M, self.Nc, max(self.Kc, 1)), np.float32)
        for m, mk in enumerate(self.masks):
            xc[m, :, :len(mk)] = Xc[:, mk]
        xg = np.zeros((self.Ng, max(self.Kg, 1)), np.float32)
        xg[:, :self.Kg_real] = Xg
        self.Xc_host, self.Xg_host = Xc, Xg
        self.Xc = torch.from_numpy(xc).to(dev)
        self.Xg = torch.from_numpy(xg[:, :max(self.Kg, 1)]).contiguous().to(dev)

        M = self.M
        # init_params fills Z_loc / Z_std_log completely and begin_stage clears the Adam moments
        self.Z_loc = torch.empty((M, self.Nc, ld), dtype=f32, device=dev)
        self.Z_std_log = torch.empty((M, self.Nc, ld), dtype=f32, device=dev)
        self.adam_Z = torch.empty((4, M, self.Nc, ld), dtype=f32, device=dev)
        self.Wc = torch.zeros((M, max(self.Kc, 1), ld), dtype=f32, device=dev)
        nsmall = self.Nc if self.cell_mode else ld
        self.intercept = torch.zeros((M, nsmall), dtype=f32, device=dev)
        self.sigma_log = torch.zeros((M, nsmall), dtype=f32, device=dev)
        self.Wg = torch.zeros((M, self.Nc, max(self.Kg, 1)), dtype=f32, device=dev)
        self.active = torch.zeros((M, ld), dtype=torch.uint8, device=dev)
        self.active[:, :self.Ng] = 1
        self.loss_trace = torch.zeros((M, self.trace_cap, ld), dtype=f32, device=dev)

        d = _lib.FitDesc()
        d.n_cells, d.n_events, d.ld, d.event_offset = self.Nc, self.Ng, ld, self.event_offset
        d.seed = self.seed
        d.n_models, d.Kc, d.Kg, d.mc_size = M, self.Kc, self.Kg, self.S
        d.n_layers, d.has_efflen, d.cell_mode = self.n_layers, int(effLen is not None), int(self.cell_mode)
        d.train_intercept, d.train_sigma = int(intercept is None), int(sigma is None)
        d.trace_cap = self.trace_cap
        d.target = _lib.TARGETS[target]
        for m in range(M):
            d.model_id[m] = self.model_ids[m]
            d.xc_mask[m] = 0 if self.wide else (1 << len(self.masks[m])) - 1
            d.xc_width[m] = len(self.masks[m])
        self.desc = d
        h = C.c_void_p()
        _lib.check(self.lib.brie_fit_create(C.byref(d), C.byref(h)))
        self.h = h
        sz = _lib.FitSizes()
        _lib.check(self.lib.brie_fit_get_sizes(h, C.byref(sz)))
        self.sizes = sz
        self.scratch = torch.zeros(int(sz.scratch_bytes // 4) + 4, dtype=f32, device=dev)
        self.adam_small = torch.zeros(max(int(sz.adam_small_floats), 4), dtype=f32, device=dev)
        b = _lib.FitBuffers()
        for i in range(3):
            b.counts[i] = self.counts[i].data_ptr() if i < self.n_layers else None
        b.efflen3 = self.eff.data_ptr() if self.eff is not None else None
        b.Xc, b.Xg = self.Xc.data_ptr(), self.Xg.data_ptr()
        b.Z_loc, b.Z_std_log, b.adam_Z = self.Z_loc.data_ptr(), self.Z_std_log.data_ptr(), self.adam_Z.data_ptr()
        b.Wc, b.intercept, b.sigma_log = self.Wc.data_ptr(), self.intercept.data_ptr(), self.sigma_log.data_ptr()
        b.Wg, b.adam_small = self.Wg.data_ptr(), self.adam_small.data_ptr()
        b.active, b.loss_trace, b.scratch = self.active.data_ptr(), self.loss_trace.data_ptr(), self.scratch.data_ptr()
        self.bufs = b
        _lib.check(self.lib.brie_fit_bind(h, C.byref(b)))
        if self.count_codes is not None:
            _lib.check(self.lib.brie_fit_set_count_codes(h, self.count_codes[0].data_ptr(), 0,
                                                         self.count_codes[1].data_ptr()))
        # Shared per-cell parameters on an event shard: the library all-reduces their gradients itself,
        # in stream order inside brie_fit_run_steps.
        self._comm = None
        if dist_group is not None and self.shared:
            from . import comm
            self._comm = comm.get(dist_group)
            _lib.check(self.lib.brie_fit_set_comm(h, self._comm.h))
        self.n_iter = None
        self.losses = None
        self.loss_gene = None
        self._lr = 0.0
        self._sub_launches = 0      # launches made by gathered sub-fits on behalf of this engine
        self.gather_rounds = 0      # extension rounds that ran on gathered sub-fits (diagnostic)

    def __del__(self):
        h = getattr(self, "h", None)
        if h is not None and h.value:
            self.lib.brie_fit_destroy(h)
            self.h = None

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def launch_count(self):
        return int(self.lib.brie_fit_launch_count(self.h)) + self._sub_launches

    def kernel_timing(self, capacity):
        _lib.check(self.lib.brie_fit_kernel_timing(self.h, int(capacity)))

    def kernel_time_ms(self):
        """(summed ms, launches) of the fused step kernel since timing was armed."""
        ms, n = C.c_double(), C.c_int32()
        _lib.check(self.lib.brie_fit_kernel_time_ms(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def init_params(self, init_objs=None):
        """Model_init (model_TFProb.py:12-31): counter-based random init on the device,
        or injected per-model init objects with attributes intercept, sigma, Z_loc,
        Z_std (or Z_std_log), Wc_loc (compact rows), Wg_loc -- the reference's
        `init_obj` hook (model_TFProb.py:45, 62-65)."""
        with torch.cuda.device(self.device):
            ic = 0.0 if self.intercept_const is None else float(self.intercept_const)
            sc = 1.0 if self.sigma_const is None else float(self.sigma_const)
            _lib.check(self.lib.brie_fit_init_params(self.h, ic, sc, self._stream()))
            if init_objs is None:
                return
            for m, ob in enumerate(init_objs):
                if ob is None:
                    continue
                f = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(self.device)
                self.Z_loc[m, :, :self.Ng] = f(ob.Z_loc)
                if hasattr(ob, 'Z_std_log'):
                    self.Z_std_log[m, :, :self.Ng] = f(ob.Z_std_log)
                else:
                    self.Z_std_log[m, :, :self.Ng] = f(np.log(np.asarray(ob.Z_std, np.float32)))
                wc = np.asarray(ob.Wc_loc, np.float32).reshape(len(self.masks[m]), self.Ng)
                if len(self.masks[m]):
                    self.Wc[m, :len(self.masks[m]), :self.Ng] = f(wc)
                if self.Kg_real > 0:
                    self.Wg[m, :, :self.Kg_real] = f(np.asarray(ob.Wg_loc).reshape(self.Nc, self.Kg_real))
                    self.Wg[m, :, self.Kg_real:] = 0
                n = self.Nc if self.cell_mode else self.Ng
                self.intercept[m, :n] = f(np.asarray(ob.intercept, np.float32).reshape(-1))
                self.sigma_log[m, :n] = f(np.log(np.asarray(ob.sigma, np.float32).reshape(-1)))

    def begin_stage(self, lr):
        self._lr = float(lr)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_begin_stage(self.h, float(lr), self._stream()))

    def step_counters(self):
        """(Adam step count of the open stage, RNG step word)."""
        t, g = C.c_int64(), C.c_uint32()
        _lib.check(self.lib.brie_fit_get_step(self.h, C.byref(t), C.byref(g)))
        return t.value, g.value

    def run_steps(self, n, trace_slot0=-1):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_run_steps(self.h, int(n), int(trace_slot0), self._stream()))

    def group_trace(self, n_slots):
        """(M, n_groups, n_slots) float64 sums of the per-event loss trace per reference batch."""
        out = torch.zeros((self.M, self.n_groups, n_slots), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_group_trace(self.h, int(n_slots), self.group_size, self.n_groups,
                                                     out.data_ptr(), self._stream()))
        # A fit handed a process group spans the ranks with ONE convergence group (fit_BRIE_matrix passes
        # dist_group only for the un-batched branch, model_wrap.py:261-269): its stop rule needs the loss
        # summed over every rank's events -- also for the per-event (gene-mode) LRT refits of a cell-mode fit.
        if self.dist_group is not None:
            import torch.distributed as dist
            dist.all_reduce(out, group=self.dist_group)
        return out.cpu().numpy()

    def set_active_groups(self, act):
        """act: (M, n_groups) bool -> per-event active mask.  When some reference batches are
        frozen the step kernel is pointed at the 8-event column blocks that still hold an active
        event (brie_fit_set_active_blocks): an extension round then costs what its active events
        cost, not what the whole shard costs.  Bit-identical to the dense walk.

        A model with no active batch left is also taken out of the step (brie_fit_set_model_mask): its per-cell
        parameters (Wg, a per-cell intercept / sigma_log), which no `active` flag covers, then stay put as its
        per-event state does.  In a sharded fit `act` comes from the all-reduced group trace, so every rank sets the
        same mask."""
        g = (np.arange(self.Ng) + self.event_offset) // self.group_size - self.first_group
        ev = np.zeros((self.M, self.ld), np.uint8)
        ev[:, :self.Ng] = act[:, g]
        self.active.copy_(torch.from_numpy(ev).to(self.device))
        mask = sum(1 << m for m in range(self.M) if act[m].any())
        _lib.check(self.lib.brie_fit_set_model_mask(self.h, mask))
        if self.shared or self.target != "ELBO" or os.environ.get("BRIE_NO_COMPACT"):
            return
        blk = ev.reshape(self.M, self.ld // 8, 8).any(axis=2)
        if blk[:, :(self.Ng + 7) // 8].all():
            self._blk_ids = None
            _lib.check(self.lib.brie_fit_set_active_blocks(self.h, None, 0, None))
            return
        n_blk = blk.sum(axis=1).astype(np.int32)
        stride = max(int(n_blk.max()), 1)
        ids = np.zeros((self.M, stride), np.int32)
        for m in range(self.M):
            ids[m, :n_blk[m]] = np.flatnonzero(blk[m])
        self._blk_ids = torch.from_numpy(ids).to(self.device)       # kept alive while the handle points at it
        _lib.check(self.lib.brie_fit_set_active_blocks(
            self.h, self._blk_ids.data_ptr(), stride, n_blk.ctypes.data_as(C.POINTER(C.c_int32))))

    # ------------------------------------------------------------------ gathered extension rounds
    def _free_bytes(self):
        free, _ = torch.cuda.mem_get_info(self.device)
        return free + torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)

    def run_steps_gathered(self, act, n_steps, force=False):
        """One convergence-extension round (model_TFProb.py:250-258) of `n_steps` traced steps on the
        events of the still-active reference batches only, act: (M, n_groups) bool.

        The active columns of every model are gathered into dense per-model tiles (state, Adam
        moments, counts, lengths), stepped as a sub-fit that keeps this engine's rows per CTA, RNG
        counters (global event ids) and Adam step count, and scattered back together with their
        loss trace -- so the round moves only bytes of active events, whatever the batch size
        (a --batchSize 500000 batch is 5 events at 100k cells, 1 event at 1M cells: finer than the
        32-byte sector the in-place block list can skip), and stays bit-identical to stepping the
        whole shard with frozen events masked.  Sub-fits are cut to the free device memory and run
        one after the other (events are independent).  Returns False, having done nothing, when the
        fit has shared per-cell parameters, memory is short, or stepping in place over the 8-event
        blocks that hold an active event (set_active_groups) moves no more bytes -- large batches,
        e.g. 100 events at 5k cells, where the per-model count tiles of the gathered form (12 B per
        model instead of 12 B shared) outweigh the few half-empty blocks: the caller then steps in
        place.  `force` skips that cost comparison (tests)."""
        if self.shared or self.wide or self.target != "ELBO":
            return False
        M, Nc, L = self.M, self.Nc, self.n_layers
        g = (np.arange(self.Ng) + self.event_offset) // self.group_size - self.first_group
        cols = [np.flatnonzero(act[m, g]) for m in range(M)]
        n_act = sum(len(c) for c in cols)
        if n_act == 0 or n_act == M * self.Ng:
            return False
        n_cnt = 1 if self.count_codes is not None else L                  # 4-byte count arrays per model column
        if not force and not gathered_round_is_cheaper(cols, self.Ng, Nc, L, n_steps, count_bytes=4 * n_cnt):
            return False
        per_col = M * Nc * (n_cnt + 6) * 4 * 1.05 + M * (n_steps + 64) * 4
        max_ld = int(0.8 * self._free_bytes() / per_col) // 128 * 128
        nmax = max(len(c) for c in cols)
        if max_ld < min(_lib.leading_dim(nmax), 256):
            return False
        n_parts = -(-nmax // max_ld)
        todo = [[np.array_split(c, n_parts)[k] for c in cols] for k in range(n_parts)]
        t0, g0 = self.step_counters()
        done = 0
        with torch.cuda.device(self.device):
            while todo:
                part = todo.pop(0)
                try:
                    sub = _GatheredFit(self, part, n_steps)
                except torch.cuda.OutOfMemoryError:
                    # the estimate was too optimistic (allocator fragmentation): nothing has been touched by this
                    # part yet: if no part has run leave the whole round to the in-place walk, else halve the part
                    sub = None
                    torch.cuda.empty_cache()
                    if done == 0:
                        return False
                    if max(len(c) for c in part) <= 32:
                        raise
                    todo[:0] = [[np.array_split(c, 2)[h] for c in part] for h in range(2)]
                    continue
                sub.run(n_steps, self._lr, t0, g0)
                sub.scatter_back()
                self._sub_launches += sub.launches()
                del sub
                done += 1
            _lib.check(self.lib.brie_fit_resume_stage(self.h, self._lr, t0 + n_steps, g0 + n_steps))
        self.gather_rounds += 1
        return True

    def eval_loss_gene(self, n_eval=500, mc_size=1):
        """Mean of n_eval per-event loss evaluations (model_TFProb.py:261-264); each evaluation
        draws `mc_size` samples -- 1 in the reference, whose loop drops the fit's MC_size."""
        out = torch.zeros((self.M, self.ld), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_eval_loss_gene(self.h, int(n_eval), int(mc_size), out.data_ptr(),
                                                        self._stream()))
        return out[:, :self.Ng]

    def posterior(self, model=0):
        """Psi, Psi95CI, Z_std (model_TFProb.py:88-106) as device tensors (Nc, Ng) views."""
        outs = [torch.empty((self.Nc, self.ld), dtype=torch.float32, device=self.device) for _ in range(3)]
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_posterior(self.h, int(model), outs[0].data_ptr(), outs[1].data_ptr(),
                                                   outs[2].data_ptr(), self._stream()))
        return [o[:, :self.Ng] for o in outs]

    def element_terms(self, model=0, counts=None, mc_size=1, margin=False, loglik=True, kl=False,
                      prior_mean=False, noise_step=None):
        """Dense (Nc, Ng) device tensors of the public model API for one model: the Monte-Carlo log-likelihood of
        every element (BRIE2.logLik_MC, model_TFProb.py:130-191), the KL term of get_loss (:208) and the prior mean
        (Z_prior, :118-127).  `counts`: device tiles (Nc, ld) to evaluate on (default: the fitted ones).  Every call
        draws fresh noise (the reference samples anew on every call) unless `noise_step` pins the counter."""
        if noise_step is None:
            self._terms_calls = getattr(self, "_terms_calls", 0) + 1
            noise_step = (1 << 20) + self._terms_calls          # apart from the loss_gene evaluations' counters
        cs = self.counts if counts is None else counts
        new = lambda want: torch.empty((self.Nc, self.ld), dtype=torch.float32, device=self.device) if want else None
        o_ll, o_kl, o_pm = new(loglik), new(kl), new(prior_mean)
        ptr = lambda t: t.data_ptr() if t is not None else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_element_terms(
                self.h, int(model), cs[0].data_ptr(), cs[1].data_ptr(), cs[2].data_ptr() if len(cs) > 2 else None,
                int(mc_size), int(noise_step), int(bool(margin)), ptr(o_ll), ptr(o_kl), ptr(o_pm), self._stream()))
        cut = lambda t: t[:, :self.Ng] if t is not None else None
        return cut(o_ll), cut(o_kl), cut(o_pm)

    def wald_info(self, m=0):
        """(Ng, K~, K~) float64 observed information of model m's per-event regression parameters from the fitted
        posterior (brie_fit_wald_info): x~ = model m's Xc columns in mask order (its Wc rows), then the intercept
        when it is per-event and trained."""
        nbytes, kt = C.c_size_t(), C.c_int32()
        _lib.check(self.lib.brie_fit_wald_sizes(self.h, int(m), C.byref(nbytes), C.byref(kt)))
        kt = kt.value
        n_pairs = kt * (kt + 1) // 2
        if n_pairs == 0:
            return np.zeros((self.Ng, 0, 0))
        packed = torch.empty((self.Ng, n_pairs), dtype=torch.float64, device=self.device)
        scratch = torch.empty(max(int(nbytes.value), 8), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.brie_fit_wald_info(self.h, int(m), packed.data_ptr(), scratch.data_ptr(),
                                                   self._stream()))
        return unpack_pairs(packed.cpu().numpy(), kt)

    def score_parts(self, m, X):
        """Score-test parts of candidate cell covariates X (Nc, J) against model m as the null model, from its fitted
        posterior (brie_fit_score_parts; DESIGN §2.3): (U, A (Ng, J), B (Ng, J, K~), Ut (Ng, K~)) float64 host arrays,
        x~ as in wald_info.  The candidates go in blocks whose device scratch and outputs stay within
        SCORE_BLOCK_BYTES (the scratch alone is up to 64 row chunks x J (K~ + 2) x ld doubles)."""
        X = self._device_candidates(X)
        J = X.shape[1]
        nbytes, c_kt = C.c_size_t(), C.c_int32()

        def scratch_of(n):
            _lib.check(self.lib.brie_fit_score_sizes(self.h, int(m), int(n), C.byref(nbytes), C.byref(c_kt)))
            return int(nbytes.value)
        s1 = scratch_of(1)
        kt = c_kt.value
        s_cand = scratch_of(2) - s1                                         # the scratch grows linearly in J
        per_cand = s_cand + 8 * self.Ng * (kt + 2)                          # + U, A and B
        fixed = s1 - s_cand + 8 * self.Ng * kt                              # + Ut
        jb = int(max(1, min(J, (SCORE_BLOCK_BYTES - fixed) // per_cand)))
        new = lambda *shape: torch.empty(shape, dtype=torch.float64, device=self.device)
        out_U, out_A, out_B, Ut = np.empty((self.Ng, J)), np.empty((self.Ng, J)), np.empty((self.Ng, J, kt)), None
        ptr = lambda t: t.data_ptr() if t.numel() else None
        for j0 in range(0, J, jb):
            n = min(jb, J - j0)
            U, A, B, T = new(self.Ng, n), new(self.Ng, n), new(self.Ng, n, kt), new(self.Ng, kt)
            scratch = torch.empty(max(scratch_of(n), 8), dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.brie_fit_score_parts(self.h, int(m), X[:, j0:].data_ptr(), int(n), int(J),
                                                         U.data_ptr(), A.data_ptr(), ptr(B), ptr(T),
                                                         scratch.data_ptr(), self._stream()))
            out_U[:, j0:j0 + n], out_A[:, j0:j0 + n] = U.cpu().numpy(), A.cpu().numpy()
            out_B[:, j0:j0 + n] = B.cpu().numpy()
            if Ut is None:
                Ut = T.cpu().numpy()
            del U, A, B, T, scratch
        return out_U, out_A, out_B, Ut

    def _device_candidates(self, X):
        X = torch.as_tensor(np.asarray(X, np.float32) if not torch.is_tensor(X) else X)
        X = X.to(device=self.device, dtype=torch.float32).contiguous()
        if X.dim() != 2 or X.shape[0] != self.Nc or X.shape[1] < 1:
            raise ValueError("brie_b200: score candidates must be (%d, J >= 1), got %s" % (self.Nc, tuple(X.shape)))
        return X

    def score_cross(self, m, X, pairs):
        """Cross terms sum_c w_cg x_cj x_cj' of candidate pairs `pairs` ((n_pairs, 2), j < j' < J) of X (Nc, J)
        against model m's fitted posterior (brie_fit_score_cross; DESIGN §2.4): (Ng, n_pairs) float64 host array.
        X may be the device tensor score_parts read (nothing is uploaded again).  The pairs go in blocks whose device
        scratch and output stay within SCORE_BLOCK_BYTES."""
        X = self._device_candidates(X)
        pairs = np.ascontiguousarray(np.asarray(pairs, np.int32).reshape(-1, 2))
        P = pairs.shape[0]
        out = np.empty((self.Ng, P))
        if P == 0:
            return out
        nbytes = C.c_size_t()

        def scratch_of(n):
            _lib.check(self.lib.brie_fit_score_cross_sizes(self.h, int(m), int(n), C.byref(nbytes)))
            return int(nbytes.value)
        per_pair = scratch_of(2) - scratch_of(1) + 8 * self.Ng           # the scratch grows linearly in n_pairs
        pb = int(max(1, min(P, SCORE_BLOCK_BYTES // per_pair)))
        for p0 in range(0, P, pb):
            n = min(pb, P - p0)
            res = torch.empty((self.Ng, n), dtype=torch.float64, device=self.device)
            scratch = torch.empty(scratch_of(n), dtype=torch.uint8, device=self.device)
            blk = pairs[p0:p0 + n]
            with torch.cuda.device(self.device):
                _lib.check(self.lib.brie_fit_score_cross(self.h, int(m), X.data_ptr(), int(X.shape[1]),
                                                         blk.ctypes.data, int(n), res.data_ptr(), scratch.data_ptr(),
                                                         self._stream()))
            out[:, p0:p0 + n] = res.cpu().numpy()
            del res, scratch
        return out

    # ------------------------------------------------------------------ schedule
    def fit(self, min_iter=1000, max_iter=5000, add_iter=500, epsilon_conv=1e-2, n_eval=500,
            init_objs=None, do_init=True):
        """BRIE2.fit (model_TFProb.py:214-273) for all batched models at once."""
        import os
        import time
        timed = bool(os.environ.get("BRIE_TIMING"))                  # diagnostic phase wall times (syncs the device)
        self.phase_s = {}

        def tick(name, t0):
            if timed:
                torch.cuda.synchronize(self.device)
                self.phase_s[name] = self.phase_s.get(name, 0.0) + time.perf_counter() - t0
            return time.perf_counter()

        t_ph = time.perf_counter()
        n_stage = int(min_iter / 6)
        k_cap = int(os.environ.get("BRIE_KERNEL_TIMING", "0"))      # diagnostic: CUDA events around the first k_cap
        if k_cap > 0:                                                # launches of the fused step kernel of this fit
            self.kernel_timing(k_cap)
        if max(n_stage, add_iter) > self.trace_cap:
            raise ValueError("trace_cap %d too small for %d-step stages" % (self.trace_cap, max(n_stage, add_iter)))
        if do_init:
            self.init_params(init_objs)
        M, NG = self.M, self.n_groups
        for i, lr in enumerate(LEARNING_RATES):                      # :234-241
            self.begin_stage(lr)
            self.run_steps(n_stage, 0 if i == len(LEARNING_RATES) - 1 else -1)
        if n_stage > 0:
            tr = self.group_trace(n_stage).astype(np.float32)        # (M, NG, n_stage)
        else:
            tr = np.zeros((M, NG, 0), np.float32)
        t_ph = tick("fit.schedule", t_ph)
        # Stop rule per (model, reference batch), vectorised over all of them (20 000 batches of one event at
        # 1M cells): only the last d2 losses of a batch enter the rule; the pieces of its trace are kept as
        # views and joined once at the end.
        n_iter = np.full((M, NG), min_iter, np.int64)                # :247
        d1 = int(min(50, add_iter / 2))
        d2 = d1 * 2
        active = np.ones((M, NG), bool)
        tail = tr[:, :, tr.shape[2] - min(d2, tr.shape[2]):]         # (M, NG, <= d2)
        pieces = [(active.copy(), tr)]
        while True:                                                  # :250-258
            a_, b_ = tail[:, :, :max(tail.shape[2] - d1, 0)], tail[:, :, max(tail.shape[2] - d1, 0):]
            if d1 > 0 and a_.shape[2] > 0 and b_.shape[2] > 0:
                with np.errstate(invalid='ignore'):
                    cond = a_.mean(axis=2, dtype=np.float32) - b_.mean(axis=2, dtype=np.float32) > epsilon_conv
            else:                                                    # an empty window compares False, as NaN does in the reference
                cond = np.zeros((M, NG), bool)
            active &= cond & (n_iter < max_iter)
            if not active.any():
                break
            if not self.run_steps_gathered(active, add_iter):
                self.set_active_groups(active)
                self.run_steps(add_iter, 0)
            tr = self.group_trace(add_iter).astype(np.float32)
            pieces.append((active.copy(), tr))
            new_tail = np.concatenate([tail, tr], axis=2)[:, :, -d2:] if d2 > 0 else tail
            tail = np.where(active[:, :, None], new_tail, tail if tail.shape[2] == new_tail.shape[2] else new_tail)
            n_iter[active] += add_iter
        self.set_active_groups(np.ones((M, NG), bool))
        t_ph = tick("fit.extensions", t_ph)
        self.n_iter = n_iter
        # BRIE_RV.concate appends the per-batch traces end to end (model_wrap.py:61): for every model, batch after
        # batch, each batch's last-stage trace followed by the rounds it was still active in
        self.pieces = pieces
        self.losses = []
        for m in range(M):
            parts = [p[m, g] for g in range(NG) for (a, p) in pieces if a[m, g]]
            self.losses.append(np.concatenate(parts) if parts else np.zeros(0, np.float32))
        self.loss_gene = self.eval_loss_gene(n_eval)                 # :261-264
        tick("fit.loss_gene", t_ph)
        if k_cap > 0:
            kms, kn = self.kernel_time_ms()
            self.phase_s["step_kernel_ms_sum"] = kms
            self.phase_s["step_kernel_launches"] = kn
            # algorithmic bytes of one full-width launch (SURVEY 8d): counts once + 48 B of state per model
            self.phase_s["step_kernel_alg_bytes_sum"] = kn * float(self.Nc) * self.Ng * (4 * self.n_layers + 48 * self.M)
            self.kernel_timing(0)
        return self.losses

    # ------------------------------------------------------------------ results
    def model_params(self, m):
        """Host copies in the reference's shapes for model m."""
        Ng = self.Ng
        out = {}
        out['Wc_loc'] = self.Wc[m, :len(self.masks[m]), :Ng].cpu().numpy()
        out['Wg_loc'] = self.Wg[m, :, :self.Kg_real].cpu().numpy()
        if self.cell_mode:
            out['intercept'] = self.intercept[m, :self.Nc].cpu().numpy().reshape(self.Nc, 1)
            out['sigma'] = np.exp(self.sigma_log[m, :self.Nc].cpu().numpy()).reshape(self.Nc, 1)
        else:
            out['intercept'] = self.intercept[m, :Ng].cpu().numpy().reshape(1, Ng)
            out['sigma'] = np.exp(self.sigma_log[m, :Ng].cpu().numpy()).reshape(1, Ng)
        return out


def _event_moments(adam_small, M, Kc, ld):
    """The per-event Adam moments (2, M, Kc + 2, ld) at the front of a fit's adam_small (brie_fit_create); the per-cell
    moments follow them."""
    return adam_small[:2 * M * (Kc + 2) * ld].view(2, M, Kc + 2, ld)


class _GatheredFit:
    """Sub-fit over gathered columns of a parent FitEngine (brie_fit_buffers.event_ids): model m's
    column j is the parent's local event cols[m][j].  Holds its own dense tiles of the state, the
    Adam moments, the counts (the parent's code words when it steps on packed codes, else its float32
    layers) and the lengths; shares Xc and the code dictionary with the parent."""

    def __init__(self, parent, cols, trace_cap):
        p = self.p = parent
        lib, dev, f32 = p.lib, p.device, torch.float32
        M, Nc, L, Kc = p.M, p.Nc, p.n_layers, p.Kc
        self.n = [len(c) for c in cols]
        nmax = max(max(self.n), 1)
        ld = self.ld = _lib.leading_dim(nmax)
        self.n_moves = 0

        d = _lib.FitDesc()
        C.memmove(C.byref(d), C.byref(p.desc), C.sizeof(d))
        d.n_events, d.ld, d.event_offset = nmax, ld, 0
        d.trace_cap = trace_cap
        d.rows_per_cta = p.sizes.rows_per_cta             # same association of the sums over cells
        self.h = C.c_void_p()
        _lib.check(lib.brie_fit_create(C.byref(d), C.byref(self.h)))
        sz = _lib.FitSizes()
        _lib.check(lib.brie_fit_get_sizes(self.h, C.byref(sz)))

        self.idx = [torch.from_numpy(np.ascontiguousarray(c, dtype=np.int64)).to(dev) for c in cols]
        ev = np.zeros((M, ld), np.int32)
        act = np.zeros((M, ld), np.uint8)
        for m, c in enumerate(cols):
            ev[m, :len(c)] = c + p.event_offset
            act[m, :len(c)] = 1
        self.ev_ids = torch.from_numpy(ev).to(dev)
        self.active = torch.from_numpy(act).to(dev)
        if p.count_codes is not None:
            self.counts = None
            self.codes = torch.empty((M, Nc, ld), dtype=torch.int32, device=dev)
        else:
            self.counts = torch.empty((L, M, Nc, ld), dtype=f32, device=dev)
            self.codes = None
        self.Z_loc = torch.empty((M, Nc, ld), dtype=f32, device=dev)
        self.Z_std_log = torch.empty((M, Nc, ld), dtype=f32, device=dev)
        self.adam_Z = torch.empty((4, M, Nc, ld), dtype=f32, device=dev)
        self.Wc = torch.zeros((M, max(Kc, 1), ld), dtype=f32, device=dev)
        self.intercept = torch.empty((M, ld), dtype=f32, device=dev)
        self.sigma_log = torch.empty((M, ld), dtype=f32, device=dev)
        self.adam_small = torch.zeros(max(int(sz.adam_small_floats), 4), dtype=f32, device=dev)
        self.mom = _event_moments(self.adam_small, M, Kc, ld)
        self.eff = torch.empty((M, 3, ld), dtype=f32, device=dev) if p.eff is not None else None
        self.loss_trace = torch.zeros((M, trace_cap, ld), dtype=f32, device=dev)
        self.scratch = torch.empty(int(sz.scratch_bytes // 4) + 4, dtype=f32, device=dev)
        self._move(gather=True)
        if self.eff is not None:
            for m in range(M):
                self.eff[m, :, self.n[m]:] = 1.0          # padding columns: harmless lengths

        b = _lib.FitBuffers()
        if self.counts is not None:
            for i in range(3):
                b.counts[i] = self.counts[i].data_ptr() if i < L else None
            b.counts_model_stride = Nc * ld
        b.efflen3 = self.eff.data_ptr() if self.eff is not None else None
        b.efflen_model_stride = 3 * ld if self.eff is not None else 0
        b.event_ids = self.ev_ids.data_ptr()
        b.Xc, b.Xg = p.Xc.data_ptr(), p.Xg.data_ptr()
        b.Z_loc, b.Z_std_log, b.adam_Z = self.Z_loc.data_ptr(), self.Z_std_log.data_ptr(), self.adam_Z.data_ptr()
        b.Wc, b.intercept, b.sigma_log = self.Wc.data_ptr(), self.intercept.data_ptr(), self.sigma_log.data_ptr()
        b.Wg, b.adam_small = p.Wg.data_ptr(), self.adam_small.data_ptr()
        b.active, b.loss_trace, b.scratch = self.active.data_ptr(), self.loss_trace.data_ptr(), self.scratch.data_ptr()
        self.bufs = b
        _lib.check(lib.brie_fit_bind(self.h, C.byref(b)))
        if self.codes is not None:
            _lib.check(lib.brie_fit_set_count_codes(self.h, self.codes.data_ptr(), Nc * ld,
                                                    p.count_codes[1].data_ptr()))

    def __del__(self):
        h = getattr(self, "h", None)
        if h is not None and h.value:
            self.p.lib.brie_fit_destroy(h)
            self.h = None

    def launches(self):
        return int(self.p.lib.brie_fit_launch_count(self.h)) + self.n_moves

    def _pairs(self, m, inputs, trace_rows):
        """(parent view, sub view) of model m, each rows x columns with the columns to move."""
        p, Kc = self.p, self.p.Kc
        pmom = _event_moments(p.adam_small, p.M, Kc, p.ld)
        out = [(p.Z_loc[m], self.Z_loc[m]), (p.Z_std_log[m], self.Z_std_log[m])]
        out += [(p.adam_Z[k, m], self.adam_Z[k, m]) for k in range(4)]
        if Kc > 0:
            out.append((p.Wc[m], self.Wc[m]))
        out += [(p.intercept[m:m + 1], self.intercept[m:m + 1]), (p.sigma_log[m:m + 1], self.sigma_log[m:m + 1])]
        out += [(pmom[j, m], self.mom[j, m]) for j in range(2)]
        if inputs:
            if self.codes is not None:
                out.append((p.count_codes[0], self.codes[m]))    # moved as 4-byte words: the bits are kept
            else:
                out += [(p.counts[i], self.counts[i, m]) for i in range(p.n_layers)]
            if self.eff is not None:
                out.append((p.eff, self.eff[m]))
        if trace_rows:
            out.append((p.loss_trace[m, :trace_rows], self.loss_trace[m, :trace_rows]))
        return out

    def _move(self, gather, trace_rows=0):
        """gather: parent -> sub (state, moments, counts, lengths); else scatter: sub -> parent (state,
        moments, loss trace)."""
        p, lib, st = self.p, self.p.lib, self.p._stream()
        for m in range(p.M):
            n, idx = self.n[m], self.idx[m].data_ptr()
            if n == 0 and not gather:
                continue
            for big, small in self._pairs(m, gather, trace_rows):
                assert big.is_contiguous() and small.is_contiguous()
                rows = big.shape[0]
                if gather:
                    _lib.check(lib.brie_gather_events(rows, p.ld, big.data_ptr(), idx, n, self.ld, small.data_ptr(), st))
                else:
                    _lib.check(lib.brie_scatter_events(rows, self.ld, small.data_ptr(), idx, n, p.ld, big.data_ptr(), st))
                self.n_moves += 1

    def run(self, n_steps, lr, adam_t, global_step):
        lib = self.p.lib
        _lib.check(lib.brie_fit_resume_stage(self.h, float(lr), int(adam_t), int(global_step)))
        _lib.check(lib.brie_fit_run_steps(self.h, int(n_steps), 0, self.p._stream()))
        self.n_ran = int(n_steps)

    def scatter_back(self):
        self._move(gather=False, trace_rows=self.n_ran)
