"""Wrap functions for running BRIE2 -- drop-in for brie/models/model_wrap.py.

`fit_BRIE_matrix` and `fitBRIE` keep the reference's signatures, defaults, prints
and outputs (brie/models/model_wrap.py:88-199, 202-314).  What changes is the
execution plan: the base/full fit and every LRT refit (the Python loop at
model_wrap.py:156-187) run as one batched `FitEngine`, and the sequential event
batches of `fitBRIE` (model_wrap.py:241-260) become convergence groups inside
the same launches, so one pass over the counts serves all of them.
"""
import hashlib
import time

import numpy as np
from scipy.stats import chi2

from ..engine import (SCORE_BLOCK_BYTES, FitEngine, group_pairs, score_from_parts, score_groups_from_parts,
                      wald_from_info, wald_groups_from_info)
from ..sharding import event_shards
from ..utils.layer_store import LayerStore, BIG_KEYS
from ..settings import verbosity


def fdr_bh(pvals):
    """Benjamini-Hochberg adjusted p-values, as statsmodels
    `multipletests(p, method="fdr_bh")[1]` used at model_wrap.py:195."""
    p = np.asarray(pvals, float)
    n = p.size
    if n == 0:
        return p.copy()
    order = np.argsort(p)
    adj = p[order] * n / np.arange(1, n + 1)
    adj = np.minimum.accumulate(adj[::-1])[::-1]
    adj[adj > 1] = 1
    out = np.empty(n)
    out[order] = adj
    return out


def fdr_by_group(pval, group_size=None, event_offset=0):
    """BH-FDR of each test column within the reference's multiple-testing scope.

    The reference corrects inside each fit_BRIE_matrix call (model_wrap.py:193-196), i.e. per
    event batch of ceil(batch_size / n_cells) events when called from fitBRIE (:241-256).
    Events fitted together here keep that scope per convergence group: `group_size` events per
    group, groups counted from global event 0 (`event_offset` = global index of row 0).
    Pinned on the reference's published result tables (tests/golden/published_lrt.npz)."""
    pval = np.asarray(pval)
    Ng = pval.shape[0]
    fdr = np.zeros(pval.shape)
    if group_size is None:
        bounds = [(0, Ng)]
    else:
        first = event_offset // group_size
        last = (event_offset + Ng - 1) // group_size
        bounds = [(max(g * group_size - event_offset, 0), min((g + 1) * group_size - event_offset, Ng))
                  for g in range(first, last + 1)]
    for lo, hi in bounds:
        for i in range(fdr.shape[1]):
            fdr[lo:hi, i] = fdr_bh(pval[lo:hi, i])
    return fdr


MAX_MODEL_IDS = 4096                       # 12-bit model word of the Philox stream (csrc/brie_philox.h)


def perm_indices(seed, t, b, Nc):
    """Cell permutation of replicate b of test position t (index into LRT_index, not the covariate number).
    It depends on (seed, t, b, Nc) alone, so every event chunk and every rank permutes the cells alike."""
    return np.random.default_rng((int(seed), 1 + int(t), int(b))).permutation(int(Nc))


def perm_model_id(t, b, n_tests, n_perm):
    """RNG model word of permuted model (t, b): after the base model (0) and the LRT refits (1..T)."""
    return 1 + n_tests + t * n_perm + b


def check_n_perm(n_perm, n_tests):
    """Validate `n_perm` for a fit with `n_tests` tested covariates (before any device work)."""
    if isinstance(n_perm, bool) or int(n_perm) != n_perm:
        raise ValueError("n_perm must be an integer, got %r" % (n_perm,))
    n_perm = int(n_perm)
    if n_perm < 0:
        raise ValueError("n_perm must be >= 0, got %d" % n_perm)
    if n_perm > 0 and n_tests == 0:
        raise ValueError("n_perm > 0 needs at least one tested covariate (LRT_index)")
    if 1 + n_tests * (1 + n_perm) > MAX_MODEL_IDS:
        raise ValueError("n_perm = %d with %d tested covariates needs %d model ids; the noise stream has %d"
                         % (n_perm, n_tests, 1 + n_tests * (1 + n_perm), MAX_MODEL_IDS))
    return n_perm


def check_groups(groups, n_cols, name):
    """Validate `groups` (before any device work): None, or a non-empty list of groups, each a non-empty list of
    distinct integer column indices in [0, n_cols).  Returned as lists of int."""
    if groups is None:
        return None
    try:
        groups = [list(G) for G in groups]
    except TypeError:
        raise ValueError("%s must be a list of groups of column indices, got %r" % (name, groups)) from None
    if not groups:
        raise ValueError("%s must hold at least one group" % name)
    for G in groups:
        if not G:
            raise ValueError("%s: a group is empty" % name)
        for k in G:
            if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)):
                raise ValueError("%s: column index %r is not an integer" % (name, k))
            if not 0 <= k < n_cols:
                raise ValueError("%s: column index %d is out of range for %d columns" % (name, k, n_cols))
        if len(set(int(k) for k in G)) != len(G):
            raise ValueError("%s: group %r repeats a column index" % (name, [int(k) for k in G]))
    return [[int(k) for k in G] for G in groups]


def _base_columns(Kc, LRT_index, full):
    """Columns of model 0 (model_wrap.py:130-136): all of Xc in base_mode 'full', else those not tested."""
    if full:
        return list(range(Kc))
    if LRT_index is not None and len(LRT_index) < Kc:
        return [k for k in range(Kc) if k not in set(int(i) for i in LRT_index)]
    return []


def group_model_id(i, n_tests, n_perm):
    """RNG model word of the refit of LRT group i: after the base model, the LRT refits and the permuted models."""
    return 1 + n_tests * (1 + n_perm) + i


def check_LRT_groups(groups, Kc, base_cols, full, n_tests, n_perm):
    """Validate `LRT_groups` (before any device work): groups of Xc columns; with base_mode 'null' a group is added to
    the base model and must not overlap its columns; every group model needs a model id of the noise stream."""
    groups = check_groups(groups, Kc, "LRT_groups")
    if groups is None:
        return None
    if not full:
        for G in groups:
            if set(G) & set(base_cols):
                raise ValueError("LRT_groups: group %r overlaps the base model's columns %r (base_mode 'null' adds "
                                 "the group to the base model)" % (G, base_cols))
    n_ids = group_model_id(len(groups), n_tests, n_perm)
    if n_ids > MAX_MODEL_IDS:
        raise ValueError("LRT_groups: %d groups with %d tested covariates and n_perm = %d need %d model ids; the noise "
                         "stream has %d" % (len(groups), n_tests, n_perm, n_ids, MAX_MODEL_IDS))
    return groups


def check_wald_groups(groups, Kc, base_cols, target):
    """Validate `wald_groups` (before any device work): groups of the columns model 0 fits (any Xc column in
    base_mode 'full', the base columns in 'null'); a marginLik fit trains no posterior."""
    if groups is None:
        return None
    if target == "marginLik":
        raise ValueError("wald_groups needs target 'ELBO': a marginLik fit has no trained posterior")
    groups = check_groups(groups, Kc, "wald_groups")
    for G in groups:
        if not set(G) <= set(base_cols):
            raise ValueError("wald_groups: group %r has columns model 0 does not fit (its columns: %r)" % (G, base_cols))
    return groups


def check_score_groups(groups, score_X, target):
    """Validate `score_groups` (before any device work): groups of columns of the (validated) score_X."""
    if groups is None:
        return None
    if target == "marginLik":
        raise ValueError("score_groups needs target 'ELBO': a marginLik fit has no trained posterior")
    if score_X is None:
        raise ValueError("score_groups needs score_X: a group is a group of score_X columns")
    return check_groups(groups, score_X.shape[1], "score_groups")


# (statistic or gain, p-value, FDR) of each kind of joint test of a group, each (Ng, groups)
GROUP_KEYS = (('ELBO_gain_group', 'pval_group', 'fdr_group'),
              ('wald_stat_group', 'pval_wald_group', 'fdr_wald_group'),
              ('score_stat_group', 'pval_score_group', 'fdr_score_group'))


def _set_fdr_groups(res):
    """fdr_group / fdr_wald_group / fdr_score_group: BH over all events of the result, per group (the pooled scope
    of fdr_wald), for each kind of group test the result holds."""
    for _, pk, fk in GROUP_KEYS:
        if hasattr(res, pk):
            p = getattr(res, pk)
            fdr = np.zeros(p.shape)
            for i in range(p.shape[1]):
                fdr[:, i] = fdr_bh(p[:, i])
            setattr(res, fk, fdr)


def _append_groups(out, r):
    """Event-axis concatenation of the group-test outputs of two results (the FDRs are recomputed over all events)."""
    for keys in GROUP_KEYS:
        if hasattr(r, keys[1]):
            for k in keys:
                setattr(out, k, np.append(getattr(out, k), getattr(r, k), axis=0))


def perm_pvalue(gain, gain_perm):
    """Pooled empirical p-values (Ng, T) of the observed gains `gain` (Ng, T) against the permutation null
    `gain_perm` (Ng, T, B) of every event: (1 + #{(g', b) : gain_perm[g', t, b] >= gain[g, t]}) / (1 + Ng * B).
    NaN compares False, as in the double loop."""
    gain, gain_perm = np.asarray(gain), np.asarray(gain_perm)
    Ng, T, B = gain_perm.shape
    out = np.empty(gain.shape, np.float64)
    for t in range(T):
        null = np.sort(gain_perm[:, t, :].reshape(-1))
        null = null[~np.isnan(null)]
        n_ge = null.size - np.searchsorted(null, gain[:, t], side='left')
        out[:, t] = (1.0 + n_ge) / (1.0 + Ng * B)
    return out


def _set_perm_outputs(res):
    """pval_perm and fdr_perm of a result holding ELBO_gain and ELBO_gain_perm, over all of its events: one
    pooled null and one BH scope per tested covariate.  This scope differs on purpose from the chi2 FDR's
    (fdr_by_group, the reference's per-batch scope, degenerate at 1-event batches)."""
    res.pval_perm = perm_pvalue(res.ELBO_gain, res.ELBO_gain_perm)
    res.fdr_perm = np.zeros(res.pval_perm.shape)
    for i in range(res.fdr_perm.shape[1]):
        res.fdr_perm[:, i] = fdr_bh(res.pval_perm[:, i])


def check_wald(wald, target):
    """Validate `wald` against the fit's `target` (before any device work): a marginLik fit trains no posterior."""
    wald = bool(wald)
    if wald and target == "marginLik":
        raise ValueError("wald=True needs target 'ELBO': a marginLik fit has no trained posterior")
    return wald


def _coef_and_info(eng, j):
    """(coef (Ng, K~), info (Ng, K~, K~)) of model j of a fitted engine: its Wc rows, then its intercept when that is
    per-event and trained, and their observed information from its posterior (FitEngine.wald_info)."""
    import torch
    w = len(eng.masks[j])
    coef = [eng.Wc[j, :w, :eng.Ng].T.double()]
    if not eng.cell_mode and eng.intercept_const is None:
        coef.append(eng.intercept[j, :eng.Ng, None].double())
    return torch.cat(coef, dim=1).cpu().numpy(), eng.wald_info(j)


def _wald_of_model(eng, j):
    """(se, pval, width) of model j of a fitted engine: Wald statistics of its Wc rows, then of its intercept when
    that is per-event and trained (_coef_and_info)."""
    se, pval = wald_from_info(*_coef_and_info(eng, j))
    return se, pval, len(eng.masks[j])


def _set_fdr_wald(res):
    """fdr_wald: BH over all events of the result, per cell_coeff row (the pooled scope of fdr_perm)."""
    res.fdr_wald = np.zeros(res.pval_wald.shape)
    for i in range(res.fdr_wald.shape[1]):
        res.fdr_wald[:, i] = fdr_bh(res.pval_wald[:, i])


def _set_wald_outputs(res, per_model, full, base_cols, tested):
    """Wald outputs in the layout of cell_coeff: model 0's Xc rows, then (base_mode 'null') the last row of each
    test model t, from model t's own information.  per_model[m] = _wald_of_model of model id m."""
    se0, p0, w0 = per_model[0]
    se, pv = [se0[:, :w0]], [p0[:, :w0]]
    if not full:
        for t in range(len(tested)):
            se_t, p_t, w_t = per_model[1 + t]
            se.append(se_t[:, w_t - 1:w_t])
            pv.append(p_t[:, w_t - 1:w_t])
    res.cell_coeff_se = np.concatenate(se, axis=1).T                # (rows, Ng), as cell_coeff
    res.pval_wald = np.concatenate(pv, axis=1)                      # (Ng, rows)
    if se0.shape[1] > w0:
        res.intercept_se = se0[:, w0][None, :]                      # (1, Ng), as a per-event intercept
    res.wald_columns = [int(k) for k in base_cols] + ([] if full else [int(k) for k in tested])
    _set_fdr_wald(res)


SCORE_KEYS = ('score_z', 'score_effect', 'pval_score', 'fdr_score')


def check_score_X(score_X, target, Nc):
    """Validate `score_X` against the fit (before any device work): None, or a finite (Nc, J >= 1) matrix of
    candidate cell covariates, returned as float32; a marginLik fit trains no posterior to score against."""
    if score_X is None:
        return None
    if target == "marginLik":
        raise ValueError("score_X needs target 'ELBO': a marginLik fit has no trained posterior")
    X = np.asarray(score_X, np.float32)
    if X.ndim != 2 or X.shape[0] != Nc or X.shape[1] < 1:
        raise ValueError("score_X must be (n_cells=%d, J >= 1), got shape %s" % (Nc, np.shape(score_X)))
    if not np.isfinite(X).all():
        raise ValueError("score_X has non-finite values")
    return X


def _score_of_model(eng, j, X, groups=None):
    """((score_z, score_effect, pval_score), group tests) of candidates X against model j of a fitted engine as the
    null model (FitEngine.score_parts with the model's information, score_from_parts).  With `groups`, the group
    tests are the joint tests (score_stat_group, pval_score_group) of those groups of candidates
    (FitEngine.score_cross, score_groups_from_parts), else None.  X goes to the device once for both passes."""
    import torch
    X = torch.from_numpy(np.ascontiguousarray(X, np.float32)).to(eng.device)
    parts, info = eng.score_parts(j, X), eng.wald_info(j)
    single = score_from_parts(parts, info)
    if groups is None:
        return single, None
    pairs = group_pairs(groups)
    return single, score_groups_from_parts(parts, eng.score_cross(j, X, pairs), pairs, info, groups)


def _set_fdr_score(res):
    """fdr_score: BH over all events of the result, per candidate (the pooled scope of fdr_wald)."""
    res.fdr_score = np.zeros(res.pval_score.shape)
    for i in range(res.fdr_score.shape[1]):
        res.fdr_score[:, i] = fdr_bh(res.pval_score[:, i])


def _append_score(out, r):
    """Event-axis concatenation of the score outputs of two results (fdr_score is recomputed over all events)."""
    for k in SCORE_KEYS:
        setattr(out, k, np.append(getattr(out, k), getattr(r, k), axis=0))


def _append_wald(out, r):
    """Event-axis concatenation of the Wald outputs of two results (fdr_wald is recomputed over all events)."""
    out.cell_coeff_se = np.append(out.cell_coeff_se, r.cell_coeff_se, axis=1)
    for k in ('pval_wald', 'fdr_wald'):
        setattr(out, k, np.append(getattr(out, k), getattr(r, k), axis=0))
    if hasattr(r, 'intercept_se'):
        out.intercept_se = np.append(out.intercept_se, r.intercept_se, axis=1)


class BRIE_RV():
    """Return value object for BRIE2 model (model_wrap.py:15-76)."""

    def __init__(self, model=None):
        if model is None:
            return
        self.Nc, self.Ng, self.Kc, self.Kg = model.Nc, model.Ng, model.Kc, model.Kg
        self.shape = (self.Nc, self.Ng)
        self.Xc, self.Xg = model.Xc, model.Xg
        self.sigma = model.sigma.numpy()
        self.intercept = model.intercept.numpy()
        self.cell_coeff = model.Wc_loc.numpy()
        self.gene_coeff = model.Wg_loc.numpy()
        self.Psi = model.Psi.numpy()
        self.Psi95CI = model.Psi95CI
        self.Z_loc = model.Z_loc.numpy()
        self.Z_std = model.Z_std.numpy()
        self.losses = model.losses.numpy()
        self.loss_gene = model.loss_gene.numpy()
        self.intercept_mode = model.intercept_mode

    @property
    def Wc_loc(self):
        return self.cell_coeff

    @property
    def Wg_loc(self):
        return self.gene_coeff

    def __str__(self):
        return "BRIE2 results for %d cells and %d genes" % (self.Nc, self.Ng)

    def concate(self, new_RV, axis=1):
        if axis != 1:
            print("Warning: only suppoting gene level concate!")
            return None
        self.Ng += new_RV.Ng
        self.shape = (self.Nc, self.Ng)
        self.losses = np.append(self.losses, new_RV.losses)
        self.loss_gene = np.append(self.loss_gene, new_RV.loss_gene)
        self.sigma = np.append(self.sigma, new_RV.sigma, axis=1)
        self.intercept = np.append(self.intercept, new_RV.intercept, axis=1)
        self.cell_coeff = np.append(self.cell_coeff, new_RV.cell_coeff, axis=1)
        self.Psi = np.append(self.Psi, new_RV.Psi, axis=1)
        self.Psi95CI = np.append(self.Psi95CI, new_RV.Psi95CI, axis=1)
        self.Z_std = np.append(self.Z_std, new_RV.Z_std, axis=1)
        self.Z_loc = np.append(self.Z_loc, new_RV.Z_loc, axis=1)
        if hasattr(new_RV, 'ELBO_gain'):
            self.fdr = np.append(self.fdr, new_RV.fdr, axis=0)
            self.pval = np.append(self.pval, new_RV.pval, axis=0)
            self.ELBO_gain = np.append(self.ELBO_gain, new_RV.ELBO_gain, axis=0)
        if hasattr(new_RV, 'ELBO_gain_perm'):           # pval_perm / fdr_perm: fitBRIE recomputes them over all events
            for k in ('ELBO_gain_perm', 'pval_perm', 'fdr_perm'):
                setattr(self, k, np.append(getattr(self, k), getattr(new_RV, k), axis=0))
        if hasattr(new_RV, 'pval_wald'):
            _append_wald(self, new_RV)
        if hasattr(new_RV, 'pval_score'):
            _append_score(self, new_RV)
        _append_groups(self, new_RV)
        if hasattr(new_RV, 'n_iter'):
            self.n_iter = np.append(self.n_iter, new_RV.n_iter, axis=1)
        if getattr(self, 'timing', None) is not None and getattr(new_RV, 'timing', None) is not None:
            for k, v in new_RV.timing.items():                      # BRIE_TIMING diagnostics add up over chunks
                self.timing[k] = self.timing.get(k, 0.0) + v


def concate(BRIE_RV_list):
    """Concate a list of BRIE results (model_wrap.py:78-85)."""
    res_merge = BRIE_RV_list[0]
    for _res in BRIE_RV_list[1:]:
        res_merge.concate(_res)
    return res_merge


class _ChunkSink:
    """Where fit_BRIE_matrix leaves the dense layers of one event chunk when fitBRIE drives it: the chunk's column
    range of a LayerStore, copied by a background thread so that the transfer overlaps the next chunk's fit.
    `before_outputs` is called before this chunk's output tensors are allocated (fitBRIE waits for the previous
    chunk's copy there, so at most one chunk's outputs are alive on the device at a time)."""

    def __init__(self, store, e0, before_outputs=None, background=True):
        self.store, self.e0, self.before_outputs, self.background = store, e0, before_outputs, background
        self.copy = None

    def wait(self):
        if self.copy is not None:
            self.copy.wait()
            self.copy = None


def _rv_from_engine(eng, m, Xc_model, Xg, intercept_mode, sink=None):
    """Result container of model m.  The dense (cells, events) arrays Psi / Psi95CI / Z_std / Z_loc go to the host
    through pinned staging (utils/d2h.py): into fresh arrays, or -- `sink` a _ChunkSink -- straight into their
    column range of the store's arrays / memory maps, leaving (cells, 0) stubs in the container."""
    from ..utils import d2h
    rv = BRIE_RV()
    rv.Nc, rv.Ng = eng.Nc, eng.Ng
    rv.Kc, rv.Kg = len(eng.masks[m]), eng.Kg_real
    rv.shape = (rv.Nc, rv.Ng)
    rv.Xc, rv.Xg = Xc_model, Xg
    p = eng.model_params(m)
    rv.sigma, rv.intercept = p['sigma'], p['intercept']
    rv.cell_coeff, rv.gene_coeff = p['Wc_loc'], p['Wg_loc']
    rv.losses = eng.losses[m]
    rv.loss_gene = eng.loss_gene[m].cpu().numpy()
    rv.intercept_mode = intercept_mode
    if sink is not None and sink.before_outputs is not None:
        sink.before_outputs()
    Psi, CI, Zstd = eng.posterior(m)
    big = dict(Psi=Psi, Psi95CI=CI, Z_std=Zstd, Z_loc=eng.Z_loc[m, :, :eng.Ng])
    if sink is None:
        for k, t in big.items():
            setattr(rv, k, d2h.to_host(t))
        return rv
    jobs = []
    for k, t in big.items():
        if k in sink.store.arrays:
            if k == 'Z_loc' and sink.background:
                t = t.clone()                      # the engine's state is freed while the copy is still running
            jobs.append((t, sink.store.arrays[k], sink.e0))
        setattr(rv, k, np.zeros((rv.Nc, 0), np.float32))
    if sink.background:
        sink.copy = d2h.BackgroundCopy(jobs, eng.device)
    else:
        for t, dst, c0 in jobs:
            d2h.to_host_columns(t, dst, c0)
    return rv


def _host_pseudo_count_inplace(data, pseudo_count):
    """Side effect of model_wrap.py:113-117 on the caller's dense arrays: where c1 + c2 > 0 add the
    pseudo-count to c1 and c2 in place.  (The fit itself reads the device tiles.)

    Read-only arrays (`np.load(mmap_mode='r')`, `writeable=False`) raise the ValueError numpy's
    in-place assignment raises in the reference; they are never written through another view."""
    for d in data[:2]:
        if not d.flags.writeable:
            raise ValueError("assignment destination is read-only")
    idx = data[0] + data[1] > 0
    for i in range(2):
        np.add(data[i], pseudo_count, out=data[i], where=idx, casting='unsafe')


def _engine_plan(base_cols, test_masks, cell_mode, intercept_mode, max_models=None, n_perm=0, tested=(),
                 n_cols=0, full=True, group_masks=()):
    """[(column masks, model ids, intercept mode)] per FitEngine: the base model (id 0) with as many LRT refits
    (ids 1..T) as one launch batches, the remaining refits in further engines of at most `max_models` models; a
    cell-mode base model sits alone, because the reference's refits always use the per-event layout
    (model_wrap.py:174-178).

    With `n_perm` = B > 0 the permuted models (t, b) follow in additional engines, never in the observed ones:
    an engine's model count sets the association of its float32 cell sums, so the observed outputs stay
    bit-identical to the B = 0 fit, and no engine is larger than the largest observed one (the device budget
    of fitBRIE holds).  Model (t, b) is the observed alternative of test t -- the full model (base_mode
    'full', base layout) or test model t (base_mode 'null', per-event layout) -- with column tested[t] replaced
    in place by column n_cols + j of the engine's design, j its position in the engine; its id is
    perm_model_id(t, b, T, B).

    The refits of LRT groups (`group_masks`, one column mask per group) follow the permuted models in further
    engines under the same size rule, in the per-event layout of the LRT refits; group i has id
    group_model_id(i, T, B)."""
    if max_models is None:
        from .._lib import BRIE_MAX_MODELS as max_models
    T = len(test_masks)
    plan = []
    if cell_mode and T > 0:
        plan.append(([base_cols], [0], intercept_mode))
        first_tests = 0
    else:
        first_tests = min(T, max_models - 1)
        plan.append(([base_cols] + test_masks[:first_tests], list(range(first_tests + 1)), intercept_mode))
    for t0 in range(first_tests, T, max_models):
        t1 = min(t0 + max_models, T)
        plan.append((test_masks[t0:t1], list(range(1 + t0, 1 + t1)), 'gene'))
    size = min(max(len(ids) for _, ids, _ in plan), max_models)
    if n_perm > 0:
        perm = [(t, b) for t in range(T) for b in range(n_perm)]
        for p0 in range(0, len(perm), size):
            part = perm[p0:p0 + size]
            masks = [[n_cols + j if k == tested[t] else k for k in (base_cols if full else test_masks[t])]
                     for j, (t, b) in enumerate(part)]
            plan.append((masks, [perm_model_id(t, b, T, n_perm) for t, b in part], intercept_mode if full else 'gene'))
    for g0 in range(0, len(group_masks), size):
        g1 = min(g0 + size, len(group_masks))
        plan.append(([list(m) for m in group_masks[g0:g1]], [group_model_id(i, T, n_perm) for i in range(g0, g1)],
                     'gene'))
    return plan


def fit_BRIE_matrix(data, Xc=None, Xg=None, effLen=None, intercept=None,
                    intercept_mode='gene', LRT_index=None, pseudo_count=0.01,
                    sigma=None, base_mode='full', tau_prior=[3, 27], score_X=None, LRT_groups=None,
                    wald_groups=None, score_groups=None, **keyargs):
    """Fit a BRIE model with cell and/or gene features (model_wrap.py:88-199).

    Extra keyword arguments consumed here (not in the reference): `seed` (noise and
    init key, default 0), `group_size` / `event_offset` / `n_events_total` (reference
    batch geometry when called from fitBRIE), `device`, `init_objs` (per-model
    injected initial values: [base, refit_0, ...]), `n_eval` (loss_gene evaluations,
    500 in the reference), `dist_group`, `n_perm` (permutation null, default 0: see below), `wald`
    (Wald tests from the fitted posterior, default False: see below).
    All other **keyargs go to the fit schedule as in the reference (`min_iter, max_iter,
    add_iter, epsilon_conv, MC_size`).

    `n_perm` = B > 0 also fits, for every test position t and replicate b < B, the observed
    alternative of test t (the full model, or test model t with base_mode 'null') with the tested
    column's cells permuted by `perm_indices(seed, t, b, Nc)`, and returns `ELBO_gain_perm`
    (Ng, T, B), its null gains; `pval_perm` (Ng, T), the pooled empirical p-values of `ELBO_gain`
    against the gains of every event and replicate (`perm_pvalue`); and `fdr_perm`, BH over all
    events.  Permuted models only evaluate `loss_gene`; the observed outputs are bit-identical to
    the n_perm = 0 fit.

    `wald=True` adds Wald statistics of the cell coefficients from the observed information of the fitted
    posterior (FitEngine.wald_info; no refit): `cell_coeff_se` in the layout of `cell_coeff` (model 0's rows;
    base_mode 'null': then the last row of each test model, from that model's own information), `intercept_se`
    (1, Ng) when the intercept is per-event and trained, `pval_wald` / `fdr_wald` (Ng, rows of cell_coeff; BH
    over all events) and `wald_columns`, the Xc column of each cell_coeff row.  Every other output is unchanged.

    `score_X` (Nc, J), candidate cell covariates aligned with the cells, adds their Rao score tests against model 0
    (the full model, or the base model with base_mode 'null') from its fitted posterior, without refits (DESIGN
    §2.3): `score_z`, `score_effect` (one-step estimate of each candidate's coefficient, logit scale), `pval_score`
    and `fdr_score` (BH per candidate over all events), each (Ng, J).  A candidate collinear with the fitted columns
    or zero on every cell, and an event whose information is not positive definite, get NaN and pval 1.  Every
    other output is unchanged.

    Joint tests of groups of columns (DESIGN §2.4; a group is a list of distinct 0-based column indices, each input a
    list of groups; at None nothing changes):
    `LRT_groups` refits, per group, the full model without the group's columns (base_mode 'null': the base model plus
    the group's columns, which must not overlap it), in the per-event layout of the LRT refits, and returns
    `ELBO_gain_group` (Ng, G), `pval_group` = chi2.sf(2 gain, df=len(group)) and `fdr_group` (BH over all events).
    Group refits only evaluate `loss_gene`.
    `wald_groups`, groups of model 0's columns, returns the joint Wald statistic beta_G^T ((I^-1)_GG)^-1 beta_G from
    model 0's information (no refit; also without `wald`): `wald_stat_group`, `pval_wald_group`, `fdr_wald_group`.
    `score_groups`, groups of score_X columns, returns their joint score statistics against model 0:
    `score_stat_group`, `pval_score_group`, `fdr_score_group`.  An undefined statistic is NaN with p-value 1.
    """
    from scipy.sparse import issparse
    seed = keyargs.pop('seed', 0)
    group_size = keyargs.pop('group_size', None)
    event_offset = keyargs.pop('event_offset', 0)
    n_events_total = keyargs.pop('n_events_total', None)
    device = keyargs.pop('device', None)
    init_objs = keyargs.pop('init_objs', None)
    dist_group = keyargs.pop('dist_group', None)
    n_eval = keyargs.pop('n_eval', 500)
    MC_size = keyargs.pop('MC_size', 1)
    target = keyargs.pop('target', "ELBO")                          # reaches BRIE2.fit through **keyargs (:144)
    host_side_effect = keyargs.pop('host_side_effect', True)
    out_sink = keyargs.pop('out_sink', None)                        # _ChunkSink: fitBRIE's output arrays
    n_tests = len(LRT_index) if LRT_index is not None else (0 if Xc is None else np.shape(Xc)[1])
    n_perm = check_n_perm(keyargs.pop('n_perm', 0), n_tests)
    wald = check_wald(keyargs.pop('wald', False), target)
    score_X = check_score_X(score_X, target, data[0].shape[0])
    full = base_mode.upper() == 'FULL'
    Kc = 0 if Xc is None else np.shape(Xc)[1]
    base_cols = _base_columns(Kc, LRT_index, full)
    LRT_groups = check_LRT_groups(LRT_groups, Kc, base_cols, full, n_tests, n_perm)
    wald_groups = check_wald_groups(wald_groups, Kc, base_cols, target)
    score_groups = check_score_groups(score_groups, score_X, target)
    for k in ('optimizer', 'learn_rate', 'verbose'):                # accepted and ignored (:214-237)
        keyargs.pop(k, None)

    import os
    import time
    import torch
    from .. import ingest
    timing = {} if (os.environ.get("BRIE_TIMING") or os.environ.get("BRIE_KERNEL_TIMING")) else None         # phase wall times (diagnostic; syncs the device)

    def _tick(name, t0):
        if timing is not None:
            torch.cuda.synchronize()
            timing[name] = timing.get(name, 0.0) + time.perf_counter() - t0
        return time.perf_counter()

    t_ph = time.perf_counter()
    if not torch.cuda.is_available():
        raise RuntimeError("brie_b200: no CUDA device (there is no CPU fallback)")
    dev = torch.device(device if device is not None else "cuda")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    Nc, Ng = data[0].shape
    print("[BRIE2] adding pseudo_count:", pseudo_count)
    # The stored counts go to the device as they are (sparse layers are NOT densified on the
    # host, :108-111), are scattered there and get the pseudo-count there (:113-117).
    tiles, h2d_bytes = [], 0
    for d in data:
        t, nb = ingest.layer_to_device(d, 0, Ng, dev)
        tiles.append(t)
        h2d_bytes += nb
    ingest.add_pseudo_count(tiles, pseudo_count)
    # the reference also leaves the pseudo-count in the caller's dense arrays (in-place add, :115-117)
    # -- only where the reference's arrays are the caller's own: fitBRIE's event batches are copies
    # (fancy indexing with a range, :245-249), so fitBRIE passes host_side_effect=False for its slices
    if host_side_effect and all(isinstance(d, np.ndarray) for d in data[:2]):
        _host_pseudo_count_inplace(data, pseudo_count)
    t_ph = _tick("pseudo_count+ingest", t_ph)
    if Xc is None:
        Xc = np.ones((Nc, 0), np.float32)
    if Xg is None:
        Xg = np.ones((Ng, 0), np.float32)
    Xc = np.asarray(Xc, np.float32)
    Xg = np.asarray(Xg, np.float32)
    if LRT_index is None:                                           # :149-150
        LRT_index = np.arange(Kc)
    LRT_index = [int(i) for i in LRT_index]

    # column masks over the full Xc: model 0 = base/full, model 1+ii = refit ii (:156-171)
    test_masks = []
    for idx_k in LRT_index:
        if full:
            if verbosity == 3:
                print("[BRIE2] fitting null model without feature %d" % (idx_k))
            test_masks.append([k for k in range(Kc) if k != idx_k])
        else:
            if verbosity == 3:
                print("[BRIE2] fitting test model by add feature %d" % (idx_k))
            test_masks.append(base_cols + [idx_k])

    trace_cap = max(int(keyargs.get('min_iter', 1000) / 6), int(keyargs.get('add_iter', 500)), 1)
    common = dict(effLen=effLen, Xc=Xc, Xg=Xg, intercept=intercept, sigma=sigma, MC_size=MC_size,
                  seed=seed, group_size=group_size, event_offset=event_offset,
                  n_events_total=n_events_total, device=dev, trace_cap=trace_cap,
                  dist_group=dist_group, n_events=Ng, target=target)
    data = tiles
    cell_mode = intercept_mode.upper() == 'CELL'
    T = len(test_masks)
    # Engine plan: (masks, model ids, intercept mode) per FitEngine.  One engine holds the base model and as
    # many refits as one launch batches (BRIE_MAX_MODELS = 32); a one-vs-rest LRT over more covariates than
    # that runs the remaining refits in further engines, one after the other, over the same device tiles.
    # NB the reference builds the refits WITHOUT intercept_mode (model_wrap.py:174-178), so they always use
    # the default per-event ('gene') intercept/sigma layout: a cell-mode base model gets an engine of its own.
    group_masks = [[k for k in range(Kc) if k not in G] if full else base_cols + G for G in (LRT_groups or [])]
    first_group = group_model_id(0, T, n_perm)
    plan = _engine_plan(base_cols, test_masks, cell_mode, intercept_mode, n_perm=n_perm, tested=LRT_index,
                        n_cols=Kc, full=full, group_masks=group_masks)
    t_ph = _tick("engine_setup", t_ph)

    brie_results = None
    n_iter_rows, lg_tests, wc_last, launches = [None] * (T + 1), [None] * T, [None] * T, 0
    lg_perm = {}                                                    # (t, b) -> loss_gene of permuted model (t, b)
    lg_group = {}                                                   # i -> loss_gene of the refit of LRT group i
    wald_out = {}                                                   # model id -> _wald_of_model (base, null-mode tests)
    codes = None                                                    # the chunk's packed count codes, encoded once
    for masks_e, ids_e, mode_e in plan:
        io, kw_e = None, common
        if T < ids_e[0] < first_group:                              # permuted models: their columns appended to Xc
            tb = [divmod(mid - 1 - T, n_perm) for mid in ids_e]
            cols = [Xc[perm_indices(seed, t, b, Nc), LRT_index[t]] for t, b in tb]
            kw_e = dict(common, Xc=np.concatenate([Xc, np.stack(cols, axis=1)], axis=1))
        elif init_objs is not None and ids_e[0] < first_group:
            io = [init_objs[i] for i in ids_e]
        eng = FitEngine(data, masks=masks_e, model_ids=ids_e, intercept_mode=mode_e, count_codes=codes, **kw_e)
        codes = eng.count_codes
        eng.fit(n_eval=n_eval, init_objs=io, **keyargs)             # :144, :180
        t_ph = _tick("fit", t_ph)
        if timing is not None:
            for k, v in eng.phase_s.items():
                timing[k] = timing.get(k, 0.0) + v
        for j, mid in enumerate(ids_e):
            if mid >= first_group:
                lg_group[mid - first_group] = eng.loss_gene[j].cpu().numpy()
                continue
            if mid > T:
                lg_perm[divmod(mid - 1 - T, n_perm)] = eng.loss_gene[j].cpu().numpy()
                continue
            n_iter_rows[mid] = eng.n_iter[j]
            if wald and (mid == 0 or not full):
                wald_out[mid] = _wald_of_model(eng, j)
            if wald_groups is not None and mid == 0:            # positions of the groups' columns in model 0
                wald_group_out = wald_groups_from_info(*_coef_and_info(eng, j),
                                                       [[base_cols.index(k) for k in G] for G in wald_groups])
            if score_X is not None and mid == 0:
                score_out, score_group_out = _score_of_model(eng, j, score_X, score_groups)
            if mid == 0:
                brie_results = _rv_from_engine(eng, j, Xc[:, base_cols], Xg, intercept_mode, out_sink)   # :146
            else:
                lg_tests[mid - 1] = eng.loss_gene[j].cpu().numpy()
                if not full:
                    wc_last[mid - 1] = eng.Wc[j, len(eng.masks[j]) - 1, :Ng].cpu().numpy()[None, :]
        launches += eng.launch_count
        del eng                                                     # the next engine reuses the state memory
        t_ph = _tick("posterior+d2h", t_ph)
    brie_results.n_iter = np.stack(n_iter_rows, axis=0)             # (1+T, groups)
    brie_results.launch_count = launches
    brie_results.h2d_bytes = h2d_bytes
    brie_results.timing = timing
    if wald:
        _set_wald_outputs(brie_results, wald_out, full, base_cols, LRT_index)
    if score_X is not None:
        brie_results.score_z, brie_results.score_effect, brie_results.pval_score = score_out
        _set_fdr_score(brie_results)
    if LRT_groups is not None:
        gain = np.zeros((Ng, len(LRT_groups)), dtype=np.float32)
        pval = np.zeros((Ng, len(LRT_groups)))
        for i, G in enumerate(LRT_groups):
            gain[:, i] = lg_group[i] - brie_results.loss_gene if full else brie_results.loss_gene - lg_group[i]
            pval[:, i] = chi2.sf(2 * gain[:, i], df=len(G))
        brie_results.ELBO_gain_group, brie_results.pval_group = gain, pval
    if wald_groups is not None:
        brie_results.wald_stat_group, brie_results.pval_wald_group = wald_group_out
    if score_groups is not None:
        brie_results.score_stat_group, brie_results.pval_score_group = score_group_out
    _set_fdr_groups(brie_results)
    if T == 0:                                                      # :152-153
        return brie_results

    ELBO_gain = np.zeros((Ng, T), dtype=np.float32)                 # :155
    for ii, idx_k in enumerate(LRT_index):
        if full:
            ELBO_gain[:, ii] = lg_tests[ii] - brie_results.loss_gene     # :183
        else:
            ELBO_gain[:, ii] = brie_results.loss_gene - lg_tests[ii]     # :185
            brie_results.cell_coeff = np.append(brie_results.cell_coeff, wc_last[ii], axis=0)  # :186-187
    brie_results.ELBO_gain = ELBO_gain                              # H1 vs NUll
    brie_results.pval = chi2.sf(2 * ELBO_gain, df=1)                # :190
    fdr = fdr_by_group(brie_results.pval, group_size, event_offset)
    brie_results.fdr = fdr
    if n_perm > 0:
        gain_perm = np.zeros((Ng, T, n_perm), dtype=np.float32)
        for (t, b), lg in lg_perm.items():
            gain_perm[:, t, b] = (lg_tests[t] if full else brie_results.loss_gene) - lg
        brie_results.ELBO_gain_perm = gain_perm
        _set_perm_outputs(brie_results)
    return brie_results


def _dist_info():
    """(torch.distributed, rank, world) -- world 1 when no process group is initialised."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist, dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return None, 0, 1


def _merge_shared(parts):
    """Merge event shards of ONE fit whose per-cell parameters and loss trace are shared (identical
    on every rank after the all-reduce): only per-event fields are concatenated."""
    out = parts[0]
    for r in parts[1:]:
        out.Ng += r.Ng
        out.loss_gene = np.append(out.loss_gene, r.loss_gene)
        out.cell_coeff = np.append(out.cell_coeff, r.cell_coeff, axis=1)
        for k in ('Psi', 'Psi95CI', 'Z_std', 'Z_loc'):
            setattr(out, k, np.append(getattr(out, k), getattr(r, k), axis=1))
        if out.intercept_mode.upper() != 'CELL':
            out.sigma = np.append(out.sigma, r.sigma, axis=1)
            out.intercept = np.append(out.intercept, r.intercept, axis=1)
        if hasattr(r, 'ELBO_gain'):
            for k in ('fdr', 'pval', 'ELBO_gain'):
                setattr(out, k, np.append(getattr(out, k), getattr(r, k), axis=0))
        if hasattr(r, 'ELBO_gain_perm'):
            for k in ('ELBO_gain_perm', 'pval_perm', 'fdr_perm'):
                setattr(out, k, np.append(getattr(out, k), getattr(r, k), axis=0))
        if hasattr(r, 'pval_wald'):
            _append_wald(out, r)
        if hasattr(r, 'pval_score'):
            _append_score(out, r)
        _append_groups(out, r)
    out.shape = (out.Nc, out.Ng)
    if hasattr(out, 'pval'):               # one fit => one multiple-testing scope over all events
        for i in range(out.fdr.shape[1]):
            out.fdr[:, i] = fdr_bh(out.pval[:, i])
    return out


def _fit_signature(Nc, Ng, Xc, LRT_index, layer_keys, n_gene, world, intercept, intercept_mode, pseudo_count,
                   sigma, base_mode, keyargs):
    """What has to be equal for checkpointed event chunks to belong to the same fit."""
    import hashlib
    kw = {k: (v if isinstance(v, (int, float, str, bool, type(None))) else repr(v))
          for k, v in sorted(keyargs.items()) if k not in ('device', 'verbose')}
    return dict(n_cells=int(Nc), n_events=int(Ng), n_gene=int(n_gene), world=int(world),
                Xc_sha1=hashlib.sha1(np.ascontiguousarray(Xc, dtype=np.float32).tobytes()).hexdigest(),
                LRT_index=[int(i) for i in LRT_index], layer_keys=list(layer_keys),
                intercept=None if intercept is None else float(intercept), intercept_mode=str(intercept_mode),
                pseudo_count=float(pseudo_count), sigma=None if sigma is None else float(sigma),
                base_mode=str(base_mode), fit=kw)


def _balanced_chunk(n_events, budget, n_gene):
    """Events per device chunk: whole convergence groups, at most `budget` events, and chunks of
    (nearly) equal size -- 10 000 events under a budget of 9 580 run as 2 x 5 000, not 9 580 + 420
    (a sliver of a chunk pays the full step count at a fraction of the bandwidth)."""
    budget = max(budget // n_gene, 1) * n_gene
    n_chunks = max(-(-n_events // budget), 1)
    groups = -(-n_events // n_gene)
    return max(-(-groups // n_chunks), 1) * n_gene


def _device_event_budget(Nc, n_models, n_layers, device=None, frac=0.7, reserve=0):
    """Events per device chunk so that counts, their packed codes, (1+T) model states and outputs fit in HBM,
    besides `reserve` bytes held for the whole fit (the score candidates and one block of the score pass)."""
    import torch
    free, _ = torch.cuda.mem_get_info(device)
    # + the step kernel's per-event scratch of two-step fits, approximated: statistic partials and a second loss row
    # (Kc <= 4: at most 8 floats per model and row chunk) at 256 cells per row chunk, the chunk size brie_fit_create
    # picks for fits large enough to be cut into device chunks; the first-step parameters (Kc + 2 floats per model
    # and event, not per cell) are left out
    per_event = Nc * 4 * (n_layers + 1 + 6 * n_models + 3 + 1 + n_models * 8 / 256) * 1.05
    return max(int(max(free - reserve, 0) * frac / per_event), 1)


def fitBRIE(adata, Xc=None, Xg=None, intercept=None, intercept_mode='gene',
            LRT_index=[], layer_keys=['isoform1', 'isoform2', 'ambiguous'],
            batch_size=500000, pseudo_count=0.01, sigma=None,
            base_mode='full', tau_prior=[3, 27], score_X=None, LRT_groups=None, wald_groups=None,
            score_groups=None, **keyargs):
    """Fit a BRIE model from AnnData with cell and/or gene features (model_wrap.py:202-314).

    `out_dir` (not in the reference): directory for `.npy` memory maps of the dense
    (cells, events) outputs Psi / Psi95CI / Z_std / Z_loc, written event chunk by event chunk
    (and rank by rank) -- for fits whose outputs exceed host RAM; default: RAM arrays.
    `out_keys` (not in the reference): which of ('Psi', 'Psi95CI', 'Z_std', 'Z_loc') to bring back from the
    device (default all four; brie-quant with --outDir drops Z_loc, which AnnData never stores).
    `resume` (not in the reference; needs `out_dir`): every finished event chunk is checkpointed
    under `out_dir`; with resume=True a re-run of the same fit (same data shape, design, seed and
    schedule) skips the chunks already there and returns what the uninterrupted fit would have.
    `n_perm` (not in the reference, default 0): permutation replicates per tested covariate, see
    fit_BRIE_matrix; `pval_perm` / `fdr_perm` are pooled over all events of the fit (every chunk and
    rank) and stored as varm['ELBO_gain_perm', 'pval_perm', 'fdr_perm'] with uns['brie_param']['n_perm'].
    `wald` (not in the reference, default False): Wald tests from the fitted posterior, see fit_BRIE_matrix;
    stored as varm['cell_coeff_se', 'pval_wald', 'fdr_wald'] (and varm['intercept_se'] in gene mode) with
    uns['brie_param']['wald'] and ['wald_columns']; fdr_wald is BH over all events of the fit.
    `score_X` (not in the reference, default None): (Nc, J) candidate cell covariates aligned with adata's cells,
    score-tested from the fitted posterior, see fit_BRIE_matrix; stored as varm['score_z', 'score_effect',
    'pval_score', 'fdr_score'] (Ng, J) with uns['brie_param']['score'] = J; fdr_score is BH over all events of the fit.
    `LRT_groups`, `wald_groups`, `score_groups` (not in the reference, default None): joint tests of groups of
    columns, see fit_BRIE_matrix; stored as varm['ELBO_gain_group', 'pval_group', 'fdr_group'],
    varm['wald_stat_group', 'pval_wald_group', 'fdr_wald_group'] and varm['score_stat_group', 'pval_score_group',
    'fdr_score_group'] with the groups in uns['brie_param']['LRT_groups' / 'wald_groups' / 'score_groups']; each FDR
    is BH over all events of the fit.

    Returns the BRIE_RV result and adds to `adata` exactly the keys the reference adds
    (obsm['Xc'], varm['cell_coeff'], varm['Xg'], obsm['gene_coeff'], varm|obsm['intercept',
    'sigma'], layers['Psi','Z_std','Psi_95CI'], uns['brie_losses'], var['loss_gene'],
    varm['fdr','pval','ELBO_gain'], uns['brie_param']).
    """
    if Xc is None:
        Xc = np.ones((adata.shape[0], 0), np.float32)
    if Xg is None:
        Xg = np.ones((adata.shape[1], 0), np.float32)
    if LRT_index is None:
        LRT_index = np.arange(Xc.shape[1])
    Nc, Ng = adata.shape
    n_models = 1 + len(LRT_index)
    n_perm = check_n_perm(keyargs.pop('n_perm', 0), len(LRT_index))
    if n_perm > 0:                         # (absent at 0: the fit signature of a checkpoint stays as it was)
        keyargs['n_perm'] = n_perm
    wald = check_wald(keyargs.pop('wald', False), keyargs.get('target', "ELBO"))
    if wald:                               # (likewise absent when False)
        keyargs['wald'] = True
    score_X = check_score_X(score_X, keyargs.get('target', "ELBO"), Nc)
    full = base_mode.upper() == 'FULL'
    base_cols = _base_columns(Xc.shape[1], LRT_index, full)
    LRT_groups = check_LRT_groups(LRT_groups, Xc.shape[1], base_cols, full, len(LRT_index), n_perm)
    wald_groups = check_wald_groups(wald_groups, Xc.shape[1], base_cols, keyargs.get('target', "ELBO"))
    score_groups = check_score_groups(score_groups, score_X, keyargs.get('target', "ELBO"))
    groups = dict(LRT_groups=LRT_groups, wald_groups=wald_groups, score_groups=score_groups)
    out_dir = keyargs.pop('out_dir', None)
    resume = keyargs.pop('resume', False)
    out_keys = tuple(keyargs.pop('out_keys', None) or BIG_KEYS)

    dist, rank, world = _dist_info()
    if (Xg is None or Xg.shape[1] == 0) and intercept_mode.upper() != 'CELL':   # :241
        # Events are independent here; the reference fits them in sequential batches of
        # _n_gene events (:242-258).  We keep _n_gene as the convergence group, fit as many
        # groups per launch as HBM holds, and give each GPU a contiguous range of groups.
        _n_gene = int(np.ceil(batch_size / Nc))
        lo, hi = event_shards(Ng, world, _n_gene)[rank]
        chunk = _device_event_budget(Nc, n_models, len(layer_keys), keyargs.get('device'),
                                     **({} if score_X is None else dict(reserve=score_X.nbytes + SCORE_BLOCK_BYTES)))
        chunk = _balanced_chunk(hi - lo, chunk, _n_gene)
        # finished chunks go straight into their column range of the output arrays (RAM, or
        # .npy memory maps under out_dir shared by all ranks) instead of np.append (:55-76)
        signature = _fit_signature(Nc, Ng, Xc, LRT_index, layer_keys, _n_gene, world, intercept, intercept_mode,
                                   pseudo_count, sigma, base_mode, keyargs) if out_dir is not None else None
        if signature is not None and score_X is not None:     # (absent without score_X)
            signature['score_X_sha1'] = hashlib.sha1(score_X.tobytes()).hexdigest()
        if signature is not None:                             # (each absent when None)
            signature.update({k: v for k, v in groups.items() if v is not None})
        store = LayerStore(Nc, Ng, out_dir, rank, world, dist, keys=out_keys, signature=signature, resume=resume)
        res_list = []
        pending = None                     # (sink, result) of the chunk whose layers are still on their way to the host

        def _land():
            nonlocal pending
            if pending is not None:
                _sink, _res = pending
                pending = None
                _t0 = time.perf_counter()
                _sink.wait()
                store.put(_sink.e0, _res)  # (checkpoint marker only after the chunk's layers are in the maps)
                if getattr(_res, 'timing', None) is not None:
                    _res.timing['store.put'] = time.perf_counter() - _t0

        for e0 in range(lo, hi, chunk):
            _done = store.load_chunk(e0, min(e0 + chunk, hi))
            if _done is not None:
                res_list.append(_done)
                print("[BRIE2] %d out %d genes done (resumed from %s)" % (min(e0 + chunk, hi) - lo, hi - lo, out_dir))
                continue
            _idx = slice(e0, min(e0 + chunk, hi))
            _count_layers = [adata.layers[_key][:, _idx] for _key in layer_keys]
            _effLen = adata.varm['effLen'][_idx, :] if 'effLen' in adata.varm else None
            # the previous chunk's layers land (and its checkpoint is written) while this chunk is fitted: at the
            # latest before this chunk's own output tensors are allocated, and also if this fit dies
            _sink = _ChunkSink(store, e0, before_outputs=_land)
            try:
                _ResVal = fit_BRIE_matrix(
                    _count_layers, Xc=Xc, Xg=Xg[_idx, :], effLen=_effLen,
                    intercept=intercept, intercept_mode=intercept_mode,
                    LRT_index=LRT_index, pseudo_count=pseudo_count, sigma=sigma,
                    base_mode=base_mode, tau_prior=tau_prior, group_size=_n_gene,
                    event_offset=e0, n_events_total=Ng, host_side_effect=False, out_sink=_sink, score_X=score_X,
                    **groups, **keyargs)
            finally:
                _land()
            pending = (_sink, _ResVal)
            res_list.append(_ResVal)
            print("[BRIE2] %d out %d genes done" % (min(e0 + chunk, hi) - lo, hi - lo))
        _land()
        timing_rank = {}                   # BRIE_TIMING diagnostics of THIS rank's chunks (the merged result sums all ranks)
        for _r in res_list:
            for k, v in (getattr(_r, 'timing', None) or {}).items():
                timing_rank[k] = timing_rank.get(k, 0.0) + v
        if world > 1:                      # per-event vectors: every rank gets all of them, in event order
            parts = [None] * world
            dist.all_gather_object(parts, res_list)
            res_list = [r for p in parts for r in p]
        ResVal = concate(res_list)
        ResVal.timing_rank = timing_rank
        for k, v in store.finish().items():
            setattr(ResVal, k, v)
    elif world > 1:
        # shared per-cell parameters: shard events, the library all-reduces the shared gradients
        # every step (engine.py / csrc/brie_comm.cu).  The dense (cells, events) outputs go into their
        # column range of the output arrays / memory maps; only per-event vectors are gathered.
        lo, hi = event_shards(Ng, world, 1)[rank]
        _idx = range(lo, hi)
        store = LayerStore(Nc, Ng, out_dir, rank, world, dist, keys=out_keys)
        _count_layers = [adata.layers[_key][:, _idx] for _key in layer_keys]
        _effLen = adata.varm['effLen'][_idx, :] if 'effLen' in adata.varm else None
        local = fit_BRIE_matrix(
            _count_layers, Xc=Xc, Xg=Xg[_idx, :], effLen=_effLen, intercept=intercept,
            intercept_mode=intercept_mode, LRT_index=LRT_index,
            pseudo_count=pseudo_count, sigma=sigma, base_mode=base_mode,
            tau_prior=tau_prior, event_offset=lo, n_events_total=Ng,
            dist_group=dist.group.WORLD, out_sink=_ChunkSink(store, lo, background=False), score_X=score_X,
            **groups, **keyargs)
        store.put(lo, local, checkpoint=False)
        parts = [None] * world
        dist.all_gather_object(parts, local)
        ResVal = _merge_shared(parts)
        for k, v in store.finish().items():
            setattr(ResVal, k, v)
    else:                                                           # :261-269
        _count_layers = [adata.layers[_key] for _key in layer_keys]
        _effLen = adata.varm['effLen'] if 'effLen' in adata.varm else None
        ResVal = fit_BRIE_matrix(
            _count_layers, Xc=Xc, Xg=Xg, effLen=_effLen, intercept=intercept,
            intercept_mode=intercept_mode, LRT_index=LRT_index,
            pseudo_count=pseudo_count, sigma=sigma, base_mode=base_mode,
            tau_prior=tau_prior, score_X=score_X, **groups, **keyargs)

    if n_perm > 0:                         # one pooled null over every event of the fit, the same on every rank
        _set_perm_outputs(ResVal)
    if wald:                               # one BH scope over every event of the fit
        _set_fdr_wald(ResVal)
    if score_X is not None:                # likewise
        _set_fdr_score(ResVal)
    _set_fdr_groups(ResVal)                # likewise, for each kind of group test

    # update adata (:271-311)
    if Xc.shape[0] > 0:
        adata.obsm['Xc'] = Xc
        adata.varm['cell_coeff'] = ResVal.cell_coeff.T
    if Xg.shape[1] > 0:
        adata.varm['Xg'] = Xg
        adata.obsm['gene_coeff'] = ResVal.gene_coeff
    if ResVal.intercept_mode == 'gene':
        adata.varm['intercept'] = ResVal.intercept.T
        adata.varm['sigma'] = ResVal.sigma.T
    elif ResVal.intercept_mode == 'cell':
        adata.obsm['intercept'] = ResVal.intercept
        adata.obsm['sigma'] = ResVal.sigma
    else:
        adata.varm['sigma'] = ResVal.sigma.T

    adata.layers['Psi'] = ResVal.Psi
    adata.layers['Z_std'] = ResVal.Z_std
    adata.layers['Psi_95CI'] = ResVal.Psi95CI

    adata.uns['brie_losses'] = ResVal.losses
    adata.var['loss_gene'] = ResVal.loss_gene

    if LRT_index is None or len(LRT_index) >= 1:
        adata.varm['fdr'] = ResVal.fdr
        adata.varm['pval'] = ResVal.pval
        adata.varm['ELBO_gain'] = ResVal.ELBO_gain
    if n_perm > 0:
        for k in ('ELBO_gain_perm', 'pval_perm', 'fdr_perm'):
            adata.varm[k] = getattr(ResVal, k)
    if wald:
        adata.varm['cell_coeff_se'] = ResVal.cell_coeff_se.T
        adata.varm['pval_wald'] = ResVal.pval_wald
        adata.varm['fdr_wald'] = ResVal.fdr_wald
        if hasattr(ResVal, 'intercept_se') and ResVal.intercept_mode == 'gene':
            adata.varm['intercept_se'] = ResVal.intercept_se.T
    if score_X is not None:
        for k in SCORE_KEYS:
            adata.varm[k] = getattr(ResVal, k)
    for (name, g), keys in zip(groups.items(), GROUP_KEYS):
        if g is not None:
            for k in keys:
                adata.varm[k] = getattr(ResVal, k)

    adata.uns['brie_param'] = {
        'LRT_index': LRT_index,
        'base_mode': base_mode,
        'intecept': intercept,
        'intercept_mode': intercept_mode,
        'sigma': sigma,
        'pseudo_count': pseudo_count,
        'layer_keys': layer_keys
    }
    if n_perm > 0:
        adata.uns['brie_param']['n_perm'] = n_perm
    if wald:
        adata.uns['brie_param']['wald'] = True
        adata.uns['brie_param']['wald_columns'] = list(ResVal.wald_columns)
    if score_X is not None:
        adata.uns['brie_param']['score'] = int(score_X.shape[1])
    for name, g in groups.items():
        if g is not None:
            adata.uns['brie_param'][name] = g
    return ResVal
