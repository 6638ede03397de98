"""Models of one shared-parameter engine that stop at different extension rounds.

A fit with per-cell parameters (Kg > 0 or intercept_mode 'cell') runs all its models in one engine with one
convergence group per model.  Once a model's stop rule fires, the engine keeps stepping the others in place with
that model's `active` flags all zero: from then on the model must not change at all -- not its per-event state, and
not the per-cell parameters (Wg, the per-cell intercept / sigma_log) that no event of it updates any more -- and the
models still stepping must not notice.

- test_frozen_model_stays_put: two engines from identical inputs; after a warm-up one steps everything, the other
  the same steps with one model frozen.  Exact: the frozen model equals its warm-up snapshot bit for bit, the others
  equal the first engine's bit for bit.
- test_staggered_lrt_matches_oracle / test_staggered_cell_mode_permutations_match_oracle: fit_BRIE_matrix end to
  end against the oracle on a schedule under which the models of one engine stop at different rounds, chosen so that
  no stop-rule comparison sits near epsilon_conv.
"""
import numpy as np
import pytest

import oracle.brie2_oracle as ob
from oracle.brie2_oracle import add_pseudo_count, oracle_fit_matrix

from util import bar_report, device_eps_provider, make_lrt_problem, make_problem

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _patched_oracle(seed, Nc, fn):
    """Run fn() with OracleBRIE2 drawing the device's noise (per model id / column offset)."""
    orig = ob.OracleBRIE2.eps
    ob.OracleBRIE2.eps = lambda self, phase, step, S: device_eps_provider(
        seed, self.model_id, Nc, self.Ng, self.col_offset)(phase, step, S)
    try:
        return fn()
    finally:
        ob.OracleBRIE2.eps = orig


# ---------------------------------------------------------------------------------------------- exact freeze test
NC, NG, S, SEED = 549, 203, 3, 17      # 64 rows per CTA: 9 row chunks, the last ragged; 2 column tiles of 128 events
WARM, K, LR = 6, 4, 0.01

# (intercept mode, Kc, Kg, target): every family with parameters shared across events
FAMILIES = {
    'gene-2-3': ('gene', 2, 3, "ELBO"),           # Kg 3 -> 4
    'gene-1-8': ('gene', 1, 8, "ELBO"),
    'cell-0-0': ('cell', 0, 0, "ELBO"),
    'cell-1-2': ('cell', 1, 2, "ELBO"),
    'cell-8-4': ('cell', 8, 4, "ELBO"),           # two rows per iteration
    'wide-gene-3-20': ('gene', 3, 20, "ELBO"),    # Kg > 8: contractions as GEMMs around the fused kernel
    'wide-cell-24-0': ('cell', 24, 0, "ELBO"),
    'margin-gene-1-3': ('gene', 1, 3, "marginLik"),
    'margin-cell-1-0': ('cell', 1, 0, "marginLik"),
}


def _engine(fam):
    from brie_b200.engine import FitEngine
    mode, Kc, Kg, target = FAMILIES[fam]
    data, effLen, Xc, Xg = make_problem(NC, NG, Kc, Kg, True, 3, seed=6, design_seed=2)
    add_pseudo_count(data, np.float32(0.01))
    # LRT refits drop one covariate each; with fewer than two the three models differ by their noise only
    masks = ([list(range(Kc))] + [[k for k in range(Kc) if k != i] for i in range(2)] if Kc >= 2
             else [list(range(Kc))] * 3)
    eng = FitEngine(data, effLen=effLen, Xc=Xc, Xg=Xg if Kg else None, masks=masks, model_ids=[0, 1, 2],
                    intercept_mode=mode, MC_size=S, seed=SEED, trace_cap=K, target=target)
    assert eng.shared and eng.n_groups == 1 and eng.sizes.rows_per_cta == 64
    assert eng.sizes.n_row_chunks == 9 and (eng.wide or eng.sizes.n_col_tiles >= 2)
    return eng


def _model_state(eng, m):
    """Every array the step path may write for model m, as host copies."""
    M, Kc, ld, Nc = eng.M, eng.Kc, eng.ld, eng.Nc
    n_ev = 2 * M * (Kc + 2) * ld
    mom_ev = eng.adam_small[:n_ev].view(2, M, Kc + 2, ld)
    mom_cell = eng.adam_small[n_ev:n_ev + 2 * M * Nc * (eng.Kg + 2)].view(2, M, Nc, eng.Kg + 2)
    torch.cuda.synchronize()
    return {'Z_loc': eng.Z_loc[m], 'Z_std_log': eng.Z_std_log[m], 'adam_Z': eng.adam_Z[:, m], 'Wc': eng.Wc[m],
            'Wg': eng.Wg[m], 'intercept': eng.intercept[m], 'sigma_log': eng.sigma_log[m],
            'adam_small (per event)': mom_ev[:, m], 'adam_small (per cell)': mom_cell[:, m],
            'loss_trace': eng.loss_trace[m]}


def _diffs(a, b):
    """Names of the arrays that differ, with the largest absolute difference of each."""
    out = []
    for k in a:
        x, y = a[k].cpu(), b[k].cpu()
        if not torch.equal(x, y):
            out.append("%s: max |drift| %.3g" % (k, float((x.double() - y.double()).abs().max())))
    return out


@pytest.mark.parametrize("frozen", [0, 2], ids=["first", "last"])
@pytest.mark.parametrize("fam", list(FAMILIES))
def test_frozen_model_stays_put(monkeypatch, fam, frozen):
    monkeypatch.setenv("BRIE_ROWS_PER_CTA", "64")
    a, b = _engine(fam), _engine(fam)
    for e in (a, b):
        e.init_params()
        e.begin_stage(LR)
        e.run_steps(WARM)
    snap = {k: v.clone() for k, v in _model_state(b, frozen).items()}
    act = np.ones((b.M, 1), bool)
    act[frozen] = False
    b.set_active_groups(act)
    a.run_steps(K, 0)
    b.run_steps(K, 0)
    bad = ["frozen model %d %s" % (frozen, d) for d in _diffs(_model_state(b, frozen), snap)]
    for m in range(b.M):
        if m != frozen:
            bad += ["model %d differs from the all-active engine: %s" % (m, d)
                    for d in _diffs(_model_state(b, m), _model_state(a, m))]
    assert a.step_counters() == b.step_counters() == (WARM + K, WARM + K)
    assert not bad, "\n".join(bad)


def test_model_mask_refused_inside_a_split_step():
    """brie_fit_set_model_mask between the two halves of a step (brie_fit_step_phase) would change which models the
    per-cell update steps after the reduce: refused, and the step then completes."""
    from brie_b200 import _lib
    from brie_b200.engine import FitEngine
    data, effLen, Xc, Xg = make_problem(64, 40, 1, 2, True, 3, seed=6)
    eng = FitEngine(data, effLen=effLen, Xc=Xc, Xg=Xg, masks=[[0], [0]], intercept_mode='cell', trace_cap=1)
    eng.init_params()
    eng.begin_stage(LR)
    lib, st = eng.lib, eng._stream()
    _lib.check(lib.brie_fit_step_phase(eng.h, 0, -1, st))
    assert lib.brie_fit_set_model_mask(eng.h, 1) == -1 and b"split step" in lib.brie_last_error()
    _lib.check(lib.brie_fit_step_phase(eng.h, 1, -1, st))
    _lib.check(lib.brie_fit_set_model_mask(eng.h, 1))
    assert eng.step_counters() == (1, 1)


# ---------------------------------------------------------------------------------------------- oracle, staggered stops
def _two_covariates(Nc, Ng, seed):
    """make_lrt_problem (planted effects on covariate 0) with a second, pure-noise covariate and 3 gene features."""
    data, effLen, x, _ = make_lrt_problem(Nc, Ng, seed=seed)
    rng = np.random.default_rng(seed + 100)
    Xc = np.concatenate([x, rng.standard_normal((Nc, 1)).astype(np.float32)], axis=1)
    Xg = rng.standard_normal((Ng, 3)).astype(np.float32)
    return data, effLen, Xc, Xg


def _stop_margins(losses, min_iter, add_iter, max_iter, epsilon_conv):
    """Signed distance from epsilon_conv of every stop-rule comparison (model_TFProb.py:250-251) that decided
    something on the oracle's loss trace (the last stage's trace, then one extension round per comparison): those
    taken below max_iter."""
    d1 = int(min(50, add_iter / 2))
    d2 = 2 * d1
    out = []
    n, n_iter = int(min_iter / 6), min_iter
    while n <= len(losses) and n_iter < max_iter:
        w = losses[:n]
        prev, last = w[-d2:-d1], w[-d1:]
        if len(prev) and len(last):
            out.append(float(np.mean(prev, dtype=np.float32) - np.mean(last, dtype=np.float32)) - epsilon_conv)
        n += add_iter
        n_iter += add_iter
    return out


MARGIN = 0.5    # the float32 and float64 oracles' comparisons differ by ~0.02 on these problems


def _check_schedule(models, kw):
    """The schedule tests something (two models stop at different rounds) and no stop decision is close."""
    n_iter = [m.n_iter for m in models]
    assert len(set(n_iter)) >= 2, "want models that stop at different rounds, got n_iter %s" % n_iter
    margins = [abs(x) for m in models
               for x in _stop_margins(m.losses, kw['min_iter'], kw['add_iter'], kw['max_iter'], kw['epsilon_conv'])]
    print("oracle n_iter %s, smallest stop-rule margin %.3f" % (n_iter, min(margins)))
    assert min(margins) > MARGIN


def test_staggered_lrt_matches_oracle():
    """Gene mode with gene features and two cell covariates, every covariate tested: base + 2 refits in one shared
    engine, stopping at 1200, 960 and 1080 steps."""
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng, seed = 60, 20, 21
    data, effLen, Xc, Xg = _two_covariates(Nc, Ng, seed=2)
    kw = dict(min_iter=360, add_iter=120, max_iter=1200, epsilon_conv=2.0, MC_size=3, n_eval=40)
    fit = lambda dt: oracle_fit_matrix([x.copy() for x in data], Xc=Xc, Xg=Xg, effLen=effLen, intercept=None,
                                       intercept_mode='gene', LRT_index=None, dtype=dt, seed=seed, **kw)
    ref = _patched_oracle(seed, Nc, lambda: fit(np.float32))
    _check_schedule([ref.model] + ref.tests, kw)
    ref64 = _patched_oracle(seed, Nc, lambda: fit(np.float64))
    assert list(ref64.n_iter) == list(ref.n_iter)
    res = fit_BRIE_matrix([x.copy() for x in data], Xc=Xc, Xg=Xg, effLen=effLen, intercept=None,
                          intercept_mode='gene', LRT_index=None, seed=seed, **kw)
    assert list(res.n_iter[:, 0]) == list(ref.n_iter)
    # Psi: the bars of test_gpu_parity.test_full_fit_with_lrt_matches_oracle
    dpsi = np.abs(res.Psi - ref.Psi)
    envelope = np.abs(ref.Psi - ref64.Psi)
    n_psi = bar_report("staggered Psi", dpsi, 1e-3, envelope)
    assert n_psi <= max(5, 2 * int((envelope > 1e-3).sum()))
    assert np.quantile(dpsi, 0.95) < 1e-3 and np.median(dpsi) < 1e-4
    assert dpsi.max() <= max(1e-3, envelope.max())
    assert np.abs(res.Psi - ref64.Psi).max() <= max(1e-3, 2 * envelope.max())
    # the shared parameters of the base model
    dwg = np.abs(res.gene_coeff - ref.gene_coeff).max()
    env_wg = np.abs(ref.gene_coeff - ref64.gene_coeff).max()
    print("gene_coeff: max %.2e | f32-vs-f64 oracle envelope %.2e" % (dwg, env_wg))
    assert dwg < max(5e-3, 2 * env_wg)
    lg_bar = 1e-4 * np.abs(ref.loss_gene).max()
    assert np.abs(res.loss_gene - ref.loss_gene).max() <= lg_bar
    # the refits, which stop first, reach the outputs through ELBO_gain = loss_gene(refit) - loss_gene(base)
    for i, mt in enumerate(ref.tests):
        assert np.abs(res.ELBO_gain[:, i] + res.loss_gene - mt.loss_gene).max() <= lg_bar, "refit %d loss_gene" % i
    # ELBO_gain: 1e-3 relative where |gain| > 1.5 and 1e-2 absolute, or as close as float32 itself gets when its own
    # oracle is farther from the float64 one (after 1200 steps here: ~3e-3 relative, ~1.2e-2 absolute)
    big = np.abs(ref.ELBO_gain) > 1.5
    dg, eg = np.abs(res.ELBO_gain - ref.ELBO_gain), np.abs(ref.ELBO_gain - ref64.ELBO_gain)
    rel, env_rel = dg[big] / np.abs(ref.ELBO_gain)[big], eg[big] / np.abs(ref64.ELBO_gain)[big]
    bar_report("staggered ELBO_gain (relative, |gain| > 1.5)", rel, 1e-3, env_rel)
    print("ELBO_gain: max abs %.2e | f32-vs-f64 oracle envelope %.2e" % (dg.max(), eg.max()))
    assert rel.max(initial=0) <= max(1e-3, 2 * env_rel.max(initial=0))
    assert dg.max() < max(1e-2, 2 * eg.max())
    assert ((res.fdr < 0.05) == (ref.fdr < 0.05)).all()


def test_staggered_cell_mode_permutations_match_oracle(monkeypatch):
    """intercept_mode 'cell' with two tested covariates and n_perm 2: the four permuted full models run two to a
    cell-mode engine, and within each engine they stop at different rounds.  Each one's n_iter and loss_gene
    against an oracle fit of its permuted design."""
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.models import model_wrap as mw
    Nc, Ng, seed, T, B = 60, 20, 5, 2, 2
    data, effLen, Xc, _ = _two_covariates(Nc, Ng, seed=3)
    kw = dict(min_iter=360, add_iter=120, max_iter=1200, epsilon_conv=1.0, MC_size=3, n_eval=40)
    d = [np.array(x, np.float32) for x in data]
    add_pseudo_count(d, np.float32(0.01))

    def run_oracle():
        out = {}
        for t in range(T):
            for b in range(B):
                Xp = Xc.copy()
                Xp[:, t] = Xc[mw.perm_indices(seed, t, b, Nc), t]
                m = ob.OracleBRIE2(Nc, Ng, 2, 0, effLen, None, 'cell', None, dtype=np.float32, seed=seed,
                                   model_id=mw.perm_model_id(t, b, T, B))
                m.fit(d, Xc=Xp, Xg=np.ones((Ng, 0), np.float32), **kw)
                out[mw.perm_model_id(t, b, T, B)] = m
        return out
    ref = _patched_oracle(seed, Nc, run_oracle)
    _check_schedule(list(ref.values()), kw)

    engines, real = [], mw.FitEngine

    def spy(*a, **k):
        engines.append(real(*a, **k))
        return engines[-1]
    monkeypatch.setattr(mw, "FitEngine", spy)
    fit_BRIE_matrix([x.copy() for x in data], Xc=Xc, effLen=effLen, intercept=None, intercept_mode='cell',
                    LRT_index=None, seed=seed, n_perm=B, **kw)
    perm = [e for e in engines if min(e.model_ids) > T]
    assert [(e.model_ids, e.cell_mode) for e in perm] == [([3, 4], True), ([5, 6], True)]
    staggered = 0
    for e in perm:
        staggered += len(set(int(ref[mid].n_iter) for mid in e.model_ids)) > 1
        for j, mid in enumerate(e.model_ids):
            assert int(e.n_iter[j, 0]) == ref[mid].n_iter, "model %d" % mid
            lg, want = e.loss_gene[j].cpu().numpy(), ref[mid].loss_gene
            err = np.abs(lg - want).max() / np.abs(want).max()
            print("permuted model %d: n_iter %d, loss_gene max relative error %.2e" % (mid, ref[mid].n_iter, err))
            assert err <= 1e-4, "model %d" % mid
    assert staggered >= 1, "no permuted engine whose models stop at different rounds"
