"""The fused step kernel against the float64 oracle at the row-chunk sizes production fits run with.

brie_fit_create sizes the row chunks from the problem: a fit as small as the other parity tests gets 8 rows per
CTA, at most one loop iteration per warp, so the two-stage row ring never cycles, row constants are never reused
two iterations on, and no warp runs several iterations and then a ragged last one.  Every production-size fit
does all of that (256 rows per CTA on the headline).  Here BRIE_ROWS_PER_CTA forces 64 and 256 rows on an odd cell
count, 549 = 2 x 256 + 37 = 8 x 64 + 37, so the last chunk is ragged and odd (the two-rows-per-iteration kernels
then end on an iteration whose second row does not exist), and 203 events end the last column tile inside a lane
vector for 128- and 64-event tiles alike.

One step is taken from a warmed-up state (6 steps at lr 0.01: sigma away from 1, the intercept trained away from
its init) and compared with the oracle on the device's own snapshot and noise, for every instantiation family of
the step kernel, both count forms and both loss-trace variants:
- the new Adam moments of every trained variable, m' = 0.9 m + 0.1 g and v' = 0.999 v + 0.001 g^2 with the
  oracle's g (the first-step bar of test_gpu_parity on g, carried through 0.1 g and 0.001 g^2);
- the per-event loss trace against the oracle's loss_gene;
- Z_loc / Z_std_log after the update, recomputed in float64 (keras Adam, +-9 clip on Z_loc) from the snapshot and
  the device's new moments: phase C's arithmetic without Adam's 1/sqrt(v) amplification of gradient rounding.
"""
import functools

import numpy as np
import pytest

from oracle import philox_np as px
from oracle.brie2_oracle import OracleBRIE2, add_pseudo_count

from util import device_eps_provider, make_problem

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

NC, NG, S, SEED = 549, 203, 3, 17
WARM, LR = 6, 0.01
DEFAULT_ROWS = 8            # what brie_fit_create picks for every family at NC x NG
ROWS = [None, 64, 256]      # None: the library's own choice

# (intercept mode, Kc, Kg, effLen, layers); the device pads Kc to 0/1/2/4/8/16 and Kg to 0/4/8, wider is the wide form
FAMILIES = {
    'gene-0-0': ('gene', 0, 0, True, 3),
    'gene-1-0': ('gene', 1, 0, True, 3),
    'gene-2-0': ('gene', 2, 0, False, 2),
    'gene-3-0': ('gene', 3, 0, True, 3),      # Kc 4
    'gene-7-0': ('gene', 7, 0, True, 3),      # Kc 8
    'gene-11-0': ('gene', 11, 0, True, 3),    # Kc 16: two rows per iteration
    'gene-1-3': ('gene', 1, 3, True, 3),      # Kg 4
    'gene-2-8': ('gene', 2, 8, True, 2),
    'gene-8-4': ('gene', 8, 4, True, 3),      # two rows per iteration
    'gene-6-7': ('gene', 6, 7, True, 3),      # Kc 8, Kg 8: two rows per iteration
    'gene-16-3': ('gene', 16, 3, True, 3),    # two events per lane, one row per iteration
    'None-11-0': ('None', 11, 0, True, 3),    # intercept fixed at 0; two rows per iteration
    'cell-0-0': ('cell', 0, 0, True, 3),
    'cell-1-2': ('cell', 1, 2, False, 2),     # Kg 4
    'cell-0-8': ('cell', 0, 8, True, 3),
    'cell-8-4': ('cell', 8, 4, True, 3),      # two rows per iteration
    'cell-9-5': ('cell', 9, 5, False, 2),     # Kc 16, Kg 8
    'gene-24-0': ('gene', 24, 0, True, 3),    # wide form
    'cell-3-20': ('cell', 3, 20, True, 3),    # wide form
}
TWO_ROW = ['gene-11-0', 'gene-8-4', 'gene-6-7', 'None-11-0', 'cell-8-4']   # step_rpi(KC, KG) == 2


@functools.lru_cache(maxsize=None)
def _problem(Kc, Kg, eff, n_layers):
    data, effLen, Xc, Xg = make_problem(NC, NG, Kc, Kg, eff, n_layers, seed=6, design_seed=2)
    add_pseudo_count(data, np.float32(0.01))
    return data, effLen, Xc, Xg


def _engine(monkeypatch, fam, rows, count_format=None, two_models=False, n_cells=NC):
    from brie_b200.engine import FitEngine
    mode, Kc, Kg, eff, n_layers = FAMILIES[fam]
    data, effLen, Xc, Xg = _problem(Kc, Kg, eff, n_layers)
    data, Xc = [x[:n_cells] for x in data], Xc[:n_cells]
    if rows is None:
        monkeypatch.delenv("BRIE_ROWS_PER_CTA", raising=False)
    else:
        monkeypatch.setenv("BRIE_ROWS_PER_CTA", str(rows))
    masks = [list(range(Kc)), [k for k in range(Kc) if k != 1]] if two_models else None
    eng = FitEngine(data, effLen=effLen, Xc=Xc, Xg=Xg if Kg else None, masks=masks,
                    intercept=0 if mode == 'None' else None, intercept_mode=mode, MC_size=S, seed=SEED, trace_cap=4,
                    count_format=count_format)
    assert eng.sizes.rows_per_cta == (DEFAULT_ROWS if rows is None else rows)
    assert eng.count_format == ('f32' if count_format == 'f32' else 'code8')
    return eng, data, effLen, Xc, Xg


def _warm_up(eng):
    eng.init_params()
    eng.begin_stage(LR)
    eng.run_steps(WARM)
    assert eng.step_counters() == (WARM, WARM)     # Adam step count, RNG step word of the next step


def _snapshot(eng):
    names = ('Z_loc', 'Z_std_log', 'adam_Z', 'adam_small', 'Wc', 'Wg', 'intercept', 'sigma_log')
    torch.cuda.synchronize()
    return {k: getattr(eng, k).cpu().numpy() for k in names}


def _oracle(eng, snap, m, data, effLen, Xc, Xg):
    """float64 oracle of model m on the device state `snap` (sigma_log taken as stored, not through exp / log)."""
    Nc = eng.Nc
    mask = eng.masks[m]
    f64 = lambda x: np.asarray(x, np.float64)
    om = OracleBRIE2(Nc, NG, len(mask), eng.Kg_real, effLen, eng.intercept_const, 'cell' if eng.cell_mode else 'gene',
                     None, dtype=np.float64, seed=SEED, model_id=eng.model_ids[m])
    n, shape = (Nc, (Nc, 1)) if eng.cell_mode else (NG, (1, NG))
    om.p['Z_loc'] = f64(snap['Z_loc'][m, :, :NG])
    om.p['Z_std_log'] = f64(snap['Z_std_log'][m, :, :NG])
    om.p['Wc_loc'] = f64(snap['Wc'][m, :len(mask), :NG])
    om.p['Wg_loc'] = f64(snap['Wg'][m, :, :eng.Kg_real])
    om.p['intercept'] = f64(snap['intercept'][m, :n]).reshape(shape)
    om.p['sigma_log'] = f64(snap['sigma_log'][m, :n]).reshape(shape)
    om.Xc = f64(Xc[:, mask])
    om.Xg = f64(Xg) if eng.Kg_real else None
    return om


def _moments(eng, snap, m):
    """{variable: (first moment, second moment)} of model m in the oracle's shapes.  adam_small holds the per-event
    moments (2, M, Kc + 2, ld) -- rows Wc, intercept, sigma_log -- then the per-cell ones (2, M, Nc, Kg + 2) -- Wg,
    intercept, sigma_log (test_gpu_parity.test_first_step_loss_and_gradients)."""
    M, Nc, KC, KG, ld = eng.M, eng.Nc, eng.Kc, eng.Kg, eng.ld
    n_ev = 2 * M * (KC + 2) * ld
    ev = snap['adam_small'][:n_ev].reshape(2, M, KC + 2, ld)[:, m].astype(np.float64)
    cell = snap['adam_small'][n_ev:n_ev + 2 * M * Nc * (KG + 2)].reshape(2, M, Nc, KG + 2)[:, m].astype(np.float64)
    aZ = snap['adam_Z'][:, m, :, :NG].astype(np.float64)
    out = {'Z_loc': (aZ[0], aZ[1]), 'Z_std_log': (aZ[2], aZ[3]),
           'Wc_loc': (ev[0, :len(eng.masks[m]), :NG], ev[1, :len(eng.masks[m]), :NG]),
           'Wg_loc': (cell[0, :, :eng.Kg_real], cell[1, :, :eng.Kg_real])}
    if eng.cell_mode:
        out['intercept'] = (cell[0, :, KG:KG + 1], cell[1, :, KG:KG + 1])
        out['sigma_log'] = (cell[0, :, KG + 1:KG + 2], cell[1, :, KG + 1:KG + 2])
    else:
        out['intercept'] = (ev[0, KC:KC + 1, :NG], ev[1, KC:KC + 1, :NG])
        out['sigma_log'] = (ev[0, KC + 1:KC + 2, :NG], ev[1, KC + 1:KC + 2, :NG])
    return out


def _adam_alpha(lr, t):
    """The step size brie_fit_step_phase hands the kernels: float32 of the double-precision bias correction."""
    return float(np.float32(float(np.float32(lr)) * np.sqrt(1.0 - 0.999 ** t) / (1.0 - 0.9 ** t)))


def _check_one_step(monkeypatch, fam, rows, count_format, loss, two_models=False, n_cells=NC):
    eng, data, effLen, Xc, Xg = _engine(monkeypatch, fam, rows, count_format, two_models, n_cells)
    _warm_up(eng)
    old = _snapshot(eng)
    eng.run_steps(1, 0 if loss else -1)
    new = _snapshot(eng)
    alpha = _adam_alpha(LR, WARM + 1)
    bad = []
    for m in range(eng.M):
        om = _oracle(eng, old, m, data, effLen, Xc, Xg)
        eps = device_eps_provider(SEED, eng.model_ids[m], n_cells, NG)(px.PHASE_TRAIN, WARM, S)
        ref_loss, loss_gene, grads = om.loss_and_grads(data, eps)
        mo, mn = _moments(eng, old, m), _moments(eng, new, m)
        for name in om.trainable():
            g = grads[name]
            scale = max(np.abs(g).max(initial=0), 1.0)
            m_ref = 0.9 * mo[name][0] + 0.1 * g
            v_ref = 0.999 * mo[name][1] + 0.001 * g * g
            e1 = np.abs(mn[name][0] - m_ref).max(initial=0) / scale
            e2 = np.abs(mn[name][1] - v_ref).max(initial=0)
            bar2 = 1e-6 * np.abs(v_ref).max(initial=0) + 4e-7 * scale * scale
            if e1 > 2e-5:
                bad.append("model %d %s first moment: %.3g x max(|g|, 1) > 2e-5" % (m, name, e1))
            if e2 > bar2:
                bad.append("model %d %s second moment: %.3g > %.3g" % (m, name, e2, bar2))
        if loss:
            tr = eng.loss_trace[m, 0, :NG].cpu().numpy().astype(np.float64)
            e = np.abs(tr - loss_gene).max() / np.abs(loss_gene).max()
            if e > 1e-4:
                bad.append("model %d loss trace: %.3g x max|loss_gene| > 1e-4 (%d events off)" % (
                    m, e, int((np.abs(tr - loss_gene) > 1e-4 * np.abs(loss_gene).max()).sum())))
            e = abs(tr.sum() - ref_loss) / abs(ref_loss)
            if e > 1e-5:
                bad.append("model %d loss trace sum: relative %.3g > 1e-5" % (m, e))
        for name, (im, iv) in (('Z_loc', (0, 1)), ('Z_std_log', (2, 3))):
            mom1 = new['adam_Z'][im, m, :, :NG].astype(np.float64)
            mom2 = new['adam_Z'][iv, m, :, :NG].astype(np.float64)
            x = old[name][m, :, :NG].astype(np.float64) - mom1 * alpha / (np.sqrt(mom2) + 1e-7)
            if name == 'Z_loc':
                x = np.clip(x, -9.0, 9.0)
            bar = 2.0 * np.spacing(np.abs(x).astype(np.float32)).astype(np.float64) + 1e-5 * LR
            e = np.abs(new[name][m, :, :NG] - x) - bar
            if e.max() > 0:
                bad.append("model %d %s after the update: %d elements off, worst by %.3g" % (
                    m, name, int((e > 0).sum()), e.max()))
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("loss", [True, False], ids=["trace", "notrace"])
@pytest.mark.parametrize("count_format", [None, 'f32'], ids=["code8", "f32"])
@pytest.mark.parametrize("rows", ROWS, ids=lambda r: "rows%s" % (r or "default"))
@pytest.mark.parametrize("fam", list(FAMILIES))
def test_step_matches_oracle_at_chunk_size(monkeypatch, fam, rows, count_format, loss):
    _check_one_step(monkeypatch, fam, rows, count_format, loss)


@pytest.mark.parametrize("rows", ROWS, ids=lambda r: "rows%s" % (r or "default"))
@pytest.mark.parametrize("fam", TWO_ROW)
def test_two_row_step_with_refit_model_matches_oracle(monkeypatch, fam, rows):
    """The two-rows-per-iteration kernels with a second model (all covariates but column 1, RNG model word 1), as an
    LRT refit runs: each model against its own oracle and noise."""
    _check_one_step(monkeypatch, fam, rows, None, True, two_models=True)


@pytest.mark.parametrize("n_cells", [NC - 1, NC])
def test_two_row_kernel_odd_last_chunk(monkeypatch, n_cells):
    """Kc 16 in gene mode (two rows per loop iteration) at 64 rows per CTA: the last chunk holds 36 rows with 548
    cells and 37 with 549.  With 37 the last iteration of its warp 2 takes row 36 and a row 37 that does not exist;
    that row is zero-filled (mu = 0, log s = 0, prior mean = the intercept) and must add nothing to the per-event
    intercept and sigma_log gradients or the loss trace."""
    _check_one_step(monkeypatch, 'gene-11-0', 64, None, True, n_cells=n_cells)


N_EVAL = 40   # more evaluations than lanes: eval_item's `it += 32` loop runs twice


@pytest.mark.parametrize("S_eval", [1, 3])
@pytest.mark.parametrize("rows", [None, 256], ids=lambda r: "rows%s" % (r or "default"))
@pytest.mark.parametrize("fam", list(FAMILIES))
def test_loss_gene_eval_matches_oracle_at_chunk_size(monkeypatch, fam, rows, S_eval):
    """eval_loss_kernel (loss_gene, which feeds ELBO_gain) on a warmed-up state, two models where the family has
    two covariates to drop one of; S_eval = 3 takes the partial last group of four normals."""
    two = FAMILIES[fam][1] >= 2
    eng, data, effLen, Xc, Xg = _engine(monkeypatch, fam, rows, two_models=two)
    _warm_up(eng)
    lg = eng.eval_loss_gene(N_EVAL, S_eval).cpu().numpy()
    snap = _snapshot(eng)
    for m in range(eng.M):
        om = _oracle(eng, snap, m, data, effLen, Xc, Xg)
        epsf = device_eps_provider(SEED, eng.model_ids[m], NC, NG)
        ref = np.zeros(NG)
        for it in range(N_EVAL):
            ref += om.loss_and_grads(data, epsf(px.PHASE_EVAL, it, S_eval), want_grads=False)[1]
        ref /= N_EVAL
        assert np.abs(lg[m] - ref).max() <= 2e-5 * np.abs(ref).max(), "model %d" % m
