"""GPU tests of the reference-facing API: fitBRIE's event batches as convergence groups,
the BRIE2 class protocol, the brie-quant driver end to end (BASELINE config C1 style)."""
import os

import numpy as np
import pytest

import oracle.brie2_oracle as ob
from oracle.brie2_oracle import oracle_fit_matrix
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


def test_fitBRIE_groups_match_sequential_reference_batches():
    """fitBRIE fits all events in one engine but stops each reference batch (ceil(batch_size/Nc)
    events, model_wrap.py:241-258) independently -- compare with the oracle fitted batch by batch."""
    from brie_b200.models import fitBRIE
    from brie_b200.utils.anndata_lite import AnnDataLite
    Nc, Ng, seed = 100, 70, 4
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=3)
    ad = AnnDataLite(X=data[0] + data[1] + data[2],
                     layers={'isoform1': data[0].copy(), 'isoform2': data[1].copy(), 'ambiguous': data[2].copy()},
                     varm={'effLen': effLen})
    kw = dict(min_iter=600, max_iter=2100, add_iter=500, MC_size=2, n_eval=20)
    batch_size = 100 * 30                                  # -> 30 events per batch: groups of 30, 30, 10
    res = fitBRIE(ad, Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=batch_size, seed=seed, **kw)
    assert res.n_iter.shape == (2, 3)

    def run_oracle():
        out = []
        for e0 in range(0, Ng, 30):
            sl = slice(e0, min(e0 + 30, Ng))
            out.append(oracle_fit_matrix([x[:, sl].copy() for x in data], Xc=Xc, effLen=effLen[sl], LRT_index=None,
                                         intercept_mode='gene', dtype=np.float32, seed=seed, col_offset=e0, **kw))
        return out
    refs = _patched_oracle(seed, Nc, run_oracle)
    for gi, r in enumerate(refs):
        assert list(res.n_iter[:, gi]) == list(r.n_iter), "group %d step counts" % gi
    print("n_iter per (model, group):", res.n_iter.tolist())
    assert len(set(res.n_iter.reshape(-1).tolist())) > 1, "want groups that stop at different times"
    Psi = np.concatenate([r.Psi for r in refs], axis=1)
    gain = np.concatenate([r.ELBO_gain for r in refs], axis=0)
    fdr = np.concatenate([r.fdr for r in refs], axis=0)              # BH per batch, as the reference
    assert np.array_equal(res.fdr < 0.05, fdr < 0.05) and np.abs(res.fdr - fdr).max() < 5e-3
    n_psi = bar_report("fitBRIE groups Psi", np.abs(res.Psi - Psi), 1e-3)
    assert n_psi <= 0.01 * Psi.size and np.quantile(np.abs(res.Psi - Psi), 0.99) < 1e-3
    big = np.abs(gain) > 1.5
    bar_report("fitBRIE groups ELBO_gain (relative, |gain| > 1.5)", (np.abs(res.ELBO_gain - gain) / np.maximum(np.abs(gain), 1e-30))[big], 1e-3)
    assert (np.abs(res.ELBO_gain - gain)[big] / np.abs(gain)[big]).max() < 1e-3
    # uns['brie_losses'] = per-batch traces appended end to end (model_wrap.py:61)
    want = np.concatenate([r.losses for r in refs])
    assert ad.uns['brie_losses'].shape == want.shape
    assert np.abs(ad.uns['brie_losses'] - want).max() <= 1e-4 * np.abs(want).max()
    # AnnData outputs (model_wrap.py:271-311)
    assert ad.layers['Psi'].shape == (Nc, Ng) and ad.layers['Psi_95CI'].shape == (Nc, Ng)
    assert ad.layers['Z_std'].shape == (Nc, Ng)
    assert ad.varm['cell_coeff'].shape == (Ng, 1) and ad.varm['intercept'].shape == (Ng, 1)
    assert ad.varm['sigma'].shape == (Ng, 1)
    for k in ('fdr', 'pval', 'ELBO_gain'):
        assert ad.varm[k].shape == (Ng, 1)
    assert np.asarray(ad.var['loss_gene']).shape == (Ng,)
    assert set(ad.uns['brie_param']) == {'LRT_index', 'base_mode', 'intecept', 'intercept_mode', 'sigma',
                                         'pseudo_count', 'layer_keys'}
    # p-values follow from the gains; FDR is computed over ALL events at once per batch in the reference
    from scipy.stats import chi2
    assert np.allclose(res.pval, chi2.sf(2 * res.ELBO_gain, df=1))


def test_BRIE2_class_protocol_and_null_base_mode():
    """BRIE2 mirror: constructor / fit / .numpy() attributes; testBase 'null' appends the tested
    feature's coefficient (model_wrap.py:164-171, 185-187)."""
    from brie_b200.models import BRIE2, fit_BRIE_matrix, Model_init
    Nc, Ng = 90, 40
    data, effLen, Xc, Xg = make_problem(Nc, Ng, 2, 0, True, 3, seed=2)
    d2 = [x.copy() for x in data]
    idx = d2[0] + d2[1] > 0
    for i in range(2):
        d2[i][idx] += 0.01
    init = Model_init(Nc, Ng, 2, 0, (1, Ng), (1, Ng), seed=5)
    m = BRIE2(Nc=Nc, Ng=Ng, Kc=2, Kg=0, effLen=effLen, intercept=None, intercept_mode='gene', init_obj=init)
    losses = m.fit(d2, Xc=Xc, Xg=None, min_iter=120, max_iter=120, MC_size=2, n_eval=10, verbose=False)
    assert losses.shape == (20,) and np.isfinite(losses).all()
    for name, shape in (('sigma', (1, Ng)), ('intercept', (1, Ng)), ('Wc_loc', (2, Ng)), ('Wg_loc', (Nc, 0)),
                        ('Psi', (Nc, Ng)), ('Z_loc', (Nc, Ng)), ('Z_std', (Nc, Ng)), ('loss_gene', (Ng,))):
        assert getattr(m, name).numpy().shape == shape, name
    assert m.Psi95CI.shape == (Nc, Ng) and (m.Psi95CI >= 0).all()
    assert np.abs(m.Z_loc.numpy()).max() <= 9.0
    with pytest.raises(ValueError, match="target"):
        m.fit(d2, Xc=Xc, target="nonsense")

    res = fit_BRIE_matrix([x.copy() for x in data], Xc=Xc, effLen=effLen, LRT_index=[1], base_mode='null',
                          intercept_mode='gene', min_iter=120, max_iter=120, MC_size=2, n_eval=10, seed=1)
    assert res.cell_coeff.shape == (2, Ng)          # base (feature 0) + appended tested feature 1
    assert res.ELBO_gain.shape == (Ng, 1) and res.n_iter.shape == (2, 1)
    ref = _patched_oracle(1, Nc, lambda: oracle_fit_matrix(
        [x.copy() for x in data], Xc=Xc, effLen=effLen, LRT_index=[1], base_mode='null', intercept_mode='gene',
        dtype=np.float32, min_iter=120, max_iter=120, MC_size=2, n_eval=10, seed=1))
    assert np.quantile(np.abs(res.Psi - ref.Psi), 0.99) < 1e-3
    assert np.abs(res.cell_coeff - ref.cell_coeff).max() < 5e-3
    assert np.abs(res.ELBO_gain - ref.ELBO_gain).max() < 2e-2


def test_cell_mode_base_with_gene_mode_refits():
    """intercept_mode='cell' + LRT: the reference's refits silently fall back to the per-event
    layout (model_wrap.py:174-178); we reproduce that with a second engine."""
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng = 80, 36
    data, effLen, Xc, Xg = make_problem(Nc, Ng, 1, 2, False, 2, seed=6)
    kw = dict(min_iter=120, max_iter=120, MC_size=2, n_eval=10)
    res = fit_BRIE_matrix([x.copy() for x in data], Xc=Xc, Xg=Xg, intercept_mode='cell', LRT_index=None, seed=2, **kw)
    assert res.intercept.shape == (Nc, 1) and res.sigma.shape == (Nc, 1) and res.gene_coeff.shape == (Nc, 2)
    ref = _patched_oracle(2, Nc, lambda: oracle_fit_matrix(
        [x.copy() for x in data], Xc=Xc, Xg=Xg, intercept_mode='cell', LRT_index=None, dtype=np.float32, seed=2, **kw))
    assert np.quantile(np.abs(res.Psi - ref.Psi), 0.99) < 1e-3
    assert np.abs(res.gene_coeff - ref.gene_coeff).max() < 5e-3
    assert np.abs(res.loss_gene - ref.loss_gene).max() <= 1e-4 * np.abs(ref.loss_gene).max()
    assert np.abs(res.ELBO_gain - ref.ELBO_gain).max() < 2e-2


def test_brie_quant_cli_end_to_end(tmp_path):
    """BASELINE config C1 in miniature: simulated 2-isoform counts, npz in, brie-quant without and
    with a cell covariate, result container + TSV out."""
    from brie_b200.bin.quant import quant
    from brie_b200.utils import io_utils
    from brie_b200.utils.anndata_lite import AnnDataLite
    Nc, Ng = 200, 60
    data, effLen, Xc, beta = make_lrt_problem(Nc, Ng, seed=11)
    eff3 = np.zeros((Ng, 2, 3), np.float32)
    eff3[:, 0, :], eff3[:, 1, :] = effLen[:, :3], effLen[:, 3:]
    cells = ["cell%03d" % i for i in range(Nc)]
    genes = ["ENSG%05d" % i for i in range(Ng)]
    inp = str(tmp_path / "brie_count.npz")
    io_utils.write_npz_counts(inp, {'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]}, eff3, cells, genes)
    out = str(tmp_path / "out" / "brie_quant.npz")
    ad = quant(inp, out_file=out, LRT_index=[], intercept=None, intercept_mode='gene', min_iter=240, max_iter=240,
               MC_size=3, batch_size=200 * 25)
    assert os.path.exists(out) and os.path.exists(out.replace(".npz", ".brie_ident.tsv"))
    assert ad.layers['Psi'].shape == ad.shape and 'ELBO_gain' not in ad.varm
    back = AnnDataLite.read_npz(out)
    assert np.array_equal(back.layers['Psi'], ad.layers['Psi'])
    # with a covariate file (shuffled rows, one unknown cell) and LRT on all features
    cf = tmp_path / "cells.tsv"
    order = np.random.default_rng(0).permutation(Nc)
    with open(cf, "w") as f:
        f.write("cellID\tgroup\n")
        f.write("ghost\t1\n")
        for i in order[:-5]:                                  # 5 cells have no covariate -> dropped
            f.write("%s\t%d\n" % (cells[i], int(Xc[i, 0])))
    out2 = str(tmp_path / "out" / "brie_quant_cell.npz")
    ad2 = quant(inp, cell_file=str(cf), out_file=out2, LRT_index=None, intercept=None, intercept_mode='gene',
                min_iter=600, max_iter=600, MC_size=3)
    assert ad2.shape[0] == Nc - 5
    tsv = open(out2.replace(".npz", ".brie_ident.tsv")).read().splitlines()
    hdr = tsv[0].split("\t")
    assert hdr[:6] == ['GeneID', 'n_counts', 'n_counts_uniq', 'cdr', 'intercept', 'sigma']
    assert hdr[6:] == ['group_ceoff', 'group_ELBO_gain', 'group_pval', 'group_FDR']
    assert len(tsv) == 1 + ad2.shape[1]
    # the planted strong effects are called, the nulls mostly not
    kept = np.array([g in set(ad2.var.index) for g in genes])
    b = beta[kept]
    fdr = ad2.varm['fdr'][:, 0]
    assert (fdr[b > 2] < 0.05).mean() > 0.9 and (fdr[b == 0] < 0.05).mean() < 0.2


def test_device_simulator_statistics_and_engine_zero_copy():
    """brie_simulate_counts follows the host recipe (same per-event parameters): detection rate,
    mean depth and isoform fractions agree; its padded device tensors feed the engine directly."""
    from brie_b200.utils.synth import simulate_counts, simulate_counts_device
    from brie_b200.engine import FitEngine
    Nc, Ng = 3000, 200
    dev = simulate_counts_device(Nc, Ng, design='binary1', seed=5)
    host = simulate_counts(Nc, Ng, design='binary1', seed=5)          # different RNG streams, same distributions
    d = [t[:, :Ng].cpu().numpy() for t in dev['layers']]
    from brie_b200._lib import leading_dim
    assert dev['layers'][0].shape == (Nc, leading_dim(Ng)) and float(dev['layers'][0][:, Ng:].abs().max()) == 0.0
    nz_d = (d[0] + d[1] + d[2] > 0)
    # pseudo-count applied exactly where c1 + c2 > 0
    frac = d[0] - np.floor(d[0])
    assert np.allclose(frac[(d[0] + d[1]) > 0.005], 0.01, atol=1e-4) and np.all(frac[(d[0] + d[1]) < 0.005] == 0)
    cdr, lam = dev['truth']['cdr'], dev['truth']['lam']
    want_det = cdr * (1 - np.exp(-lam))
    assert np.abs(nz_d.mean(0) - want_det).max() < 0.05
    tot = np.floor(d[0]) + np.floor(d[1]) + d[2]
    assert np.abs(tot.mean(0) - cdr * lam).max() < 0.15 * (1 + (cdr * lam).max())
    assert abs(nz_d.mean() - 0.165) < 0.04          # ~16 % non-zero, as the published tables' cdr
    eng = FitEngine(dev['layers'], effLen=dev['effLen'], Xc=dev['Xc'], n_events=Ng, MC_size=2, trace_cap=4)
    assert eng.counts[0].data_ptr() == dev['layers'][0].data_ptr()
    eng.init_params(); eng.begin_stage(0.01); eng.run_steps(2, 0)
    torch.cuda.synchronize()
    assert np.isfinite(eng.loss_trace[0, 1, :Ng].cpu().numpy()).all()


def test_fitBRIE_chunked_memmap_outputs_equal_single_chunk(tmp_path, monkeypatch):
    """Event chunking (HBM budget) and the out_dir memory-mapped writer do not change results:
    noise and init are keyed by global event ids, chunks are aligned to convergence groups."""
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    from brie_b200.utils.anndata_lite import AnnDataLite
    from scipy.sparse import csc_matrix
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10)

    def run(chunk_events, out_dir, sparse):
        wrap = csc_matrix if sparse else (lambda x: x.copy())
        ad = AnnDataLite(X=data[0] + data[1] + data[2],
                         layers={'isoform1': wrap(data[0]), 'isoform2': wrap(data[1]), 'ambiguous': wrap(data[2])},
                         varm={'effLen': effLen})
        if chunk_events:
            monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: chunk_events)
        else:
            monkeypatch.undo()
        return fitBRIE(ad, out_dir=out_dir, **kw), ad

    r1, ad1 = run(None, None, False)
    r2, ad2 = run(45, str(tmp_path / "layers"), True)          # 45 -> 40 events per chunk: chunks of 40, 40, 10
    assert isinstance(ad2.layers['Psi'], np.memmap) and os.path.exists(str(tmp_path / "layers" / "Psi.npy"))
    for k in ('Psi', 'Psi95CI', 'Z_std', 'Z_loc', 'loss_gene', 'ELBO_gain', 'pval', 'fdr', 'losses', 'cell_coeff',
              'sigma', 'intercept', 'n_iter'):
        assert np.array_equal(np.asarray(getattr(r1, k)), np.asarray(getattr(r2, k))), k
    assert np.array_equal(np.asarray(ad1.layers['Psi_95CI']), np.asarray(ad2.layers['Psi_95CI']))


def test_fitBRIE_resume_from_checkpointed_chunks(tmp_path, monkeypatch):
    """A fit that dies after two of three event chunks and is re-run with resume=True refits only the
    last chunk and returns exactly what the uninterrupted fit returns (SURVEY f4)."""
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    from brie_b200.utils.anndata_lite import AnnDataLite
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10)
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)        # chunks of 40, 40, 10 events

    def adata():
        return AnnDataLite(X=data[0] + data[1] + data[2],
                           layers={'isoform1': data[0].copy(), 'isoform2': data[1].copy(), 'ambiguous': data[2].copy()},
                           varm={'effLen': effLen})

    ref = fitBRIE(adata(), out_dir=str(tmp_path / "a"), **kw)
    real_fit, calls = mw.fit_BRIE_matrix, []

    def dying_fit(*a, **k):
        if len(calls) == 2:
            raise KeyboardInterrupt("job killed")
        calls.append(k['event_offset'])
        return real_fit(*a, **k)

    monkeypatch.setattr(mw, "fit_BRIE_matrix", dying_fit)
    with pytest.raises(KeyboardInterrupt):
        fitBRIE(adata(), out_dir=str(tmp_path / "b"), resume=True, **kw)
    assert calls == [0, 40] and os.path.exists(str(tmp_path / "b" / "chunk_40_80.pkl"))
    calls2 = []
    monkeypatch.setattr(mw, "fit_BRIE_matrix", lambda *a, **k: (calls2.append(k['event_offset']), real_fit(*a, **k))[1])
    ad = adata()
    res = fitBRIE(ad, out_dir=str(tmp_path / "b"), resume=True, **kw)
    assert calls2 == [80]                                                       # only the missing chunk was fitted
    for k in ('Psi', 'Psi95CI', 'Z_std', 'Z_loc', 'loss_gene', 'ELBO_gain', 'pval', 'fdr', 'losses', 'cell_coeff',
              'sigma', 'intercept', 'n_iter'):
        assert np.array_equal(np.asarray(getattr(ref, k)), np.asarray(getattr(res, k))), k
    assert np.array_equal(np.asarray(ad.layers['Psi']), np.asarray(ref.Psi))
    # a different seed is a different fit: nothing is reused
    calls2.clear()
    fitBRIE(adata(), out_dir=str(tmp_path / "b"), resume=True, **dict(kw, seed=5))
    assert calls2 == [0, 40, 80]


def test_one_vs_rest_lrt_with_15_covariates_null_base():
    """The reference's dentate-gyrus run (brie-tutorials/dentateGyrus/run_brie2.sh:31-36): 15 cell
    covariates (detection rate + 14 cluster indicators), --testBase null, LRT on 1..14.  Each
    batched model only carries its own columns (base: [0]; test ii: [0, idx]), so the device
    design width is 2, not 15."""
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.engine import FitEngine
    Nc, Ng, T = 120, 24, 14
    rng = np.random.default_rng(3)
    data, effLen, _, _ = make_problem(Nc, Ng, 0, 0, False, 2, seed=9)
    cluster = rng.integers(0, T, Nc)
    Xc = np.zeros((Nc, 1 + T), np.float32)
    Xc[:, 0] = rng.uniform(0.05, 0.3, Nc)
    Xc[np.arange(Nc), 1 + cluster] = 1
    kw = dict(Xc=Xc, LRT_index=list(range(1, T + 1)), base_mode='null', intercept_mode='gene', min_iter=120,
              max_iter=120, MC_size=2, n_eval=10)
    res = fit_BRIE_matrix([x.copy() for x in data], seed=1, **kw)
    assert res.ELBO_gain.shape == (Ng, T) and res.cell_coeff.shape == (1 + T, Ng) and res.n_iter.shape == (1 + T, 1)
    ref = _patched_oracle(1, Nc, lambda: oracle_fit_matrix([x.copy() for x in data], dtype=np.float32, seed=1, **kw))
    assert np.quantile(np.abs(res.Psi - ref.Psi), 0.99) < 1e-3
    assert np.abs(res.cell_coeff - ref.cell_coeff).max() < 5e-3
    assert np.abs(res.ELBO_gain - ref.ELBO_gain).max() < 2e-2
    eng = FitEngine([x.copy() for x in data], Xc=Xc, masks=[[0]] + [[0, k] for k in range(1, T + 1)])
    assert eng.Kc == 2 and eng.Xc.shape == (1 + T, Nc, 2)
    # the same design in full mode (each refit drops one of the 15 columns) needs width 15 -> 16
    eng = FitEngine([x.copy() for x in data], Xc=Xc, masks=[list(range(15))] + [[k for k in range(15) if k != i]
                                                                               for i in range(1, 15)])
    assert eng.Kc == 16 and eng.sizes.n_col_tiles == 1
    # beyond 16 columns the design is "wide": contractions as GEMMs around the fused kernel, any width
    eng = FitEngine([x.copy() for x in data], Xc=np.ones((Nc, 40), np.float32))
    assert eng.wide and eng.Kc == 40
    with pytest.raises(ValueError, match="exceeds the supported maximum"):
        FitEngine([x.copy() for x in data], Xc=np.ones((Nc, 5000), np.float32))


def test_BRIE2_public_model_api_matches_oracle():
    """BRIE2.logLik_MC / get_loss / Z_prior / Z / PsiDist (model_TFProb.py:96-127, 130-211) on the device path,
    against the oracle with the device's noise; re-exports of brie/models/__init__.py:4."""
    from oracle import philox_np as px
    from oracle.brie2_oracle import OracleBRIE2, add_pseudo_count, kl_normal_normal
    from brie_b200 import models
    assert all(hasattr(models, n) for n in ("BRIE2", "fitBRIE", "fit_BRIE_matrix", "get_CI95", "BRIE_base_lik", "LogitNormal"))
    Nc, Ng, seed, S = 70, 53, 6, 4
    for mode, Kc, Kg, eff, nl in (('gene', 2, 0, True, 3), ('cell', 1, 3, False, 2)):
        data, effLen, Xc, Xg = make_problem(Nc, Ng, Kc, Kg, eff, nl, seed=4)
        add_pseudo_count(data, np.float32(0.01))
        m = models.BRIE2(Nc=Nc, Ng=Ng, Kc=Kc, Kg=Kg, effLen=effLen, intercept=None, intercept_mode=mode, seed=seed)
        m.fit(data, Xc=Xc, Xg=Xg if Kg else None, min_iter=60, max_iter=60, MC_size=2, n_eval=4, verbose=False)
        e = m._engine
        om = OracleBRIE2(Nc, Ng, Kc, Kg, effLen, None, mode, None, dtype=np.float64, seed=seed)
        om.p['Z_loc'], om.p['Z_std_log'] = m.Z_loc.numpy().astype(np.float64), np.log(m.Z_std.numpy().astype(np.float64))
        om.p['Wc_loc'], om.p['Wg_loc'] = m.Wc_loc.numpy().astype(np.float64), m.Wg_loc.numpy().astype(np.float64)
        om.p['intercept'], om.p['sigma_log'] = m.intercept.numpy().astype(np.float64), np.log(m.sigma.numpy().astype(np.float64))
        om.Xc, om.Xg = Xc.astype(np.float64), Xg.astype(np.float64)
        # Z_prior / Z / PsiDist
        zp = m.Z_prior
        assert np.abs(zp.parameters['loc'] - om.prior_mean()).max() < 2e-5
        assert zp.sample(3, seed=1).shape == (3, Nc, Ng)
        assert np.abs(m.Z.loc - om.p['Z_loc']).max() == 0
        assert np.abs(m.PsiDist.quantile(0.975) - m.PsiDist.quantile(0.025) - m.Psi95CI).max() < 2e-6
        # logLik_MC with pinned noise counters (element_terms), ELBO and marginLik targets
        epsf = device_eps_provider(seed, 0, Nc, Ng)
        for margin in (False, True):
            ll, kl, _ = e.element_terms(0, mc_size=S, margin=margin, kl=True, noise_step=77)
            eps = epsf(px.PHASE_EVAL, 77, S).astype(np.float64)
            c = [np.asarray(x, np.float64) for x in data]
            if margin:
                z = om.prior_mean()[None] + (np.exp(om.p['sigma_log']) + np.zeros((Nc, Ng)))[None] * eps
                ls = om._loglik_samples(c, z)[0]
                ref = np.log(np.exp(ls - ls.max(0)[None]).mean(0)) + ls.max(0)
            else:
                z = om.p['Z_loc'][None] + np.exp(om.p['Z_std_log'])[None] * eps
                ref = om._loglik_samples(c, z)[0].mean(0)
            assert np.abs(ll.cpu().numpy() - ref).max() <= 2e-5 * max(np.abs(ref).max(), 1.0), (mode, margin)
            ref_kl = kl_normal_normal(om.p['Z_loc'], om.p['Z_std_log'], om.prior_mean(), om.p['sigma_log'] + np.zeros((Nc, Ng)))
            assert np.abs(kl.cpu().numpy() - ref_kl).max() <= 2e-5 * max(ref_kl.max(), 1.0)
        # the public methods: shapes, reductions and consistency (fresh noise on every call)
        ll = m.logLik_MC(data, MC_size=64).numpy()
        assert ll.shape == (Nc, Ng) and (ll <= 1e-6).all()
        lg = m.get_loss(data, axis=0, MC_size=64).numpy()
        tot = float(m.get_loss(data, MC_size=64).numpy())
        assert lg.shape == (Ng,) and m.get_loss(data, axis=1).numpy().shape == (Nc,)
        ref_lg = om.loss_and_grads(data, epsf(px.PHASE_EVAL, 5, 64), want_grads=False)[1]
        assert np.abs(lg - ref_lg).max() <= 0.05 * np.abs(ref_lg).max()        # different noise: MC error only
        assert abs(tot - lg.sum()) <= 0.02 * abs(tot)
        ml = m.get_loss(data, target="marginLik", axis=0, MC_size=8).numpy()
        assert ml.shape == (Ng,) and np.isfinite(ml).all()
        # other count layers than the fitted ones are honoured (get_loss takes count_layers as an argument)
        zero = [np.zeros_like(x) for x in data]
        assert np.abs(m.logLik_MC(zero, MC_size=2).numpy()).max() == 0


def test_device_simulator_mirrors_reference_semantics():
    """brie.models.simulator (simulator.py:7-75): counts ~ Multinomial(observed total, Phi) on the device --
    totals preserved exactly, category frequencies follow Phi, posterior / prior modes, side effects on adata."""
    from brie_b200.models.simulator import simulator
    from brie_b200.utils.anndata_lite import AnnDataLite
    Nc, Ng = 400, 60
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=5)
    rng = np.random.default_rng(0)
    Psi = rng.uniform(0.05, 0.95, (1, Ng)).astype(np.float32) * np.ones((Nc, 1), np.float32)
    ad = AnnDataLite(X=data[0] + data[1] + data[2],
                     layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2], 'Psi': Psi},
                     varm={'effLen': effLen})
    sim = simulator(ad, seed=3)
    tot = data[0] + data[1] + data[2]
    c = [sim.layers[k] for k in ('isoform1', 'isoform2', 'ambiguous')]
    assert np.array_equal(c[0] + c[1] + c[2], tot)                       # depth is conserved element by element
    assert all((x >= 0).all() and np.array_equal(x, np.rint(x)) for x in c)
    assert sim is not ad and np.array_equal(ad.layers['isoform1'], data[0])      # input counts untouched
    assert np.array_equal(ad.layers['Psi_sim'], Psi)                     # side effect of simulator.py:42
    L = effLen[:, [0, 4, 5]]
    w = np.stack([Psi[0] * L[:, 0], (1 - Psi[0]) * L[:, 1], L[:, 2]], 1)
    phi = w / w.sum(1, keepdims=True)
    n_g = tot.sum(0)
    for k in range(3):                                                   # column frequencies within 5 binomial sd
        f = c[k].sum(0) / n_g
        sd = np.sqrt(phi[:, k] * (1 - phi[:, k]) / n_g)
        assert (np.abs(f - phi[:, k]) < 5 * sd + 1e-6).all(), k
    assert not np.array_equal(simulator(ad, seed=4).layers['isoform1'], c[0])
    assert np.array_equal(simulator(ad, seed=3).layers['isoform1'], c[0])        # counter-based: reproducible
    # prior mode: Psi from the fitted coefficients + N(0, sigma) noise, clipped in logit space
    ad.obsm['Xc'], ad.varm['cell_coeff'] = Xc, rng.normal(0, 1, (Ng, 1)).astype(np.float32)
    ad.varm['intercept'] = rng.normal(0, 2, (Ng, 1)).astype(np.float32)
    ad.varm['sigma'] = np.full((Ng, 1), 0.3, np.float32)
    sim2 = simulator(ad, mode="prior", seed=1)
    z0 = Xc @ ad.varm['cell_coeff'].T + ad.varm['intercept'].T
    assert np.allclose(ad.layers['Psi_sim_noNoise'], 1 / (1 + np.exp(-z0)), atol=1e-6)
    zs = np.log(ad.layers['Psi_sim'] / (1 - ad.layers['Psi_sim']))
    assert abs(np.std(zs - z0) - 0.3) < 0.02 and np.abs(zs).max() <= 9.0 + 1e-3
    assert np.array_equal(sum(sim2.layers[k] for k in ('isoform1', 'isoform2', 'ambiguous')), tot)
    sim3 = simulator(ad, mode="prior", prior_sigma=1.5, seed=1)
    zs3 = np.log(ad.layers['Psi_sim'] / (1 - ad.layers['Psi_sim']))
    assert abs(np.std(np.clip(zs3 - z0, -20, 20)) - 1.5) < 0.1


def test_bench_dump_outputs_hold_the_state_after_the_timed_steps(tmp_path, monkeypatch):
    """bench.py --dump-outputs on a small shape with the headline's layout (M = 4, Kc = 3, gene intercept): the
    files are the engine state after the warm-up and exactly --steps timed steps, and the same arguments give the
    same inputs, so two runs dump the same arrays bit for bit."""
    import bench
    monkeypatch.setitem(bench.SHAPES, "T", dict(bench.SHAPES[bench.HEAD], cells=300, events=70))
    ctx = bench.Ctx()
    dumps = []
    for run, K in enumerate((4, 4, 5)):
        (lo, hi), group, Ng = bench.shard_of(ctx, "T")
        eng, _ = bench.build_engine(ctx, "T", lo, hi, Ng, group)
        bench.time_steps(ctx, eng, K, 3)
        assert eng.step_counters()[0] == 3 + K
        out = str(tmp_path / str(run))
        bench.dump_outputs(ctx, eng, out, n_cells=16)
        d = {f[:-len(".npy")]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
        assert set(d) == {"Z_loc", "Z_std_log", "Wc", "intercept", "sigma_log"}
        assert all(v.dtype == np.float32 for v in d.values())
        cells = np.sort(np.random.default_rng(0).choice(300, 16, replace=False))
        assert d["Z_loc"].shape == (4, 16, 70) and d["Wc"].shape == (4, 3, 70) and d["sigma_log"].shape == (4, 70)
        assert np.array_equal(d["Z_loc"], eng.Z_loc[:, cells, :70].cpu().numpy())
        assert np.array_equal(d["Z_std_log"], eng.Z_std_log[:, cells, :70].cpu().numpy())
        assert np.array_equal(d["intercept"], eng.intercept[:, :70].cpu().numpy())
        dumps.append(d)
        del eng
    for k in dumps[0]:
        assert np.array_equal(dumps[0][k], dumps[1][k]), k
    assert not np.array_equal(dumps[0]["Z_loc"], dumps[2]["Z_loc"])
