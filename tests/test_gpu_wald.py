"""GPU tests of the Wald tests from the fitted posterior (wald / brie-quant --wald): the information kernel against
its float64 restatement on the engine's own state, determinism, that nothing else moves, calibration under no effect
(and that the naive information fails it), chunking, resume, the CLI and event sharding over two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import wald_ref
from oracle.brie2_oracle import add_pseudo_count
from util import make_lrt_problem, make_problem

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WALD_KEYS = ('cell_coeff_se', 'pval_wald', 'fdr_wald', 'intercept_se', 'wald_columns')


def _close(got, want):
    """<= 1e-6 relative per entry (plus a floor far below the entry's scale, for entries that cancel to ~0)."""
    d = np.sqrt(np.abs(np.diagonal(want, axis1=1, axis2=2)))
    floor = 1e-12 * d[:, :, None] * d[:, None, :]
    err = np.abs(got - want)
    rel = err / np.maximum(np.abs(want), floor + 1e-300)
    print("information vs float64 restatement: max rel %.2e over %d entries" % (rel.max(initial=0), want.size))
    assert (err <= 1e-6 * np.abs(want) + floor).all()


def _check_engine(eng):
    for m in range(eng.M):
        got = eng.wald_info(m)
        want = wald_ref.engine_reference(eng, m)
        kt = len(eng.masks[m]) + (not eng.cell_mode and eng.intercept_const is None)
        assert got.shape == (eng.Ng, kt, kt)
        _close(got, want)
        assert np.array_equal(got, eng.wald_info(m))              # repeated calls: bit-identical
        if kt:
            assert (np.diagonal(got, axis1=1, axis2=2) > 0).any()


# (Kc, Kg, intercept mode, masks): Kc 0, 1, 3 and 16; gene, None and cell; Kg 4; the wide form at Kc 24
CASES = [(0, 0, 'gene', None), (1, 0, 'gene', [[0], []]), (3, 0, 'None', [[0, 1, 2], [0, 2]]),
         (3, 0, 'cell', None), (16, 0, 'gene', [list(range(16)), list(range(1, 16))]), (2, 4, 'gene', None),
         (1, 4, 'cell', None), (24, 0, 'gene', [list(range(24)), list(range(23))])]


@pytest.mark.parametrize("Kc,Kg,mode,masks", CASES)
def test_information_kernel_matches_the_float64_restatement(Kc, Kg, mode, masks):
    from brie_b200.engine import FitEngine
    Nc, Ng = 300, 130                                          # tails: 300 rows, 130 events (not multiples of 32)
    data, effLen, Xc, Xg = make_problem(Nc, Ng, Kc, Kg, True, 3, seed=4)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, Xg=Xg, masks=masks, intercept=0 if mode == 'None' else None,
                    intercept_mode=mode, MC_size=2, seed=3, trace_cap=8)
    eng.init_params()
    eng.begin_stage(0.02)
    eng.run_steps(80)
    _check_engine(eng)


def test_information_after_gathered_extension_rounds():
    from brie_b200.engine import FitEngine
    Nc, Ng, group = 300, 700, 3
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=8)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, masks=[[0, 1], [1]], model_ids=[0, 1], MC_size=3, seed=12,
                    trace_cap=8, group_size=group)
    eng.init_params(); eng.begin_stage(0.01); eng.run_steps(40)
    for frac in (0.3, 0.05):
        act = np.random.default_rng(int(frac * 100)).random((2, eng.n_groups)) < frac
        act[1, 0] = True
        assert eng.run_steps_gathered(act, 30, force=True)
    assert eng.gather_rounds == 2
    _check_engine(eng)


def _fields(r):
    return {k: v for k, v in vars(r).items() if k not in WALD_KEYS + ('timing', 'timing_rank', 'launch_count')}


def _same(a, b):
    fa, fb = _fields(a), _fields(b)
    assert set(fa) == set(fb)
    for k in fa:
        assert np.array_equal(np.asarray(fa[k]), np.asarray(fb[k])), k


@pytest.mark.parametrize("base_mode,n_perm", [("full", 0), ("null", 0), ("full", 2), ("null", 2)])
def test_fit_matrix_outputs_bit_identical_with_and_without_wald(base_mode, n_perm):
    from brie_b200.engine import wald_from_info
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng = 120, 40
    data, effLen, Xc, Xg = make_problem(Nc, Ng, 3, 0, True, 3, seed=2)
    kw = dict(Xc=Xc, effLen=effLen, LRT_index=[0, 2], base_mode=base_mode, intercept_mode='gene', min_iter=240,
              max_iter=740, MC_size=2, n_eval=10, seed=3, n_perm=n_perm)
    r0 = fit_BRIE_matrix([x.copy() for x in data], **kw)
    r1 = fit_BRIE_matrix([x.copy() for x in data], wald=True, **kw)
    _same(r0, r1)
    assert not any(hasattr(r0, k) for k in WALD_KEYS)
    rows = r1.cell_coeff.shape[0]
    assert r1.cell_coeff_se.shape == r1.cell_coeff.shape and r1.pval_wald.shape == (Ng, rows)
    assert r1.intercept_se.shape == r1.intercept.shape
    assert r1.wald_columns == ([0, 1, 2] if base_mode == "full" else [1, 0, 2])
    assert ((r1.pval_wald > 0) & (r1.pval_wald <= 1)).all()
    # an event whose cells with reads cannot separate a coefficient from the intercept (e.g. all on one side of the
    # binary covariate) has a singular information: se NaN, pval 1
    bad = ~np.isfinite(r1.cell_coeff_se.T)
    assert bad.mean() < 0.1 and (r1.pval_wald[bad] == 1).all()
    # elsewhere z of a cell_coeff row = its coefficient over its standard error
    from scipy.stats import chi2
    want = chi2.sf((r1.cell_coeff / r1.cell_coeff_se).T ** 2, 1)
    assert np.allclose(r1.pval_wald[~bad], want[~bad])


def _adata(data, effLen):
    from brie_b200.utils.anndata_lite import AnnDataLite
    return AnnDataLite(X=data[0] + data[1] + data[2],
                       layers={'isoform1': data[0].copy(), 'isoform2': data[1].copy(), 'ambiguous': data[2].copy()},
                       varm={'effLen': effLen})


def _same_adata(a, b, skip=()):
    for grp in ('obsm', 'varm', 'layers'):
        da, db = getattr(a, grp), getattr(b, grp)
        assert set(da) - set(skip) == set(db) - set(skip), grp
        for k in set(da) - set(skip):
            assert np.array_equal(np.asarray(da[k]), np.asarray(db[k])), (grp, k)
    assert np.array_equal(np.asarray(a.var['loss_gene']), np.asarray(b.var['loss_gene']))


@pytest.mark.parametrize("base_mode,cell", [("full", False), ("null", False), ("full", True)])
def test_fitBRIE_outputs_bit_identical_with_and_without_wald(base_mode, cell):
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 60
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=5)
    kw = dict(Xc=Xc, LRT_index=[1], base_mode=base_mode, intercept_mode='cell' if cell else 'gene',
              batch_size=100 * 20, seed=4, min_iter=300, max_iter=800, MC_size=2, n_eval=10, n_perm=2)
    a0, a1 = _adata(data, effLen), _adata(data, effLen)
    r0, r1 = fitBRIE(a0, **kw), fitBRIE(a1, wald=True, **kw)
    _same(r0, r1)
    new = {'cell_coeff_se', 'pval_wald', 'fdr_wald'} | (set() if cell else {'intercept_se'})
    assert set(a1.varm) - set(a0.varm) == new
    _same_adata(a0, a1, skip=new)
    assert 'wald' not in a0.uns['brie_param'] and a1.uns['brie_param']['wald'] is True
    assert a1.uns['brie_param']['wald_columns'] == ([0, 1] if base_mode == "full" else [0, 1])
    assert a1.varm['cell_coeff_se'].shape == a1.varm['cell_coeff'].shape


def _no_effect_problem(Nc, Ng, n_strong, seed):
    """make_lrt_problem's generator with the covariate effect zero on all but the last `n_strong` events (the
    design of test_gpu_perm.py)."""
    rng = np.random.default_rng(seed)
    x = rng.binomial(1, 0.5, Nc).astype(np.float32)
    beta = np.zeros(Ng)
    beta[Ng - n_strong:] = 2.5
    z = rng.normal(0, 1.0, Ng)[None, :] + x[:, None] * beta[None, :] + rng.normal(0, 0.5, (Nc, Ng))
    psi = 1 / (1 + np.exp(-z))
    ex = rng.uniform(50, 300, (Ng, 3))
    L1, L2, L3 = ex[:, 1] + 72, np.full(Ng, 72.0), ex[:, 0] + ex[:, 2] - 16
    effLen = np.zeros((Ng, 6), np.float32)
    effLen[:, 0], effLen[:, 2], effLen[:, 4], effLen[:, 5] = L1, L3, L2, L3
    n = rng.poisson(25, (Nc, Ng)) * (rng.uniform(size=(Nc, Ng)) < 0.7)
    p1, p2 = psi * L1, (1 - psi) * L2
    D = p1 + p2 + L3
    c1 = rng.binomial(n, p1 / D)
    c2 = rng.binomial(n - c1, p2 / (D - p1))
    c3 = n - c1 - c2
    return [c1.astype(np.float32), c2.astype(np.float32), c3.astype(np.float32)], effLen, x[:, None], beta


FIT = dict(intercept_mode='gene', min_iter=600, max_iter=2100, MC_size=2, n_eval=500, seed=5)


def test_wald_pvalues_calibrated_under_no_effect():
    from scipy.stats import kstest, spearmanr
    from brie_b200.models import fit_BRIE_matrix
    data, effLen, Xc, beta = _no_effect_problem(150, 120, 16, seed=12)
    res = fit_BRIE_matrix(data, Xc=Xc, effLen=effLen, LRT_index=[0], wald=True, **FIT)
    null, strong = beta == 0, beta > 0
    pw, pc = res.pval_wald[:, 0], res.pval[:, 0]
    ks = kstest(pw[null], "uniform")
    z2 = (res.cell_coeff[0] / res.cell_coeff_se[0]) ** 2
    rho = spearmanr(z2, 2 * res.ELBO_gain[:, 0]).correlation
    r = np.corrcoef(z2, 2 * res.ELBO_gain[:, 0])[0, 1]
    print("no-effect events (%d): rejection at 0.05 -- chi2 %.3f, Wald %.3f; Wald KS vs uniform p %.3g"
          % (null.sum(), (pc[null] < 0.05).mean(), (pw[null] < 0.05).mean(), ks.pvalue))
    print("planted effects (%d): rejection at 0.05 -- chi2 %.3f, Wald %.3f; z^2 vs 2 ELBO_gain over all events: "
          "Spearman %.3f, Pearson %.3f; no-effect events only: Spearman %.3f"
          % (strong.sum(), (pc[strong] < 0.05).mean(), (pw[strong] < 0.05).mean(), rho, r,
             spearmanr(z2[null], res.ELBO_gain[null, 0]).correlation))
    assert ks.pvalue > 1e-3
    assert (pw[null] < 0.05).mean() <= 0.10
    assert (pw[strong] < 0.05).mean() >= 0.9
    # Spearman over all events stays below Pearson: on the no-effect events both statistics are near zero and the
    # Monte-Carlo noise of ELBO_gain sets their ranks (DESIGN §2.2)
    assert r > 0.9 and rho > 0.75


def test_naive_complete_data_information_is_visibly_miscalibrated():
    """The same fitted state, with the information sum_c x x^T / sigma^2 that drops the missing-information term:
    the calibration check above tells the two apart."""
    from brie_b200.engine import FitEngine, wald_from_info
    data, effLen, Xc, beta = _no_effect_problem(150, 120, 16, seed=12)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, MC_size=FIT['MC_size'], seed=FIT['seed'], trace_cap=500)
    eng.fit(min_iter=FIT['min_iter'], max_iter=FIT['max_iter'], n_eval=FIT['n_eval'])
    coef = np.stack([eng.Wc[0, 0, :eng.Ng].cpu().numpy(), eng.intercept[0, :eng.Ng].cpu().numpy()], axis=1)
    Xt = wald_ref.design_rows(Xc, True)
    naive = wald_ref.naive_info(eng.sigma_log[0, :eng.Ng].cpu().numpy(), Xt, eng.Ng)
    null = beta == 0
    rej_louis = (wald_from_info(coef, eng.wald_info(0))[1][null, 0] < 0.05).mean()
    rej_naive = (wald_from_info(coef, naive)[1][null, 0] < 0.05).mean()
    print("no-effect rejection at 0.05: Louis information %.3f, naive complete-data information %.3f"
          % (rej_louis, rej_naive))
    assert rej_naive >= 0.2 and rej_naive >= rej_louis + 0.1


def test_fitBRIE_chunked_equals_unchunked_and_fdr_wald_is_pooled(monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    from brie_b200.models.model_wrap import fdr_bh
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=[], intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10, wald=True)
    ad_one = _adata(data, effLen)
    one = fitBRIE(ad_one, **kw)                                                  # one chunk
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)         # chunks of 40, 40, 10 events
    ad = _adata(data, effLen)
    r = fitBRIE(ad, **kw)
    for k in ('cell_coeff', 'cell_coeff_se', 'intercept_se', 'pval_wald', 'fdr_wald'):
        assert np.array_equal(getattr(one, k), getattr(r, k)), k
    assert np.array_equal(r.fdr_wald[:, 0], fdr_bh(r.pval_wald[:, 0]))         # BH over all 90 events
    for k in ('cell_coeff_se', 'pval_wald', 'fdr_wald', 'intercept_se'):
        assert np.array_equal(ad.varm[k], ad_one.varm[k]), k
    assert ad.uns['brie_param']['wald_columns'] == [0] and 'ELBO_gain' not in ad.varm


def test_fitBRIE_resume_with_wald(tmp_path, monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10, wald=True)
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)
    ref = fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "a"), **kw)
    real_fit, calls = mw.fit_BRIE_matrix, []

    def dying_fit(*a, **k):
        if len(calls) == 2:
            raise KeyboardInterrupt("job killed")
        calls.append(k['event_offset'])
        return real_fit(*a, **k)
    monkeypatch.setattr(mw, "fit_BRIE_matrix", dying_fit)
    with pytest.raises(KeyboardInterrupt):
        fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, **kw)
    calls2 = []
    monkeypatch.setattr(mw, "fit_BRIE_matrix", lambda *a, **k: (calls2.append(k['event_offset']), real_fit(*a, **k))[1])
    res = fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, **kw)
    assert calls2 == [80]
    for k in ('cell_coeff_se', 'intercept_se', 'pval_wald', 'fdr_wald', 'ELBO_gain', 'pval'):
        assert np.array_equal(np.asarray(getattr(ref, k)), np.asarray(getattr(res, k))), k
    # a fit without wald is another fit: nothing is reused
    calls2.clear()
    fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, **dict(kw, wald=False))
    assert calls2 == [0, 40, 80]


def test_brie_quant_cli_with_wald(tmp_path):
    from brie_b200.utils import io_utils
    from brie_b200.utils.anndata_lite import AnnDataLite
    Nc, Ng = 120, 60
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=21)
    eff3 = np.zeros((Ng, 2, 3), np.float32)
    eff3[:, 0, :], eff3[:, 1, :] = effLen[:, :3], effLen[:, 3:]
    cells = ["cell%03d" % i for i in range(Nc)]
    inp = str(tmp_path / "counts.npz")
    io_utils.write_npz_counts(inp, {'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]}, eff3, cells,
                              ["g%03d" % i for i in range(Ng)])
    rng = np.random.default_rng(0)
    cf = tmp_path / "cells.tsv"
    with open(cf, "w") as f:
        f.write("cellID\tgroup\tbatch\n")
        for i in range(Nc):
            f.write("%s\t%d\t%.3f\n" % (cells[i], int(Xc[i, 0]), rng.normal()))
    out = str(tmp_path / "o" / "brie_quant.npz")
    p = subprocess.run([sys.executable, "-m", "brie_b200.bin.quant", "-i", inp, "-c", str(cf), "-o", out,
                        "--LRTindex", "1", "--testBase", "null", "--interceptMode", "gene", "--minIter", "300",
                        "--maxIter", "800", "--MCsize", "2", "--minCount", "10", "--minUniqCount", "5", "--minCell",
                        "5", "--wald"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
    assert p.returncode == 0, p.stderr[-3000:]
    ad = AnnDataLite.read_npz(out)
    G = ad.shape[1]
    for k in ('cell_coeff_se', 'pval_wald', 'fdr_wald'):
        assert ad.varm[k].shape == (G, 2), k
    assert ad.varm['intercept_se'].shape == (G, 1)
    assert ad.uns['brie_param']['wald'] is True and list(ad.uns['brie_param']['wald_columns']) == [0, 1]
    tsv = open(out.replace(".npz", ".brie_ident.tsv")).read().splitlines()
    hdr = tsv[0].split("\t")
    # null base: cell_coeff rows are base covariate 0 ('group'), then the tested covariate 1 ('batch'); the LRT
    # columns take cell_coeff by loop position (the reference's quirk), the Wald ones by wald_columns
    assert hdr == ['GeneID', 'n_counts', 'n_counts_uniq', 'cdr', 'intercept', 'sigma', 'batch_ceoff',
                   'batch_ELBO_gain', 'batch_pval', 'batch_FDR', 'group_se', 'group_pval_wald', 'group_FDR_wald',
                   'batch_se', 'batch_pval_wald', 'batch_FDR_wald']
    assert len(tsv) == 1 + G


WORKER = r'''
import os, sys, pickle
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
from util import make_lrt_problem, make_problem
from brie_b200.models import fitBRIE
from brie_b200.utils.anndata_lite import AnnDataLite
world = int(os.environ.get("WORLD_SIZE", "1"))
if world > 1:
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
out = {}
data, effLen, Xc, _ = make_lrt_problem(100, 130, seed=3)
ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]}, varm={'effLen': effLen})
r = fitBRIE(ad, Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4,
            min_iter=600, max_iter=1600, MC_size=2, n_eval=20, wald=True)
out['a'] = dict(se=r.cell_coeff_se, ise=r.intercept_se, pw=r.pval_wald, fw=r.fdr_wald, n_iter=r.n_iter)
data, effLen, Xc, Xg = make_problem(80, 64, 1, 2, False, 2, seed=6)
ad = AnnDataLite(X=data[0], layers={'spliced': data[0], 'unspliced': data[1]})
r = fitBRIE(ad, Xc=Xc, Xg=Xg, LRT_index=None, intercept_mode='cell', layer_keys=['spliced', 'unspliced'], seed=2,
            min_iter=360, max_iter=1860, MC_size=2, n_eval=20, wald=True)
out['c'] = dict(se=r.cell_coeff_se, pw=r.pval_wald, fw=r.fdr_wald, n_iter=r.n_iter)
if world == 1 or dist.get_rank() == 0:
    pickle.dump(out, open(%(out)r, "wb"))
if world > 1:
    dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_fitBRIE_with_wald_matches_single_gpu(tmp_path):
    import pickle
    from brie_b200.models.model_wrap import fdr_bh
    res = {}
    for world in (1, 2):
        out = str(tmp_path / ("w%d.pkl" % world))
        script = tmp_path / ("worker%d.py" % world)
        script.write_text(WORKER % dict(root=ROOT, out=out))
        if world == 1:
            cmd = [sys.executable, str(script)]
        else:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                   "--master-addr", "127.0.0.1", "--master-port", "29661", str(script)]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        res[world] = pickle.load(open(out, "rb"))
    for case in ('a', 'c'):
        for w in (1, 2):
            r = res[w][case]
            assert np.array_equal(r['fw'][:, 0], fdr_bh(r['pw'][:, 0])), (case, w)     # pooled over all ranks
        assert res[1][case]['se'].shape == res[2][case]['se'].shape
        assert np.array_equal(res[1][case]['n_iter'], res[2][case]['n_iter'])
    a1, a2 = res[1]['a'], res[2]['a']
    # independent events: the state is the same up to the tolerance of the observed gains in test_gpu_multi
    assert np.allclose(a1['se'], a2['se'], rtol=1e-3) and np.allclose(a1['ise'], a2['ise'], rtol=1e-3)
    c1, c2 = res[1]['c'], res[2]['c']
    assert np.allclose(c1['se'], c2['se'], rtol=1e-2)
