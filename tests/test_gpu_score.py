"""GPU tests of the score tests of candidate cell covariates (score_X / brie-quant --scoreFile): the score-parts
kernel against its float64 restatement on the engine's own state, determinism, that nothing else moves,
calibration and power on the no-effect design, chunking, resume, the CLI and event sharding over two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import score_ref
from oracle.brie2_oracle import add_pseudo_count
from test_gpu_wald import CASES, _adata, _no_effect_problem, _same_adata
from util import make_lrt_problem, make_problem

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCORE_KEYS = ('score_z', 'score_effect', 'pval_score', 'fdr_score')


def _close(name, got, want, mag):
    """<= 1e-6 relative per entry, with a floor of 1e-12 x the entry's absolute-value sum for entries that cancel."""
    err = np.abs(got - want)
    floor = 1e-12 * mag
    rel = err / np.maximum(np.abs(want), floor + 1e-300)
    print("%s vs float64 restatement: max rel %.2e over %d entries" % (name, rel.max(initial=0), want.size))
    assert (err <= 1e-6 * np.abs(want) + floor).all(), name


def _candidates(Nc, J, seed):
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(Nc, J)).astype(np.float32)
    X[:, ::3] = rng.binomial(1, 0.4, size=(Nc, len(range(0, J, 3))))
    return X


def _check_engine(eng, J):
    X = _candidates(eng.Nc, J, J)
    for m in range(eng.M):
        got = eng.score_parts(m, X)
        want = score_ref.engine_reference(eng, m, X)
        # absolute-value sums of every term, for the floor: |r| <= (|Z_loc| + |prior mean|) / sigma^2
        n = eng.Nc if eng.cell_mode else eng.Ng
        abs_parts = score_ref.parts(np.abs(eng.Z_loc[m, :, :eng.Ng].cpu().numpy()), eng.Z_std_log[m, :, :eng.Ng].cpu()
                                    .numpy(), eng.sigma_log[m, :n].cpu().numpy(), -np.abs(score_ref.prior_mean(eng, m)),
                                    np.abs(_xt(eng, m)), np.abs(X), eng.cell_mode)
        kt = _xt(eng, m).shape[1]
        assert got[0].shape == (eng.Ng, J) and got[2].shape == (eng.Ng, J, kt) and got[3].shape == (eng.Ng, kt)
        for name, g, w, a in zip(("U", "A", "B", "Ut"), got, want, abs_parts):
            _close(name, g, w, np.abs(a))
        again = eng.score_parts(m, X)
        assert all(np.array_equal(a, b) for a, b in zip(got, again))        # repeated calls: bit-identical


def _xt(eng, m):
    import wald_ref
    has_b = not eng.cell_mode and eng.intercept_const is None
    return wald_ref.design_rows(eng.Xc[m, :, :len(eng.masks[m])].cpu().numpy(), has_b)


@pytest.mark.parametrize("J", [1, 37, 300])
@pytest.mark.parametrize("Kc,Kg,mode,masks", CASES)
def test_score_parts_kernel_matches_the_float64_restatement(Kc, Kg, mode, masks, J):
    from brie_b200.engine import FitEngine
    Nc, Ng = 300, 130
    data, effLen, Xc, Xg = make_problem(Nc, Ng, Kc, Kg, True, 3, seed=4)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, Xg=Xg, masks=masks, intercept=0 if mode == 'None' else None,
                    intercept_mode=mode, MC_size=2, seed=3, trace_cap=8)
    eng.init_params()
    eng.begin_stage(0.02)
    eng.run_steps(80)
    _check_engine(eng, J)


def test_score_parts_after_gathered_extension_rounds():
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
    _check_engine(eng, 37)


def test_candidate_blocks_give_the_same_bits(monkeypatch):
    """Candidates split into blocks (SCORE_BLOCK_BYTES) give the bits of one call."""
    import brie_b200.engine as E
    from brie_b200.engine import FitEngine
    data, effLen, Xc, _ = make_problem(300, 130, 3, 0, True, 3, seed=4)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, MC_size=2, seed=3, trace_cap=8)
    eng.init_params(); eng.begin_stage(0.02); eng.run_steps(40)
    X = _candidates(300, 40, 1)
    one = eng.score_parts(0, X)
    monkeypatch.setattr(E, "SCORE_BLOCK_BYTES", 200_000)                       # blocks of a few candidates
    blocks = eng.score_parts(0, X)
    assert all(np.array_equal(a, b) for a, b in zip(one, blocks))


def _fields(r):
    return {k: v for k, v in vars(r).items() if k not in SCORE_KEYS + ('timing', 'timing_rank', 'launch_count')}


def _same(a, b):
    fa, fb = _fields(a), _fields(b)
    assert set(fa) == set(fb)
    for k in fa:
        x, y = np.asarray(fa[k]), np.asarray(fb[k])
        # NaN where an output is undefined (a Wald se of a singular information) is the same output
        assert np.array_equal(x, y, equal_nan=x.dtype.kind in 'fc'), k


@pytest.mark.parametrize("base_mode,n_perm,wald", [("full", 0, False), ("null", 0, True), ("full", 2, True),
                                                   ("null", 2, False)])
def test_fit_matrix_outputs_bit_identical_with_and_without_score(base_mode, n_perm, wald):
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng = 120, 40
    data, effLen, Xc, _ = make_problem(Nc, Ng, 3, 0, True, 3, seed=2)
    kw = dict(Xc=Xc, effLen=effLen, LRT_index=[0, 2], base_mode=base_mode, intercept_mode='gene', min_iter=240,
              max_iter=740, MC_size=2, n_eval=10, seed=3, n_perm=n_perm, wald=wald)
    X = _candidates(Nc, 5, 3)
    X[:, 4] = Xc[:, 1]                                            # a column model 0 fits in both modes
    r0 = fit_BRIE_matrix([x.copy() for x in data], **kw)
    r1 = fit_BRIE_matrix([x.copy() for x in data], score_X=X, **kw)
    _same(r0, r1)
    assert not any(hasattr(r0, k) for k in SCORE_KEYS)
    for k in SCORE_KEYS:
        assert getattr(r1, k).shape == (Ng, 5), k
    p = r1.pval_score
    assert ((p > 0) & (p <= 1)).all()
    assert (p[:, 4] == 1).all() and np.isnan(r1.score_z[:, 4]).all()   # a candidate equal to a fitted column
    assert np.isfinite(r1.score_z[:, :4]).mean() > 0.9


@pytest.mark.parametrize("base_mode,cell", [("full", False), ("null", False), ("full", True)])
def test_fitBRIE_outputs_bit_identical_with_and_without_score(base_mode, cell):
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 60
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=5)
    kw = dict(Xc=Xc, LRT_index=[1], base_mode=base_mode, intercept_mode='cell' if cell else 'gene',
              batch_size=100 * 20, seed=4, min_iter=300, max_iter=800, MC_size=2, n_eval=10, n_perm=2)
    a0, a1 = _adata(data, effLen), _adata(data, effLen)
    r0, r1 = fitBRIE(a0, **kw), fitBRIE(a1, score_X=_candidates(Nc, 3, 4), **kw)
    _same(r0, r1)
    assert set(a1.varm) - set(a0.varm) == set(SCORE_KEYS)
    _same_adata(a0, a1, skip=SCORE_KEYS)
    assert 'score' not in a0.uns['brie_param'] and a1.uns['brie_param']['score'] == 3
    assert a1.varm['score_z'].shape == (Ng, 3)


FIT = dict(intercept_mode='gene', min_iter=600, max_iter=2100, MC_size=2, n_eval=500, seed=5)


def test_score_calibration_and_power():
    from scipy.stats import kstest, pearsonr, spearmanr
    from brie_b200.models import fit_BRIE_matrix
    data, effLen, Xc, beta = _no_effect_problem(150, 120, 16, seed=12)
    rng = np.random.default_rng(3)
    rand = np.concatenate([rng.binomial(1, 0.5, (150, 16)), rng.normal(size=(150, 15))], axis=1)
    X = np.concatenate([Xc, rand], axis=1).astype(np.float32)
    res = fit_BRIE_matrix([d.copy() for d in data], effLen=effLen, score_X=X, **FIT)   # no covariates fitted
    full = fit_BRIE_matrix([d.copy() for d in data], Xc=Xc, effLen=effLen, LRT_index=[0], wald=True, **FIT)
    null, strong = beta == 0, beta > 0
    p, stat = res.pval_score[:, 0], res.score_z[:, 0] ** 2
    ks = kstest(p[null], "uniform")
    rej_null, rej_strong, rej_rand = (p[null] < 0.05).mean(), (p[strong] < 0.05).mean(), \
        (res.pval_score[:, 1:] < 0.05).mean()
    z2 = (full.cell_coeff[0] / full.cell_coeff_se[0]) ** 2
    gain = 2 * full.ELBO_gain[:, 0]
    ok = np.isfinite(stat)
    print("score: no-effect rejection at 0.05 %.3f (KS p %.3g), planted %.3f, random candidates %.3f; "
          "median planted stat %.2f vs no-effect 99th pct %.2f"
          % (rej_null, ks.pvalue, rej_strong, rej_rand, np.median(stat[strong]), np.percentile(stat[null], 99)))
    print("score stat vs Wald z^2: Spearman %.3f, Pearson %.3f; vs 2 ELBO_gain: Spearman %.3f, Pearson %.3f"
          % (spearmanr(stat[ok], z2[ok]).correlation, pearsonr(stat[ok], z2[ok])[0],
             spearmanr(stat[ok], gain[ok]).correlation, pearsonr(stat[ok], gain[ok])[0]))
    assert ok.all()
    assert rej_null <= 0.10 and ks.pvalue > 1e-3
    assert rej_strong >= 0.9
    assert rej_rand <= 0.10
    assert np.median(stat[strong]) > np.percentile(stat[null], 99)


def test_fitBRIE_chunked_equals_unchunked_and_fdr_score_is_pooled(monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    from brie_b200.models.model_wrap import fdr_bh
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=[], intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10, score_X=_candidates(Nc, 4, 9))
    ad_one = _adata(data, effLen)
    one = fitBRIE(ad_one, **kw)
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)         # chunks of 40, 40, 10 events
    ad = _adata(data, effLen)
    r = fitBRIE(ad, **kw)
    for k in SCORE_KEYS + ('cell_coeff',):
        assert np.array_equal(getattr(one, k), getattr(r, k), equal_nan=True), k
    for j in range(4):
        assert np.array_equal(r.fdr_score[:, j], fdr_bh(r.pval_score[:, j]))   # BH over all 90 events
    for k in SCORE_KEYS:
        assert np.array_equal(ad.varm[k], ad_one.varm[k], equal_nan=True), k


def test_fitBRIE_resume_with_score(tmp_path, monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    X = _candidates(Nc, 3, 2)
    kw = dict(Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10)
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)
    ref = fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "a"), score_X=X, **kw)
    real_fit, calls = mw.fit_BRIE_matrix, []

    def dying_fit(*a, **k):
        if len(calls) == 2:
            raise KeyboardInterrupt("job killed")
        calls.append(k['event_offset'])
        return real_fit(*a, **k)
    monkeypatch.setattr(mw, "fit_BRIE_matrix", dying_fit)
    with pytest.raises(KeyboardInterrupt):
        fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, score_X=X, **kw)
    calls2 = []
    monkeypatch.setattr(mw, "fit_BRIE_matrix", lambda *a, **k: (calls2.append(k['event_offset']), real_fit(*a, **k))[1])
    res = fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, score_X=X, **kw)
    assert calls2 == [80]
    for k in SCORE_KEYS + ('ELBO_gain', 'pval'):
        assert np.array_equal(np.asarray(getattr(ref, k)), np.asarray(getattr(res, k)), equal_nan=True), k
    # other candidates, or none, make another fit: nothing is reused
    for other in (X[:, ::-1].copy(), None):
        calls2.clear()
        fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, score_X=other, **kw)
        assert calls2 == [0, 40, 80]


def test_brie_quant_cli_with_score_file(tmp_path):
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
    sf = tmp_path / "score.tsv"
    with open(sf, "w") as f:
        f.write("cellID\tgroup\tRBFOX2\n")
        for i in np.random.default_rng(1).permutation(Nc):
            f.write("%s\t%d\t%.3f\n" % (cells[i], int(Xc[i, 0]), rng.normal()))
    out = str(tmp_path / "o" / "brie_quant.npz")
    args = [sys.executable, "-m", "brie_b200.bin.quant", "-i", inp, "-o", out, "--interceptMode", "gene",
            "--minIter", "300", "--maxIter", "800", "--MCsize", "2", "--minCount", "10", "--minUniqCount", "5",
            "--minCell", "5", "--scoreFile", str(sf)]
    p = subprocess.run(args, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
    assert p.returncode == 0, p.stderr[-3000:]
    ad = AnnDataLite.read_npz(out)
    G = ad.shape[1]
    for k in SCORE_KEYS:
        assert ad.varm[k].shape == (G, 2), k
    assert ad.uns['brie_param']['score'] == 2 and list(ad.uns['score_ids']) == ['group', 'RBFOX2']
    tsv = open(out.replace(".npz", ".brie_score.tsv")).read().splitlines()
    assert tsv[0].split("\t") == ['GeneID', 'group_score_z', 'group_pval_score', 'group_FDR_score',
                                  'RBFOX2_score_z', 'RBFOX2_pval_score', 'RBFOX2_FDR_score']
    assert len(tsv) == 1 + G
    ident = open(out.replace(".npz", ".brie_ident.tsv")).read().splitlines()[0].split("\t")
    assert not any('score' in c for c in ident)
    # a cell missing from the score file
    sf.write_text("\n".join(open(sf).read().splitlines()[:-1]) + "\n")
    p = subprocess.run(args, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
    assert p.returncode == 1 and "missing from --scoreFile" in p.stdout


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
rng = np.random.default_rng(0)
data, effLen, Xc, _ = make_lrt_problem(100, 130, seed=3)
ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]}, varm={'effLen': effLen})
r = fitBRIE(ad, Xc=Xc, LRT_index=[], intercept_mode='gene', batch_size=100 * 20, seed=4,
            min_iter=600, max_iter=1600, MC_size=2, n_eval=20, score_X=rng.normal(size=(100, 3)))
out['a'] = {k: getattr(r, k) for k in ('score_z', 'score_effect', 'pval_score', 'fdr_score', 'n_iter')}
data, effLen, Xc, Xg = make_problem(80, 64, 1, 2, False, 2, seed=6)
ad = AnnDataLite(X=data[0], layers={'spliced': data[0], 'unspliced': data[1]})
r = fitBRIE(ad, Xc=Xc, Xg=Xg, LRT_index=[], intercept_mode='cell', layer_keys=['spliced', 'unspliced'], seed=2,
            min_iter=360, max_iter=1860, MC_size=2, n_eval=20, score_X=rng.normal(size=(80, 2)))
out['c'] = {k: getattr(r, k) for k in ('score_z', 'score_effect', 'pval_score', 'fdr_score', 'n_iter')}
if world == 1 or dist.get_rank() == 0:
    pickle.dump(out, open(%(out)r, "wb"))
if world > 1:
    dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_fitBRIE_with_score_matches_single_gpu(tmp_path):
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
                   "--master-addr", "127.0.0.1", "--master-port", "29663", str(script)]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        res[world] = pickle.load(open(out, "rb"))
    for case in ('a', 'c'):
        for w in (1, 2):
            r = res[w][case]
            for j in range(r['pval_score'].shape[1]):
                assert np.array_equal(r['fdr_score'][:, j], fdr_bh(r['pval_score'][:, j])), (case, w)
        assert np.array_equal(res[1][case]['n_iter'], res[2][case]['n_iter'])
    # independent events (gene mode): each shard's events see the same fit
    a1, a2 = res[1]['a'], res[2]['a']
    assert np.allclose(a1['score_z'], a2['score_z'], rtol=1e-3, atol=1e-3, equal_nan=True)
    # shared per-cell parameters (cell mode): the all-reduced fit, up to its float32 reduction order
    c1, c2 = res[1]['c'], res[2]['c']
    assert np.allclose(c1['score_z'], c2['score_z'], rtol=1e-2, atol=1e-2, equal_nan=True)
