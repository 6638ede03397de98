"""GPU tests of the permutation null of the LRT (n_perm / brie-quant --nPerm): the observed outputs stay
bit-identical, the permuted refits match the oracle, the p-values are pooled over the whole fit, calibrated under
no effect, and survive chunking, resume, the CLI and event sharding over two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle.brie2_oracle as ob
from util import device_eps_provider, make_lrt_problem, make_problem

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

OBSERVED = ('Psi', 'Psi95CI', 'Z_std', 'loss_gene', 'ELBO_gain', 'pval', 'fdr', 'n_iter')


def _patched_oracle(seed, Nc, fn):
    orig = ob.OracleBRIE2.eps
    ob.OracleBRIE2.eps = lambda self, phase, step, S: device_eps_provider(
        seed, self.model_id, Nc, self.Ng, self.col_offset)(phase, step, S)
    try:
        return fn()
    finally:
        ob.OracleBRIE2.eps = orig


def _same_observed(r0, r1, keys=OBSERVED):
    for k in keys:
        assert np.array_equal(np.asarray(getattr(r0, k)), np.asarray(getattr(r1, k))), k


def _check_perm_outputs(res, Ng, T, B):
    from brie_b200.models.model_wrap import fdr_bh, perm_pvalue
    assert res.ELBO_gain_perm.shape == (Ng, T, B) and res.ELBO_gain_perm.dtype == np.float32
    assert np.isfinite(res.ELBO_gain_perm).all()
    assert np.array_equal(res.pval_perm, perm_pvalue(res.ELBO_gain, res.ELBO_gain_perm))
    for t in range(T):
        assert np.array_equal(res.fdr_perm[:, t], fdr_bh(res.pval_perm[:, t]))


@pytest.mark.parametrize("base_mode", ["full", "null"])
def test_fit_matrix_observed_outputs_bit_identical(base_mode):
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng = 120, 40
    data, effLen, Xc, Xg = make_problem(Nc, Ng, 2, 0, True, 3, seed=2)
    kw = dict(Xc=Xc, effLen=effLen, LRT_index=[0, 1], base_mode=base_mode, intercept_mode='gene', min_iter=240,
              max_iter=740, MC_size=2, n_eval=10, seed=3)
    r0 = fit_BRIE_matrix([x.copy() for x in data], **kw)
    r1 = fit_BRIE_matrix([x.copy() for x in data], n_perm=4, **kw)
    _same_observed(r0, r1)
    assert np.array_equal(r0.cell_coeff, r1.cell_coeff)
    assert not hasattr(r0, 'ELBO_gain_perm') and not hasattr(r0, 'pval_perm')
    _check_perm_outputs(r1, Ng, 2, 4)


def test_cell_mode_base_bit_identical_and_cell_mode_permuted_engines(monkeypatch):
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.models import model_wrap as mw
    Nc, Ng = 80, 36
    data, effLen, Xc, Xg = make_problem(Nc, Ng, 1, 2, False, 2, seed=6)
    kw = dict(Xc=Xc, Xg=Xg, intercept_mode='cell', LRT_index=None, min_iter=120, max_iter=620, MC_size=2, n_eval=10,
              seed=2)
    r0 = fit_BRIE_matrix([x.copy() for x in data], **kw)
    modes, real = [], mw.FitEngine

    def spy(*a, **k):
        modes.append((tuple(k['model_ids']), k['intercept_mode']))
        return real(*a, **k)
    monkeypatch.setattr(mw, "FitEngine", spy)
    r1 = fit_BRIE_matrix([x.copy() for x in data], n_perm=4, **kw)
    _same_observed(r0, r1)
    assert np.array_equal(r0.gene_coeff, r1.gene_coeff) and np.array_equal(r0.intercept, r1.intercept)
    # base alone (cell), refit (gene), then 4 permuted full models of the base's layout, one per engine
    assert modes == [((0,), 'cell'), ((1,), 'gene')] + [((2 + b,), 'cell') for b in range(4)]
    _check_perm_outputs(r1, Ng, 1, 4)


def _adata(data, effLen):
    from brie_b200.utils.anndata_lite import AnnDataLite
    return AnnDataLite(X=data[0] + data[1] + data[2],
                       layers={'isoform1': data[0].copy(), 'isoform2': data[1].copy(), 'ambiguous': data[2].copy()},
                       varm={'effLen': effLen})


def test_fitBRIE_chunked_bit_identical_and_pooled_over_all_events(monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10)
    ad_one = _adata(data, effLen)
    one = fitBRIE(ad_one, n_perm=3, **kw)                                       # one chunk
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)         # chunks of 40, 40, 10 events
    r0 = fitBRIE(_adata(data, effLen), **kw)
    ad = _adata(data, effLen)
    r1 = fitBRIE(ad, n_perm=3, **kw)
    _same_observed(r0, r1, OBSERVED + ('Z_loc', 'losses', 'cell_coeff', 'sigma', 'intercept'))
    # the pooled null spans every event of the fit, not one chunk's
    _check_perm_outputs(r1, Ng, 1, 3)
    assert np.array_equal(one.ELBO_gain_perm, r1.ELBO_gain_perm) and np.array_equal(one.pval_perm, r1.pval_perm)
    for k in ('ELBO_gain_perm', 'pval_perm', 'fdr_perm'):
        assert np.array_equal(ad.varm[k], getattr(r1, k)) and np.array_equal(ad_one.varm[k], getattr(one, k)), k
    assert ad.uns['brie_param']['n_perm'] == 3


def test_permuted_refit_matches_oracle():
    """ELBO_gain_perm[:, t, b] = loss_gene(null refit t) - loss_gene(full model with column t permuted), the oracle
    fitting that design with the permuted model's id and the device's noise."""
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.models.model_wrap import perm_indices, perm_model_id
    Nc, Ng, seed, B = 90, 24, 1, 3
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=2)
    kw = dict(effLen=effLen, LRT_index=[1], intercept_mode='gene', min_iter=120, max_iter=120, MC_size=2, n_eval=10)
    res = fit_BRIE_matrix([x.copy() for x in data], Xc=Xc, seed=seed, n_perm=B, **kw)
    t, b = 0, 2
    Xp = Xc.copy()
    Xp[:, 1] = Xc[perm_indices(seed, t, b, Nc), 1]

    def run():
        ref = ob.oracle_fit_matrix([x.copy() for x in data], Xc=Xc, dtype=np.float32, seed=seed, **kw)
        d = [np.array(x, np.float32) for x in data]
        ob.add_pseudo_count(d, np.float32(0.01))
        m = ob.OracleBRIE2(Nc, Ng, 2, 0, effLen, None, 'gene', None, dtype=np.float32, seed=seed,
                           model_id=perm_model_id(t, b, 1, B))
        m.fit(d, Xc=Xp, Xg=np.ones((Ng, 0), np.float32), min_iter=120, max_iter=120, MC_size=2, n_eval=10)
        return ref, m
    ref, m = _patched_oracle(seed, Nc, run)
    want = ref.tests[0].loss_gene - m.loss_gene
    err = np.abs(res.ELBO_gain_perm[:, t, b] - want)
    print("permuted refit gain vs oracle: max %.2e" % err.max())
    assert err.max() < 2e-2
    assert np.abs(res.ELBO_gain - ref.ELBO_gain).max() < 2e-2


def _no_effect_problem(Nc, Ng, n_strong, seed):
    """make_lrt_problem's generator with the covariate effect zero on all but the last `n_strong` events."""
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


def test_permutation_pvalues_calibrated_under_no_effect():
    from scipy.stats import kstest
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng, B = 150, 120, 4
    data, effLen, Xc, beta = _no_effect_problem(Nc, Ng, 16, seed=12)
    res = fit_BRIE_matrix(data, Xc=Xc, effLen=effLen, LRT_index=[0], intercept_mode='gene', min_iter=600,
                          max_iter=2100, MC_size=2, n_eval=50, seed=5, n_perm=B)
    null, strong = beta == 0, beta > 0
    pp, pc = res.pval_perm[:, 0], res.pval[:, 0]
    ks = kstest(pp[null], "uniform")
    print("no-effect events (%d): rejection at 0.05 -- chi2 %.3f, permutation %.3f; KS vs uniform p %.3g"
          % (null.sum(), (pc[null] < 0.05).mean(), (pp[null] < 0.05).mean(), ks.pvalue))
    print("planted effects (%d): rejection at 0.05 -- chi2 %.3f, permutation %.3f"
          % (strong.sum(), (pc[strong] < 0.05).mean(), (pp[strong] < 0.05).mean()))
    assert ks.pvalue > 1e-3
    assert (pp[strong] < 0.05).mean() >= 0.9


def test_fitBRIE_resume_with_permutations(tmp_path, monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    kw = dict(Xc=Xc, LRT_index=None, intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10, n_perm=2)
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
    for k in OBSERVED + ('ELBO_gain_perm', 'pval_perm', 'fdr_perm'):
        assert np.array_equal(np.asarray(getattr(ref, k)), np.asarray(getattr(res, k))), k
    # another n_perm is another fit: nothing is reused
    calls2.clear()
    fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, **dict(kw, n_perm=3))
    assert calls2 == [0, 40, 80]


def test_brie_quant_cli_with_nperm(tmp_path):
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
    cf = tmp_path / "cells.tsv"
    with open(cf, "w") as f:
        f.write("cellID\tgroup\n")
        for i in range(Nc):
            f.write("%s\t%d\n" % (cells[i], int(Xc[i, 0])))
    out = str(tmp_path / "o" / "brie_quant.npz")
    p = subprocess.run([sys.executable, "-m", "brie_b200.bin.quant", "-i", inp, "-c", str(cf), "-o", out,
                        "--LRTindex", "All", "--interceptMode", "gene", "--minIter", "300", "--maxIter", "800",
                        "--MCsize", "2", "--minCount", "10", "--minUniqCount", "5", "--minCell", "5", "--nPerm", "3"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
    assert p.returncode == 0, p.stderr[-3000:]
    ad = AnnDataLite.read_npz(out)
    G = ad.shape[1]
    assert ad.varm['ELBO_gain_perm'].shape == (G, 1, 3)
    assert ad.varm['pval_perm'].shape == (G, 1) and ad.varm['fdr_perm'].shape == (G, 1)
    assert ad.uns['brie_param']['n_perm'] == 3
    tsv = open(out.replace(".npz", ".brie_ident.tsv")).read().splitlines()
    hdr = tsv[0].split("\t")
    assert hdr == ['GeneID', 'n_counts', 'n_counts_uniq', 'cdr', 'intercept', 'sigma', 'group_ceoff',
                   'group_ELBO_gain', 'group_pval', 'group_FDR', 'group_pval_perm', 'group_FDR_perm']
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
            min_iter=600, max_iter=1600, MC_size=2, n_eval=20, n_perm=3)
out['a'] = dict(gain=r.ELBO_gain, gp=r.ELBO_gain_perm, pp=r.pval_perm, n_iter=r.n_iter)
data, effLen, Xc, Xg = make_problem(80, 64, 1, 2, False, 2, seed=6)
ad = AnnDataLite(X=data[0], layers={'spliced': data[0], 'unspliced': data[1]})
r = fitBRIE(ad, Xc=Xc, Xg=Xg, LRT_index=None, intercept_mode='cell', layer_keys=['spliced', 'unspliced'], seed=2,
            min_iter=360, max_iter=1860, MC_size=2, n_eval=20, n_perm=2)
out['c'] = dict(gain=r.ELBO_gain, gp=r.ELBO_gain_perm, pp=r.pval_perm, n_iter=r.n_iter)
if world == 1 or dist.get_rank() == 0:
    pickle.dump(out, open(%(out)r, "wb"))
if world > 1:
    dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_fitBRIE_with_permutations_matches_single_gpu(tmp_path):
    import pickle
    from brie_b200.models.model_wrap import perm_pvalue
    res = {}
    for world in (1, 2):
        out = str(tmp_path / ("w%d.pkl" % world))
        script = tmp_path / ("worker%d.py" % world)
        script.write_text(WORKER % dict(root=ROOT, out=out))
        if world == 1:
            cmd = [sys.executable, str(script)]
        else:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                   "--master-addr", "127.0.0.1", "--master-port", "29659", str(script)]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        res[world] = pickle.load(open(out, "rb"))
    for case in ('a', 'c'):
        for w in (1, 2):
            r = res[w][case]
            assert np.array_equal(r['pp'], perm_pvalue(r['gain'], r['gp'])), (case, w)    # pooled over all ranks
        assert res[1][case]['gp'].shape == res[2][case]['gp'].shape
        assert np.array_equal(res[1][case]['n_iter'], res[2][case]['n_iter'])
    a1, a2 = res[1]['a'], res[2]['a']
    # independent events: the tolerance of the observed gains in test_gpu_multi
    assert np.abs(a1['gp'] - a2['gp']).max() < 1e-3 and np.abs(a1['gain'] - a2['gain']).max() < 1e-3
