"""GPU tests of the joint tests of groups of covariates (LRT_groups, wald_groups, score_groups): the cross-term kernel
against its float64 restatement on the engine's own state, determinism and pair blocks, a group refit against the
oracle, that nothing else moves, calibration and power on a 3-level categorical, chunking, resume, the CLI and event
sharding over two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import groups_ref
import oracle.brie2_oracle as ob
from oracle.brie2_oracle import add_pseudo_count
from test_gpu_perm import _patched_oracle
from test_gpu_wald import CASES, _adata
from util import make_lrt_problem, make_problem

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GROUP_KEYS = ('ELBO_gain_group', 'pval_group', 'fdr_group', 'wald_stat_group', 'pval_wald_group', 'fdr_wald_group',
              'score_stat_group', 'pval_score_group', 'fdr_score_group')
GROUPS = [[0, 1], list(range(2, 9)), list(range(20, 60))]          # 2, 7 and 40 columns: 1 + 21 + 780 pairs


def _candidates(Nc, J, seed):
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(Nc, J)).astype(np.float32)
    X[:, ::3] = rng.binomial(1, 0.4, size=(Nc, len(range(0, J, 3))))
    return X


def _check_engine(eng):
    from brie_b200.engine import group_pairs
    X = _candidates(eng.Nc, 80, 5)
    pairs = group_pairs(GROUPS)
    assert len(pairs) == 1 + 21 + 780
    for m in range(eng.M):
        got = eng.score_cross(m, X, pairs)
        want = groups_ref.engine_cross(eng, m, X, pairs)
        # sums that cancel to a small fraction of their terms' absolute sum `mag` differ by the float64 rounding of
        # two summation orders, up to ~ n_cells x 1.1e-16 x mag: a floor of 1e-13 x mag for those
        mag = groups_ref.engine_cross(eng, m, np.abs(X), pairs)            # sum of |terms| (w >= 0)
        err = np.abs(got - want)
        rel = err / np.maximum(np.abs(want), 1e-4 * mag + 1e-300)
        print("cross terms vs float64 restatement: max rel %.2e over %d entries (max err / mag %.2e)"
              % (rel.max(initial=0), want.size, (err / np.maximum(mag, 1e-300)).max(initial=0)))
        assert got.shape == (eng.Ng, len(pairs)) and (err <= 1e-9 * np.abs(want) + 1e-13 * mag).all()
        assert np.array_equal(got, eng.score_cross(m, X, pairs))          # repeated calls: bit-identical


@pytest.mark.parametrize("Kc,Kg,mode,masks", CASES)
def test_cross_kernel_matches_the_float64_restatement(Kc, Kg, mode, masks):
    from brie_b200.engine import FitEngine
    Nc, Ng = 300, 130
    data, effLen, Xc, Xg = make_problem(Nc, Ng, Kc, Kg, True, 3, seed=4)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, Xg=Xg, masks=masks, intercept=0 if mode == 'None' else None,
                    intercept_mode=mode, MC_size=2, seed=3, trace_cap=8)
    eng.init_params()
    eng.begin_stage(0.02)
    eng.run_steps(80)
    _check_engine(eng)


def test_cross_terms_after_gathered_extension_rounds():
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
    _check_engine(eng)


def test_pair_blocks_give_the_same_bits(monkeypatch):
    """Pairs split into blocks (SCORE_BLOCK_BYTES), and a device X, give the bits of one call."""
    import brie_b200.engine as E
    from brie_b200.engine import FitEngine, group_pairs
    data, effLen, Xc, _ = make_problem(300, 130, 3, 0, True, 3, seed=4)
    add_pseudo_count(data, np.float32(0.01))
    eng = FitEngine(data, effLen=effLen, Xc=Xc, MC_size=2, seed=3, trace_cap=8)
    eng.init_params(); eng.begin_stage(0.02); eng.run_steps(40)
    X = _candidates(300, 80, 1)
    pairs = group_pairs(GROUPS)
    one = eng.score_cross(0, X, pairs)
    monkeypatch.setattr(E, "SCORE_BLOCK_BYTES", 200_000)                      # blocks of a few pairs
    blocks = eng.score_cross(0, torch.from_numpy(X).to(eng.device), pairs)
    assert np.array_equal(one, blocks)


def test_group_refit_matches_oracle():
    """ELBO_gain_group[:, 0] = loss_gene(full model without the group) - loss_gene(full model), the oracle fitting the
    reduced design with the group model's id and the device's noise."""
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.models.model_wrap import group_model_id
    Nc, Ng, seed = 90, 24, 1
    data, effLen, Xc, _ = make_problem(Nc, Ng, 3, 0, True, 3, seed=2)
    kw = dict(effLen=effLen, LRT_index=[1], intercept_mode='gene', min_iter=120, max_iter=120, MC_size=2, n_eval=10)
    res = fit_BRIE_matrix([x.copy() for x in data], Xc=Xc, seed=seed, LRT_groups=[[0, 2]], **kw)

    def run():
        ref = ob.oracle_fit_matrix([x.copy() for x in data], Xc=Xc, dtype=np.float32, seed=seed, **kw)
        d = [np.array(x, np.float32) for x in data]
        ob.add_pseudo_count(d, np.float32(0.01))
        m = ob.OracleBRIE2(Nc, Ng, 1, 0, effLen, None, 'gene', None, dtype=np.float32, seed=seed,
                           model_id=group_model_id(0, 1, 0))
        m.fit(d, Xc=Xc[:, [1]], Xg=np.ones((Ng, 0), np.float32), min_iter=120, max_iter=120, MC_size=2, n_eval=10)
        return ref, m
    ref, m = _patched_oracle(seed, Nc, run)
    assert np.abs(res.loss_gene - ref.loss_gene).max() <= 1e-4 * np.abs(ref.loss_gene).max()
    lg_group = res.ELBO_gain_group[:, 0].astype(np.float64) + res.loss_gene
    err = np.abs(lg_group - m.loss_gene)
    print("group refit loss_gene vs oracle: max %.2e (bar %.2e)" % (err.max(), 1e-4 * np.abs(m.loss_gene).max()))
    assert err.max() <= 1e-4 * np.abs(m.loss_gene).max()


def _same_adata(a, b, skip=()):
    """Every container entry but `skip` equal; NaN where an output is undefined (a Wald se of a singular
    information) is the same output."""
    for grp in ('obsm', 'varm', 'layers'):
        da, db = getattr(a, grp), getattr(b, grp)
        assert set(da) - set(skip) == set(db) - set(skip), grp
        for k in set(da) - set(skip):
            x, y = np.asarray(da[k]), np.asarray(db[k])
            assert np.array_equal(x, y, equal_nan=x.dtype.kind in 'fc'), (grp, k)
    assert np.array_equal(np.asarray(a.var['loss_gene']), np.asarray(b.var['loss_gene']))


def _fields(r):
    return {k: v for k, v in vars(r).items() if k not in GROUP_KEYS + ('timing', 'timing_rank', 'launch_count')}


def _same(a, b):
    fa, fb = _fields(a), _fields(b)
    assert set(fa) == set(fb)
    for k in fa:
        x, y = np.asarray(fa[k]), np.asarray(fb[k])
        assert np.array_equal(x, y, equal_nan=x.dtype.kind in 'fc'), k


@pytest.mark.parametrize("base_mode,n_perm,wald,cell", [("full", 0, False, False), ("null", 2, True, False),
                                                        ("full", 2, True, True)])
def test_fit_matrix_outputs_bit_identical_with_and_without_groups(base_mode, n_perm, wald, cell):
    from brie_b200.models import fit_BRIE_matrix
    Nc, Ng = 120, 40
    data, effLen, Xc, _ = make_problem(Nc, Ng, 3, 0, True, 3, seed=2)
    kw = dict(Xc=Xc, effLen=effLen, LRT_index=[0, 2], base_mode=base_mode, intercept_mode='cell' if cell else 'gene',
              min_iter=240, max_iter=740, MC_size=2, n_eval=10, seed=3, n_perm=n_perm, wald=wald,
              score_X=_candidates(Nc, 5, 3))
    fitted = [0, 1, 2] if base_mode == 'full' else [1]
    groups = dict(LRT_groups=[[0, 2], [1]] if base_mode == 'full' else [[0, 2], [2]],
                  wald_groups=[fitted, fitted[:1]], score_groups=[[0, 1, 2], [3, 4], [4]])
    r0 = fit_BRIE_matrix([x.copy() for x in data], **kw)
    for name, g in groups.items():
        r1 = fit_BRIE_matrix([x.copy() for x in data], **{name: g}, **kw)
        _same(r0, r1)
    r1 = fit_BRIE_matrix([x.copy() for x in data], **groups, **kw)
    _same(r0, r1)
    assert not any(hasattr(r0, k) for k in GROUP_KEYS)
    for k, H in zip(GROUP_KEYS, [2] * 6 + [3] * 3):
        assert getattr(r1, k).shape == (Ng, H), k
    for k in ('pval_group', 'pval_wald_group', 'pval_score_group'):
        p = getattr(r1, k)
        assert ((p > 0) & (p <= 1)).all(), k
    assert np.isfinite(r1.wald_stat_group).mean() > 0.9 and np.isfinite(r1.score_stat_group).mean() > 0.9
    # a singleton group is the one-column test
    assert np.allclose(r1.score_stat_group[:, 2], r1.score_z[:, 4] ** 2, rtol=1e-9, equal_nan=True)


@pytest.mark.parametrize("base_mode,cell", [("full", False), ("null", False), ("full", True)])
def test_fitBRIE_outputs_bit_identical_with_and_without_groups(base_mode, cell):
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 60
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=5)
    kw = dict(Xc=Xc, LRT_index=[1], base_mode=base_mode, intercept_mode='cell' if cell else 'gene',
              batch_size=100 * 20, seed=4, min_iter=300, max_iter=800, MC_size=2, n_eval=10, n_perm=2, wald=True,
              score_X=_candidates(Nc, 3, 4))
    groups = dict(LRT_groups=[[0, 1]] if base_mode == 'full' else [[1]], wald_groups=[[0]],
                  score_groups=[[0, 1, 2]])
    a0, a1 = _adata(data, effLen), _adata(data, effLen)
    r0, r1 = fitBRIE(a0, **kw), fitBRIE(a1, **groups, **kw)
    _same(r0, r1)
    assert set(a1.varm) - set(a0.varm) == set(GROUP_KEYS)
    _same_adata(a0, a1, skip=GROUP_KEYS)
    for k, g in groups.items():
        assert k not in a0.uns['brie_param'] and a1.uns['brie_param'][k] == g


def _categorical_problem(Nc, Ng, n_strong, seed):
    """A 3-level categorical (2 indicator columns) with no effect on all but the last `n_strong` events (the
    generator of test_gpu_wald's no-effect design)."""
    rng = np.random.default_rng(seed)
    level = rng.integers(0, 3, Nc)
    Xc = np.stack([level == 1, level == 2], axis=1).astype(np.float32)
    beta = np.zeros((Ng, 2))
    beta[Ng - n_strong:] = [2.0, -2.0]
    z = rng.normal(0, 1.0, Ng)[None, :] + Xc @ beta.T + rng.normal(0, 0.5, (Nc, Ng))
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
    return [c.astype(np.float32) for c in (c1, c2, c3)], effLen, Xc, beta[:, 0] != 0


FIT = dict(intercept_mode='gene', min_iter=600, max_iter=2100, MC_size=2, n_eval=500, seed=5)


def test_group_calibration_and_power():
    from brie_b200.models import fit_BRIE_matrix
    data, effLen, Xc, strong = _categorical_problem(150, 120, 16, seed=12)
    res = fit_BRIE_matrix([d.copy() for d in data], Xc=Xc, effLen=effLen, LRT_index=[], LRT_groups=[[0, 1]],
                          wald_groups=[[0, 1]], **FIT)
    sc = fit_BRIE_matrix([d.copy() for d in data], effLen=effLen, score_X=Xc, score_groups=[[0, 1]], **FIT)
    null = ~strong
    for name, p in (("group LRT", res.pval_group[:, 0]), ("joint Wald", res.pval_wald_group[:, 0]),
                    ("joint score", sc.pval_score_group[:, 0])):
        rej_null, rej_strong = (p[null] < 0.05).mean(), (p[strong] < 0.05).mean()
        print("%s: no-effect rejection at 0.05 %.3f (%d events), planted %.3f (%d events)"
              % (name, rej_null, null.sum(), rej_strong, strong.sum()))
        assert rej_null <= 0.10, name
        assert rej_strong >= 0.9, name


def test_fitBRIE_chunked_equals_unchunked_and_group_fdrs_are_pooled(monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    from brie_b200.models.model_wrap import fdr_bh
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=7)
    kw = dict(Xc=Xc, LRT_index=[0], intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10, score_X=_candidates(Nc, 4, 9), LRT_groups=[[0, 1], [1]], wald_groups=[[0, 1]],
              score_groups=[[0, 1, 2], [3, 1]])
    ad_one = _adata(data, effLen)
    one = fitBRIE(ad_one, **kw)
    monkeypatch.setattr(mw, "_device_event_budget", lambda *a, **k: 45)         # chunks of 40, 40, 10 events
    ad = _adata(data, effLen)
    r = fitBRIE(ad, **kw)
    # events are independent and keyed by global ids: chunks give the LRT gains' bits, and so the group gains'
    assert np.array_equal(one.ELBO_gain, r.ELBO_gain)
    for k in GROUP_KEYS:
        assert np.array_equal(getattr(one, k), getattr(r, k), equal_nan=True), k
    for _, pk, fk in (GROUP_KEYS[0:3], GROUP_KEYS[3:6], GROUP_KEYS[6:9]):
        for j in range(getattr(r, pk).shape[1]):
            assert np.array_equal(getattr(r, fk)[:, j], fdr_bh(getattr(r, pk)[:, j]))   # BH over all 90 events
    for k in GROUP_KEYS:
        assert np.array_equal(ad.varm[k], getattr(r, k), equal_nan=True), k


def test_fitBRIE_resume_with_groups(tmp_path, monkeypatch):
    import brie_b200.models.model_wrap as mw
    from brie_b200.models import fitBRIE
    Nc, Ng = 100, 90
    data, effLen, Xc, _ = make_lrt_problem(Nc, Ng, seed=7)
    X = _candidates(Nc, 3, 2)
    kw = dict(Xc=Xc, LRT_index=[], intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=300, max_iter=800,
              MC_size=2, n_eval=10, score_X=X, LRT_groups=[[0]], wald_groups=[[0]], score_groups=[[0, 2]])
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
    for k in GROUP_KEYS:
        assert np.array_equal(np.asarray(getattr(ref, k)), np.asarray(getattr(res, k)), equal_nan=True), k
    # other groups, or none, make another fit: nothing is reused
    for other in (dict(score_groups=[[1, 2]]), dict(LRT_groups=None)):
        calls2.clear()
        fitBRIE(_adata(data, effLen), out_dir=str(tmp_path / "b"), resume=True, **dict(kw, **other))
        assert calls2 == [0, 40, 80]


def test_brie_quant_cli_with_group_options(tmp_path):
    from brie_b200.utils import io_utils
    from brie_b200.utils.anndata_lite import AnnDataLite
    Nc, Ng = 120, 60
    data, effLen, Xc, _ = make_problem(Nc, Ng, 3, 0, True, 3, seed=21)
    eff3 = np.zeros((Ng, 2, 3), np.float32)
    eff3[:, 0, :], eff3[:, 1, :] = effLen[:, :3], effLen[:, 3:]
    cells = ["cell%03d" % i for i in range(Nc)]
    inp = str(tmp_path / "counts.npz")
    io_utils.write_npz_counts(inp, {'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]}, eff3, cells,
                              ["g%03d" % i for i in range(Ng)])
    cf, sf = tmp_path / "cells.tsv", tmp_path / "score.tsv"
    rng = np.random.default_rng(0)
    with open(cf, "w") as f, open(sf, "w") as g:
        f.write("cellID\ta\tb\tc\n")
        g.write("cellID\tRBFOX2\trs1\n")
        for i in range(Nc):
            f.write("%s\t%.4f\t%.4f\t%.4f\n" % ((cells[i],) + tuple(Xc[i])))
            g.write("%s\t%.3f\t%d\n" % (cells[i], rng.normal(), rng.integers(0, 3)))
    out = str(tmp_path / "o" / "brie_quant.npz")
    args = [sys.executable, "-m", "brie_b200.bin.quant", "-i", inp, "-o", out, "-c", str(cf), "--interceptMode",
            "gene", "--minIter", "300", "--maxIter", "800", "--MCsize", "2", "--minCount", "10", "--minUniqCount", "5",
            "--minCell", "5", "--LRTindex", "0", "--LRTgroups", "1,2;0,2", "--waldGroups", "0,1,2",
            "--scoreFile", str(sf), "--scoreGroups", "0,1"]
    p = subprocess.run(args, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, PYTHONPATH=ROOT))
    assert p.returncode == 0, p.stderr[-3000:]
    ad = AnnDataLite.read_npz(out)
    G = ad.shape[1]
    for k, H in zip(GROUP_KEYS, [2] * 3 + [1] * 6):
        assert ad.varm[k].shape == (G, H), k
    assert ad.uns['brie_param']['LRT_groups'] == [[1, 2], [0, 2]]
    ident = open(out.replace(".npz", ".brie_ident.tsv")).read().splitlines()
    assert ident[0].split("\t")[-8:] == ['b+c_ELBO_gain_group', 'b+c_pval_group', 'b+c_FDR_group',
                                         'a+c_ELBO_gain_group', 'a+c_pval_group', 'a+c_FDR_group',
                                         'a+b+c_pval_wald_group', 'a+b+c_FDR_wald_group']
    assert len(ident) == 1 + G
    score = open(out.replace(".npz", ".brie_score.tsv")).read().splitlines()[0].split("\t")
    assert score[-3:] == ['RBFOX2+rs1_score_stat_group', 'RBFOX2+rs1_pval_score_group', 'RBFOX2+rs1_FDR_score_group']


WORKER = r'''
import os, sys, pickle
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
from util import make_lrt_problem, make_problem
from brie_b200.models import fitBRIE
from brie_b200.utils.anndata_lite import AnnDataLite
KEYS = %(keys)r
world = int(os.environ.get("WORLD_SIZE", "1"))
if world > 1:
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
out = {}
rng = np.random.default_rng(0)
data, effLen, Xc, _ = make_problem(100, 130, 2, 0, True, 3, seed=3)
ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]}, varm={'effLen': effLen})
r = fitBRIE(ad, Xc=Xc, LRT_index=[], intercept_mode='gene', batch_size=100 * 20, seed=4, min_iter=600, max_iter=1600,
            MC_size=2, n_eval=20, score_X=rng.normal(size=(100, 3)), LRT_groups=[[0, 1]], wald_groups=[[0, 1]],
            score_groups=[[0, 2]])
out['a'] = {k: getattr(r, k) for k in KEYS}
data, effLen, Xc, Xg = make_problem(80, 64, 2, 2, False, 2, seed=6)
ad = AnnDataLite(X=data[0], layers={'spliced': data[0], 'unspliced': data[1]})
r = fitBRIE(ad, Xc=Xc, Xg=Xg, LRT_index=[], intercept_mode='cell', layer_keys=['spliced', 'unspliced'], seed=2,
            min_iter=360, max_iter=1860, MC_size=2, n_eval=20, score_X=rng.normal(size=(80, 2)), LRT_groups=[[0, 1]],
            wald_groups=[[0, 1]], score_groups=[[0, 1]])
out['c'] = {k: getattr(r, k) for k in KEYS}
if world == 1 or dist.get_rank() == 0:
    pickle.dump(out, open(%(out)r, "wb"))
if world > 1:
    dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_fitBRIE_with_groups_matches_single_gpu(tmp_path):
    import pickle
    from brie_b200.models.model_wrap import fdr_bh
    res = {}
    for world in (1, 2):
        out = str(tmp_path / ("w%d.pkl" % world))
        script = tmp_path / ("worker%d.py" % world)
        script.write_text(WORKER % dict(root=ROOT, out=out, keys=GROUP_KEYS))
        if world == 1:
            cmd = [sys.executable, str(script)]
        else:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                   "--master-addr", "127.0.0.1", "--master-port", "29667", str(script)]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        res[world] = pickle.load(open(out, "rb"))
    for case in ('a', 'c'):
        for w in (1, 2):
            r = res[w][case]
            for pk, fk in (('pval_group', 'fdr_group'), ('pval_wald_group', 'fdr_wald_group'),
                           ('pval_score_group', 'fdr_score_group')):
                for j in range(r[pk].shape[1]):
                    assert np.array_equal(r[fk][:, j], fdr_bh(r[pk][:, j])), (case, w, pk)
    # independent events (gene mode): each shard's events see the same fit
    a1, a2 = res[1]['a'], res[2]['a']
    for k in ('wald_stat_group', 'score_stat_group', 'ELBO_gain_group'):
        assert np.allclose(a1[k], a2[k], rtol=1e-3, atol=1e-3, equal_nan=True), k
    # shared per-cell parameters (cell mode): the all-reduced fit, up to its float32 reduction order
    c1, c2 = res[1]['c'], res[2]['c']
    for k in ('wald_stat_group', 'score_stat_group'):
        assert np.allclose(c1[k], c2[k], rtol=1e-2, atol=1e-2, equal_nan=True), k
