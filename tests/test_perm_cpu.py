"""Permutation null of the LRT (n_perm / brie-quant --nPerm): the host side -- pooled p-values, permutations,
engine plan, refusals, CLI and result table.  No GPU needed."""
import os
import subprocess
import sys

import numpy as np
import pytest

from brie_b200.models.model_wrap import (_engine_plan, check_n_perm, fdr_bh, _set_perm_outputs, perm_indices,
                                         perm_model_id, perm_pvalue, fit_BRIE_matrix, fitBRIE)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _brute_pvalue(G, Gp):
    Ng, T, B = Gp.shape
    out = np.zeros((Ng, T))
    for g in range(Ng):
        for t in range(T):
            n = 0
            for g2 in range(Ng):
                for b in range(B):
                    n += Gp[g2, t, b] >= G[g, t]
            out[g, t] = (1 + n) / (1 + Ng * B)
    return out


@pytest.mark.parametrize("Ng,T,B", [(13, 2, 3), (9, 1, 1), (1, 3, 1), (20, 1, 5)])
def test_pval_perm_matches_double_loop_with_ties(Ng, T, B):
    rng = np.random.default_rng(Ng * 100 + T * 10 + B)
    # small integer grid: many ties between observed and null gains and inside the null
    G = rng.integers(-3, 4, (Ng, T)).astype(np.float32)
    Gp = rng.integers(-3, 4, (Ng, T, B)).astype(np.float32)
    assert np.array_equal(perm_pvalue(G, Gp), _brute_pvalue(G, Gp))
    G = rng.standard_normal((Ng, T)).astype(np.float32)
    Gp = rng.standard_normal((Ng, T, B)).astype(np.float32)
    Gp[0, 0, 0] = G[-1, 0]                                     # an exact tie
    G[0, -1] = np.nan                                          # NaN compares False both ways
    Gp[-1, -1, -1] = np.nan
    assert np.array_equal(perm_pvalue(G, Gp), _brute_pvalue(G, Gp))


def test_fdr_perm_is_bh_per_column_over_all_events():
    class R:
        pass
    rng = np.random.default_rng(1)
    r = R()
    r.ELBO_gain = rng.standard_normal((30, 2)).astype(np.float32)
    r.ELBO_gain_perm = rng.standard_normal((30, 2, 4)).astype(np.float32)
    _set_perm_outputs(r)
    assert r.pval_perm.shape == (30, 2) and r.fdr_perm.shape == (30, 2)
    assert np.array_equal(r.pval_perm, perm_pvalue(r.ELBO_gain, r.ELBO_gain_perm))
    for t in range(2):
        assert np.array_equal(r.fdr_perm[:, t], fdr_bh(r.pval_perm[:, t]))


def test_perm_indices_deterministic_and_independent_of_chunk_and_rank():
    p = perm_indices(7, 1, 2, 1000)
    assert np.array_equal(np.sort(p), np.arange(1000))
    assert np.array_equal(p, perm_indices(7, 1, 2, 1000))
    assert np.array_equal(p, np.random.default_rng((7, 2, 2)).permutation(1000))
    # a fresh process (another rank) draws the same permutation
    code = "from brie_b200.models.model_wrap import perm_indices; print(perm_indices(7, 1, 2, 1000).tolist())"
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300,
                         env=dict(os.environ, PYTHONPATH=ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    assert eval(out.stdout) == p.tolist()
    # different test positions, replicates and seeds differ
    others = [perm_indices(7, 0, 2, 1000), perm_indices(7, 1, 3, 1000), perm_indices(8, 1, 2, 1000)]
    assert all(not np.array_equal(p, o) for o in others)


def _plan_args(Kc, tested, full):
    base = list(range(Kc)) if full else [k for k in range(Kc) if k not in tested]
    tests = [[k for k in range(Kc) if k != i] for i in tested] if full else [base + [i] for i in tested]
    return base, tests


@pytest.mark.parametrize("Kc,tested,full,cell,max_models", [
    (1, [0], True, False, None), (3, [0, 2], True, False, None), (3, [0, 2], True, True, None),
    (40, list(range(40)), True, False, None), (4, [1, 2, 3], False, False, None), (4, [1, 2, 3], False, True, None),
    (2, [0, 1], True, False, 2)])
def test_engine_plan_with_permutations(Kc, tested, full, cell, max_models):
    base, tests = _plan_args(Kc, tested, full)
    mode = 'cell' if cell else 'gene'
    kw = {} if max_models is None else dict(max_models=max_models)
    ref = _engine_plan(base, tests, cell, mode, **kw)
    assert _engine_plan(base, tests, cell, mode, n_perm=0, tested=tested, n_cols=Kc, full=full, **kw) == ref
    T, B = len(tested), 5
    plan = _engine_plan(base, tests, cell, mode, n_perm=B, tested=tested, n_cols=Kc, full=full, **kw)
    assert plan[:len(ref)] == ref                                   # observed engines untouched
    extra = plan[len(ref):]
    size = min(max(len(p[1]) for p in ref), max_models or 32)
    assert extra and all(len(p[1]) <= size for p in extra)
    ids = [i for p in plan for i in p[1]]
    assert len(ids) == len(set(ids)) and max(ids) < 4096
    assert sorted(i for p in extra for i in p[1]) == list(range(1 + T, 1 + T + T * B))
    for masks, ids_e, mode_e in extra:
        assert mode_e == (mode if full else 'gene')                 # full + cell -> cell; null base -> gene
        assert len(masks) == len(ids_e)
        for j, (mk, mid) in enumerate(zip(masks, ids_e)):
            t, b = divmod(mid - 1 - T, B)
            assert mid == perm_model_id(t, b, T, B)
            alt = base if full else tests[t]
            # the tested column replaced in place by the engine's j-th appended column
            assert mk == [Kc + j if k == tested[t] else k for k in alt] and (Kc + j) in mk
            assert len(mk) == len(alt) and tested[t] not in mk


def test_refusals_raise_before_any_device_work(monkeypatch):
    import torch
    # a call that got past the checks would reach the device: make that loud on any machine
    monkeypatch.setattr(torch.cuda, "is_available", lambda: (_ for _ in ()).throw(AssertionError("device touched")))
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a: (_ for _ in ()).throw(AssertionError("device touched")))
    data = [np.ones((6, 4), np.float32)] * 3
    Xc = np.ones((6, 2), np.float32)
    for kw, msg in ((dict(LRT_index=[0], n_perm=-1), ">= 0"), (dict(LRT_index=[], n_perm=2), "tested covariate"),
                    (dict(Xc=np.ones((6, 0), np.float32), LRT_index=None, n_perm=1), "tested covariate"),
                    (dict(LRT_index=[0, 1], n_perm=2047), "model ids")):
        kw = dict(dict(Xc=Xc), **kw)
        with pytest.raises(ValueError, match=msg):
            fit_BRIE_matrix([d.copy() for d in data], **kw)
    from brie_b200.utils.anndata_lite import AnnDataLite
    ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]})
    for kw, msg in ((dict(LRT_index=[0], n_perm=-3), ">= 0"), (dict(LRT_index=[], n_perm=1), "tested covariate"),
                    (dict(LRT_index=None, n_perm=2047), "model ids")):
        with pytest.raises(ValueError, match=msg):
            fitBRIE(ad, Xc=Xc, **kw)
    # the id budget: 1 + T (1 + B) <= 4096
    assert check_n_perm(2046, 2) == 2046 and check_n_perm(4094, 1) == 4094 and check_n_perm(0, 0) == 0
    with pytest.raises(ValueError):
        check_n_perm(4095, 1)


@pytest.mark.parametrize("args,msg", [(["--nPerm", "-1", "--LRTindex", "0"], "--nPerm needs to be 0 or more"),
                                      (["--nPerm", "3", "--LRTindex", "None"], "--nPerm needs tested features"),
                                      (["--nPerm", "3"], "--nPerm needs tested features")])
def test_cli_refuses_bad_nperm(tmp_path, args, msg):
    out = subprocess.run([sys.executable, "-m", "brie_b200.bin.quant", "-i", str(tmp_path / "missing.npz")] + args,
                         capture_output=True, text=True, cwd=ROOT, timeout=300, env=dict(os.environ, PYTHONPATH=ROOT))
    assert out.returncode == 1 and msg in out.stdout, out.stdout + out.stderr[-2000:]


def test_cli_help_lists_nperm():
    out = subprocess.run([sys.executable, "-m", "brie_b200.bin.quant", "--help"], capture_output=True, text=True,
                         cwd=ROOT, timeout=300)
    assert out.returncode == 0 and "--nPerm" in out.stdout and "Calibration (not in the reference)" in out.stdout


def _table_adata(with_perm):
    import pandas as pd
    from brie_b200.utils.anndata_lite import AnnDataLite
    rng = np.random.default_rng(0)
    X = rng.poisson(0.3, (6, 4)).astype(np.float32)
    ad = AnnDataLite(X=X, var=pd.DataFrame({'n_counts': X.sum(0), 'n_counts_uniq': X.sum(0)},
                                           index=pd.Index(list("abcd"), name="GeneID")))
    ad.varm['intercept'] = rng.normal(size=(4, 1))
    ad.varm['sigma'] = rng.uniform(size=(4, 1))
    for k in ('cell_coeff', 'ELBO_gain', 'pval', 'fdr'):
        ad.varm[k] = rng.uniform(size=(4, 2))
    ad.uns['brie_param'] = {'LRT_index': [0, 1]}
    ad.uns['Xc_ids'] = ['isEAE', 'isCD1']
    if with_perm:
        ad.varm['ELBO_gain_perm'] = rng.normal(size=(4, 2, 3)).astype(np.float32)
        ad.varm['pval_perm'] = rng.uniform(size=(4, 2))
        ad.varm['fdr_perm'] = rng.uniform(size=(4, 2))
        ad.uns['brie_param']['n_perm'] = 3
    return ad


def test_dump_results_appends_perm_columns_after_the_old_ones():
    from brie_b200.utils.io_utils import dump_results
    old = dump_results(_table_adata(False))
    new = dump_results(_table_adata(True))
    n = len(old.columns)
    assert 'isEAE_pval_perm' not in old.columns and n == 5 + 4 * 2
    assert list(new.columns[:n]) == list(old.columns)
    assert list(new.columns[n:]) == ['isEAE_pval_perm', 'isEAE_FDR_perm', 'isCD1_pval_perm', 'isCD1_FDR_perm']
    ad = _table_adata(True)
    assert np.array_equal(new['isCD1_FDR_perm'].values, ad.varm['fdr_perm'][:, 1])


def test_npz_container_round_trips_the_3d_null_gains(tmp_path):
    from brie_b200.utils.anndata_lite import AnnDataLite
    ad = _table_adata(True)
    p = str(tmp_path / "out.npz")
    ad.write_npz(p)
    back = AnnDataLite.read_npz(p)
    for k in ('ELBO_gain_perm', 'pval_perm', 'fdr_perm'):
        assert back.varm[k].shape == ad.varm[k].shape and np.array_equal(back.varm[k], ad.varm[k]), k
    assert back.uns['brie_param']['n_perm'] == 3
    sub = back[:, [0, 2]]
    assert np.array_equal(sub.varm['ELBO_gain_perm'], ad.varm['ELBO_gain_perm'][[0, 2]])
