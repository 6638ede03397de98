"""Wald tests of the cell coefficients from the fitted posterior (wald / brie-quant --wald): the host side -- the
float64 restatement of the information, wald_from_info, pair packing, the marginLik refusal, the output layout,
the result table, the container and the CLI.  No GPU needed."""
import math
import os
import sys

import numpy as np
import pytest

import wald_ref
from brie_b200.engine import pair_index, unpack_pairs, wald_from_info
from brie_b200.models.model_wrap import (BRIE_RV, _merge_shared, _set_fdr_wald, _set_wald_outputs, check_wald,
                                         fdr_bh, fit_BRIE_matrix, fitBRIE)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle_state(mode):
    from oracle.brie2_oracle import oracle_fit_matrix
    from util import make_problem
    data, effLen, Xc, _ = make_problem(30, 8, 2, 0, True, 3, seed=3)
    res = oracle_fit_matrix(data, Xc=Xc, effLen=effLen, intercept=0 if mode == 'None' else None,
                            intercept_mode=mode, LRT_index=[], dtype=np.float64, min_iter=60, max_iter=60, n_eval=1,
                            MC_size=2)
    return res.model, Xc


@pytest.mark.parametrize("mode", ['gene', 'None', 'cell'])
def test_restatement_on_an_oracle_fit_matches_a_scalar_loop(mode):
    m, Xc = _oracle_state(mode)
    cell = mode == 'cell'
    has_b = mode == 'gene'
    lam, tau = m.p['Z_std_log'], m.p['sigma_log'].reshape(-1)
    Xt = wald_ref.design_rows(Xc, has_b)
    I = wald_ref.info(lam, tau, Xt, cell)
    Nc, Ng = lam.shape
    K = 2 + has_b
    assert I.shape == (Ng, K, K)
    for g in range(Ng):
        want = np.zeros((K, K))
        for c in range(Nc):
            sig2 = math.exp(2 * (tau[c] if cell else tau[g]))
            s2 = math.exp(2 * lam[c, g])
            x = [float(Xc[c, 0]), float(Xc[c, 1])] + ([1.0] if has_b else [])
            for k in range(K):
                for l in range(K):
                    want[k, l] += max(sig2 - s2, 0.0) / sig2 ** 2 * x[k] * x[l]
        assert np.allclose(I[g], want, rtol=1e-10, atol=0)
        assert np.allclose(I[g], I[g].T)
        # the missing information only removes information: naive - Louis is positive semi-definite
        naive = wald_ref.naive_info(tau, Xt, Ng, cell)[g]
        assert np.linalg.eigvalsh(naive - I[g]).min() > -1e-9 * np.abs(naive).max()
    assert (wald_ref.weights(lam, tau, cell) >= 0).all()


def test_louis_information_is_the_exact_marginal_information_of_a_conjugate_model():
    """y_c ~ N(z_c, v_c), z_c ~ N(x_c b, sigma^2): the exact posterior variance is s^2 = 1 / (1/sigma^2 + 1/v_c) and
    y_c ~ N(x_c b, sigma^2 + v_c) has information sum_c x x^T / (sigma^2 + v_c).  The formula gives exactly that,
    and the complete-data term alone does not."""
    rng = np.random.default_rng(0)
    Nc = 200
    Xt = np.stack([rng.binomial(1, 0.5, Nc), rng.normal(size=Nc), np.ones(Nc)], axis=1)
    tau = np.array([0.3])
    sig2 = math.exp(2 * tau[0])
    v = rng.uniform(0.05, 20, Nc)
    lam = 0.5 * np.log(1 / (1 / sig2 + 1 / v))[:, None]
    exact = np.einsum('c,ck,cl->kl', 1 / (sig2 + v), Xt, Xt)
    assert np.allclose(wald_ref.info(lam, tau, Xt)[0], exact, rtol=1e-12)
    assert not np.allclose(wald_ref.naive_info(tau, Xt, 1)[0], exact, rtol=0.1)


def test_pair_packing_is_row_major_over_the_upper_triangle():
    k, l = pair_index(3)
    assert list(zip(k.tolist(), l.tolist())) == [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    A = np.random.default_rng(1).normal(size=(5, 4, 4))
    A = A + A.transpose(0, 2, 1)
    k, l = pair_index(4)
    assert np.array_equal(unpack_pairs(A[:, k, l], 4), A)
    assert unpack_pairs(np.zeros((7, 1)), 1).shape == (7, 1, 1)


def test_wald_from_info_matches_a_direct_inverse():
    from scipy.stats import chi2
    rng = np.random.default_rng(2)
    Ng, K = 40, 3
    X = rng.normal(size=(Ng, 60, K))
    info = np.einsum('gck,gcl->gkl', X, X) * rng.uniform(0.1, 10, (Ng, 1, 1))
    coef = rng.normal(size=(Ng, K))
    se, pval = wald_from_info(coef, info)
    want = np.sqrt(np.diagonal(np.linalg.inv(info), axis1=1, axis2=2))
    assert np.allclose(se, want, rtol=1e-10)
    assert np.allclose(pval, chi2.sf((coef / want) ** 2, 1), rtol=1e-9)
    # one coefficient
    se1, p1 = wald_from_info(coef[:, :1], info[:, :1, :1])
    assert np.allclose(se1[:, 0], 1 / np.sqrt(info[:, 0, 0]))
    assert wald_from_info(np.zeros((4, 0)), np.zeros((4, 0, 0)))[0].shape == (4, 0)


def test_non_positive_definite_information_gives_nan_se_and_pval_one():
    rng = np.random.default_rng(3)
    X = rng.normal(size=(6, 50, 2))
    info = np.einsum('gck,gcl->gkl', X, X)
    info[0] = 0.0                                              # no cell with reads
    info[1] = [[1.0, 1.0], [1.0, 1.0]]                         # singular
    info[2] = [[1.0, 2.0], [2.0, 1.0]]                         # indefinite
    info[3] = [[-1.0, 0.0], [0.0, 1.0]]                        # negative diagonal
    info[4, 0, 0] = np.nan
    info[5] = [[1.0, 1.0 - 1e-15], [1.0 - 1e-15, 1.0]]         # numerically singular
    coef = np.ones((6, 2))
    se, pval = wald_from_info(coef, info)
    assert np.isnan(se).all() and (pval == 1.0).all()
    good = np.einsum('ck,cl->kl', X[0], X[0])
    se, pval = wald_from_info(np.ones((2, 2)), np.stack([good, np.zeros((2, 2))]))
    assert np.isfinite(se[0]).all() and np.isnan(se[1]).all() and (pval[1] == 1.0).all() and (pval[0] < 1).all()


def test_marginlik_refusal_before_any_device_work(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: (_ for _ in ()).throw(AssertionError("device touched")))
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a: (_ for _ in ()).throw(AssertionError("device touched")))
    data = [np.ones((6, 4), np.float32)] * 3
    Xc = np.ones((6, 2), np.float32)
    with pytest.raises(ValueError, match="marginLik"):
        fit_BRIE_matrix([d.copy() for d in data], Xc=Xc, LRT_index=[], wald=True, target="marginLik")
    from brie_b200.utils.anndata_lite import AnnDataLite
    ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]})
    with pytest.raises(ValueError, match="marginLik"):
        fitBRIE(ad, Xc=Xc, LRT_index=[0], wald=True, target="marginLik")
    assert check_wald(False, "marginLik") is False and check_wald(True, "ELBO") is True


def _per_model(rng, Ng, widths, has_b):
    return {m: (rng.uniform(0.1, 1, (Ng, w + has_b)), rng.uniform(size=(Ng, w + has_b)), w)
            for m, w in enumerate(widths)}


def test_output_layout_full_and_null_mode():
    rng = np.random.default_rng(4)
    Ng = 7
    r = BRIE_RV()
    pm = _per_model(rng, Ng, [3], True)                        # full: model 0 only, Kc = 3, gene intercept
    _set_wald_outputs(r, pm, True, [0, 1, 2], [0, 2])
    assert r.cell_coeff_se.shape == (3, Ng) and np.array_equal(r.cell_coeff_se, pm[0][0][:, :3].T)
    assert np.array_equal(r.pval_wald, pm[0][1][:, :3]) and np.array_equal(r.intercept_se[0], pm[0][0][:, 3])
    assert r.wald_columns == [0, 1, 2]
    for i in range(3):
        assert np.array_equal(r.fdr_wald[:, i], fdr_bh(r.pval_wald[:, i]))
    r = BRIE_RV()                                              # null: base [1], tests [0], [2]: base + [t]
    pm = _per_model(rng, Ng, [1, 2, 2], False)
    _set_wald_outputs(r, pm, False, [1], [0, 2])
    assert r.cell_coeff_se.shape == (3, Ng) and not hasattr(r, 'intercept_se')
    assert np.array_equal(r.cell_coeff_se[0], pm[0][0][:, 0])
    assert np.array_equal(r.cell_coeff_se[1], pm[1][0][:, 1]) and np.array_equal(r.cell_coeff_se[2], pm[2][0][:, 1])
    assert np.array_equal(r.pval_wald[:, 2], pm[2][1][:, 1])
    assert r.wald_columns == [1, 0, 2]


def _rv(rng, Ng, with_b=True):
    r = BRIE_RV()
    r.Nc, r.Ng, r.intercept_mode = 5, Ng, 'gene'
    r.losses = np.zeros(3)
    r.loss_gene = rng.normal(size=Ng)
    for k, shape in (('sigma', (1, Ng)), ('intercept', (1, Ng)), ('cell_coeff', (2, Ng)), ('Psi', (5, Ng)),
                     ('Psi95CI', (5, Ng)), ('Z_std', (5, Ng)), ('Z_loc', (5, Ng))):
        setattr(r, k, rng.normal(size=shape))
    _set_wald_outputs(r, _per_model(rng, Ng, [2], with_b), True, [0, 1], [])
    return r


@pytest.mark.parametrize("merge", ["concate", "shared"])
def test_chunks_and_ranks_carry_the_wald_outputs(merge):
    rng = np.random.default_rng(5)
    a, b = _rv(rng, 4), _rv(rng, 3)
    se = np.concatenate([a.cell_coeff_se, b.cell_coeff_se], axis=1)
    pv = np.concatenate([a.pval_wald, b.pval_wald])
    ise = np.concatenate([a.intercept_se, b.intercept_se], axis=1)
    if merge == "concate":
        a.concate(b)
        out = a
    else:
        out = _merge_shared([a, b])
    _set_fdr_wald(out)
    assert np.array_equal(out.cell_coeff_se, se) and np.array_equal(out.pval_wald, pv)
    assert np.array_equal(out.intercept_se, ise) and out.wald_columns == [0, 1]
    for i in range(2):
        assert np.array_equal(out.fdr_wald[:, i], fdr_bh(pv[:, i]))          # pooled over both parts


def _table_adata(wald, names=True, cols=(0, 1)):
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
    ad.varm['pval_perm'] = rng.uniform(size=(4, 1))
    ad.varm['fdr_perm'] = rng.uniform(size=(4, 1))
    ad.uns['brie_param'] = {'LRT_index': [1], 'n_perm': 2}
    if names:
        ad.uns['Xc_ids'] = ['isEAE', 'isCD1']
    if wald:
        for k in ('cell_coeff_se', 'pval_wald', 'fdr_wald'):
            ad.varm[k] = rng.uniform(size=(4, 2))
        ad.varm['intercept_se'] = rng.uniform(size=(4, 1))
        ad.uns['brie_param']['wald'] = True
        ad.uns['brie_param']['wald_columns'] = list(cols)
    return ad


def test_dump_results_appends_wald_columns_labelled_by_covariate():
    from brie_b200.utils.io_utils import dump_results
    old = dump_results(_table_adata(False))
    n = len(old.columns)
    # full mode: rows in covariate order; the LRT columns keep the reference's loop-position label
    new = dump_results(_table_adata(True))
    assert list(new.columns[:n]) == list(old.columns) and old.columns[-1] == 'isCD1_FDR_perm'
    assert list(new.columns[n:]) == ['isEAE_se', 'isEAE_pval_wald', 'isEAE_FDR_wald',
                                     'isCD1_se', 'isCD1_pval_wald', 'isCD1_FDR_wald']
    ad = _table_adata(True)
    assert np.array_equal(new['isCD1_pval_wald'].values, ad.varm['pval_wald'][:, 1])
    assert np.array_equal(new['isEAE_se'].values, ad.varm['cell_coeff_se'][:, 0])
    # null mode: base rows, then the tested ones -- cell_coeff row 0 is covariate 1 here
    new = dump_results(_table_adata(True, cols=(1, 0)))
    assert list(new.columns[n:]) == ['isCD1_se', 'isCD1_pval_wald', 'isCD1_FDR_wald',
                                     'isEAE_se', 'isEAE_pval_wald', 'isEAE_FDR_wald']
    assert np.array_equal(new['isCD1_FDR_wald'].values, _table_adata(True, cols=(1, 0)).varm['fdr_wald'][:, 0])
    new = dump_results(_table_adata(True, names=False, cols=(1, 0)))
    assert list(new.columns[-6:]) == ['X1_se', 'X1_pval_wald', 'X1_FDR_wald', 'X0_se', 'X0_pval_wald', 'X0_FDR_wald']


def test_npz_container_round_trips_the_wald_keys(tmp_path):
    from brie_b200.utils.anndata_lite import AnnDataLite
    ad = _table_adata(True, cols=(1, 0))
    p = str(tmp_path / "out.npz")
    ad.write_npz(p)
    back = AnnDataLite.read_npz(p)
    for k in ('cell_coeff_se', 'pval_wald', 'fdr_wald', 'intercept_se'):
        assert np.array_equal(back.varm[k], ad.varm[k]), k
    assert back.uns['brie_param']['wald'] is True and list(back.uns['brie_param']['wald_columns']) == [1, 0]
    assert np.array_equal(back[:, [0, 2]].varm['pval_wald'], ad.varm['pval_wald'][[0, 2]])


def test_cli_flag_parses_and_reaches_fitBRIE(tmp_path, monkeypatch):
    import brie_b200.models as models
    from brie_b200.bin import quant as q
    from brie_b200.utils import io_utils
    seen = {}
    real_quant = q.quant

    def spy_quant(*a):
        seen['args'] = a
        return real_quant(*a)

    class Stop(Exception):
        pass

    def spy_fit(adata, **kw):
        seen['fit'] = kw
        raise Stop()
    Nc, Ng = 6, 3
    layers = {k: np.ones((Nc, Ng), np.float32) for k in ('isoform1', 'isoform2', 'ambiguous')}
    inp = str(tmp_path / "c.npz")
    io_utils.write_npz_counts(inp, layers, np.ones((Ng, 2, 3), np.float32), ["c%d" % i for i in range(Nc)],
                              ["g%d" % i for i in range(Ng)])
    monkeypatch.setattr(q, "quant", spy_quant)
    monkeypatch.setattr(q, "filter_genes", lambda adata, **kw: adata)
    monkeypatch.setattr(models, "fitBRIE", spy_fit)
    for argv, want in (([], False), (["--wald"], True)):
        monkeypatch.setattr(sys, "argv", ["brie-quant", "-i", inp, "-o", str(tmp_path / "o.npz")] + argv)
        with pytest.raises(Stop):
            q.main()
        assert seen['args'][-1] is want and seen['fit']['wald'] is want
    out = __import__('subprocess').run([sys.executable, "-m", "brie_b200.bin.quant", "--help"], capture_output=True,
                                       text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0 and "--wald" in out.stdout
