"""Score tests of candidate cell covariates from the fitted posterior (score_X / brie-quant --scoreFile): the host
side -- the float64 restatement on a conjugate model with known answers, score_from_parts, the degenerate rules, the
refusals, the output layout and merges, the container, the CLI and the score table, and the ABI refusals.  No GPU
needed."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy.stats import chi2

import score_ref
import wald_ref
from brie_b200.engine import score_from_parts
from brie_b200.models.model_wrap import (BRIE_RV, SCORE_KEYS, _merge_shared, _set_fdr_score, check_score_X, fdr_bh,
                                         fit_BRIE_matrix, fitBRIE)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _conjugate(theta_shift=0.0, seed=0):
    """Z ~ N(x~ theta + x beta, sigma^2), y | Z ~ N(Z, tau^2), 400 cells, 3 events; the candidate x is correlated with
    a fitted column.  Returns the null model's exact posterior at theta_hat + theta_shift, and the marginal model's
    full fit (beta_hat, its Wald z^2, 2 delta loglik), per event."""
    rng = np.random.default_rng(seed)
    Nc, Ng = 400, 3
    x1 = rng.normal(size=Nc)
    Xt = np.stack([x1, np.ones(Nc)], axis=1)                       # a covariate and the per-event intercept
    x = 0.6 * x1 + rng.normal(size=Nc)
    sig, tau = np.array([0.8, 1.1, 0.5]), 0.7
    v = sig ** 2 + tau ** 2                                         # marginal variance of y
    y = (Xt @ rng.normal(size=(2, Ng)) + x[:, None] * np.array([0.3, 0.0, -0.2])[None, :]
         + rng.normal(size=(Nc, Ng)) * np.sqrt(v))
    theta = np.linalg.lstsq(Xt, y, rcond=None)[0] + theta_shift     # null MLE (known variance)
    m = Xt @ theta
    s2 = 1.0 / (1.0 / sig ** 2 + 1.0 / tau ** 2)
    mu = s2 * (m / sig ** 2 + y / tau ** 2)                         # exact posterior of Z given y
    Xf = np.concatenate([Xt, x[:, None]], axis=1)
    coef = np.linalg.lstsq(Xf, y, rcond=None)[0]
    beta = coef[2]
    var_beta = np.linalg.inv(Xf.T @ Xf)[2, 2] * v
    rss0 = ((y - Xt @ (theta - theta_shift)) ** 2).sum(0)
    rss1 = ((y - Xf @ coef) ** 2).sum(0)
    lam = np.broadcast_to(0.5 * np.log(s2), (Nc, Ng))
    return dict(Z_loc=mu, Z_std_log=lam, sigma_log=np.log(sig), prior_mean=m, Xt=Xt, X=x[:, None], beta=beta,
                wald_z2=beta ** 2 / var_beta, lrt=(rss0 - rss1) / v)


def _score(c, X=None):
    X = c['X'] if X is None else X
    parts = score_ref.parts(c['Z_loc'], c['Z_std_log'], c['sigma_log'], c['prior_mean'], c['Xt'], X)
    return score_from_parts(parts, wald_ref.info(c['Z_std_log'], c['sigma_log'], c['Xt']))


def test_conjugate_known_answers():
    c = _conjugate()
    z, eff, p = _score(c)
    stat = z[:, 0] ** 2
    assert np.allclose(stat, c['wald_z2'], rtol=1e-9, atol=0)
    assert np.allclose(stat, c['lrt'], rtol=1e-9, atol=0)
    assert np.allclose(eff[:, 0], c['beta'], rtol=1e-9, atol=0)          # one-step estimate = full-fit coefficient
    assert np.allclose(p[:, 0], chi2.sf(stat, 1))


def test_conjugate_statistic_is_invariant_to_an_unconverged_theta():
    c0 = _conjugate()
    c1 = _conjugate(theta_shift=np.array([[0.05, -0.02, 0.1], [0.1, 0.03, -0.05]]))
    z0, e0, _ = _score(c0)
    z1, e1, _ = _score(c1)
    assert np.allclose(z1, z0, rtol=1e-9) and np.allclose(e1, e0, rtol=1e-9)
    # the plain score U / sqrt(V) moves
    U, A, B, Ut = score_ref.parts(c1['Z_loc'], c1['Z_std_log'], c1['sigma_log'], c1['prior_mean'], c1['Xt'], c1['X'])
    assert np.abs(Ut).max() > 1.0


def _random_parts(rng, Ng, J, K):
    Xt = rng.normal(size=(50, K))
    X = rng.normal(size=(50, J))
    w = rng.uniform(0.2, 1.0, size=(50, Ng))
    r = rng.normal(size=(50, Ng))
    info = np.einsum('cg,ck,cl->gkl', w, Xt, Xt)
    return (r.T @ X, w.T @ X ** 2, np.einsum('cg,cj,ck->gjk', w, X, Xt), r.T @ Xt), info


def test_score_from_parts_matches_a_direct_inverse():
    rng = np.random.default_rng(1)
    (U, A, B, Ut), info = _random_parts(rng, 7, 5, 3)
    z, eff, p = score_from_parts((U, A, B, Ut), info)
    for g in range(7):
        Ii = np.linalg.inv(info[g])
        V = A[g] - np.einsum('jk,kl,jl->j', B[g], Ii, B[g])
        Ue = U[g] - B[g] @ Ii @ Ut[g]
        assert np.allclose(z[g], Ue / np.sqrt(V), rtol=1e-10)
        assert np.allclose(eff[g], Ue / V, rtol=1e-10)
        assert np.allclose(p[g], chi2.sf(Ue ** 2 / V, 1), rtol=1e-10)


def test_no_fitted_column_gives_the_plain_score():
    rng = np.random.default_rng(2)
    U, A = rng.normal(size=(4, 3)), rng.uniform(1, 2, size=(4, 3))
    z, eff, p = score_from_parts((U, A, np.zeros((4, 3, 0)), np.zeros((4, 0))), np.zeros((4, 0, 0)))
    assert np.allclose(z, U / np.sqrt(A)) and np.allclose(eff, U / A)


def test_degenerate_candidates_and_information():
    c = _conjugate()
    Nc = c['X'].shape[0]
    X = np.stack([c['Xt'][:, 0] * 2.0, np.ones(Nc), np.zeros(Nc), c['X'][:, 0]], axis=1)
    z, eff, p = _score(c, X)
    # collinear with the fitted column, constant with a gene intercept, zero on every cell
    assert np.isnan(z[:, :3]).all() and np.isnan(eff[:, :3]).all() and (p[:, :3] == 1).all()
    assert np.isfinite(z[:, 3]).all()
    # an information that is not positive definite: the whole event
    parts = score_ref.parts(c['Z_loc'], c['Z_std_log'], c['sigma_log'], c['prior_mean'], c['Xt'], X)
    info = wald_ref.info(c['Z_std_log'], c['sigma_log'], c['Xt'])
    info[1] = np.array([[1.0, 1.0], [1.0, 1.0]])
    z, eff, p = score_from_parts(parts, info)
    assert np.isnan(z[1]).all() and (p[1] == 1).all() and np.isfinite(z[[0, 2], 3]).all()


def test_refusals_before_any_device_work(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: (_ for _ in ()).throw(AssertionError("device touched")))
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a: (_ for _ in ()).throw(AssertionError("device touched")))
    from brie_b200.utils.anndata_lite import AnnDataLite
    data = [np.ones((6, 3), np.float32) for _ in range(3)]
    good = np.zeros((6, 2))
    bad_inf = good.copy()
    bad_inf[2, 1] = np.inf
    for kw, msg in ((dict(score_X=good, target='marginLik'), 'marginLik'), (dict(score_X=np.zeros((5, 2))), 'shape'),
                    (dict(score_X=np.zeros(6)), 'shape'), (dict(score_X=np.zeros((6, 0))), 'shape'),
                    (dict(score_X=bad_inf), 'non-finite'), (dict(score_X=np.full((6, 1), np.nan)), 'non-finite')):
        with pytest.raises(ValueError, match=msg):
            fit_BRIE_matrix([d.copy() for d in data], **kw)
        ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]})
        with pytest.raises(ValueError, match=msg):
            fitBRIE(ad, **kw)
    assert check_score_X(None, 'marginLik', 6) is None
    assert check_score_X(good, 'ELBO', 6).dtype == np.float32


def _rv(rng, Ng, J=2):
    r = BRIE_RV()
    r.Nc, r.Ng, r.intercept_mode = 5, Ng, 'gene'
    r.losses = np.zeros(3)
    r.loss_gene = rng.normal(size=Ng)
    for k, shape in (('sigma', (1, Ng)), ('intercept', (1, Ng)), ('cell_coeff', (2, Ng)), ('Psi', (5, Ng)),
                     ('Psi95CI', (5, Ng)), ('Z_std', (5, Ng)), ('Z_loc', (5, Ng))):
        setattr(r, k, rng.normal(size=shape))
    r.score_z, r.score_effect = rng.normal(size=(Ng, J)), rng.normal(size=(Ng, J))
    r.pval_score = rng.uniform(size=(Ng, J))
    _set_fdr_score(r)
    return r


@pytest.mark.parametrize("merge", ["concate", "shared"])
def test_chunks_and_ranks_carry_the_score_outputs(merge):
    rng = np.random.default_rng(5)
    a, b = _rv(rng, 4), _rv(rng, 3)
    want = {k: np.concatenate([getattr(a, k), getattr(b, k)]) for k in ('score_z', 'score_effect', 'pval_score')}
    if merge == "concate":
        a.concate(b)
        out = a
    else:
        out = _merge_shared([a, b])
    _set_fdr_score(out)
    for k, v in want.items():
        assert np.array_equal(getattr(out, k), v), k
    for j in range(2):
        assert np.array_equal(out.fdr_score[:, j], fdr_bh(want['pval_score'][:, j]))   # pooled over both parts


def _score_adata():
    import pandas as pd
    from brie_b200.utils.anndata_lite import AnnDataLite
    rng = np.random.default_rng(0)
    X = rng.poisson(0.3, (6, 4)).astype(np.float32)
    ad = AnnDataLite(X=X, var=pd.DataFrame({'n_counts': X.sum(0), 'n_counts_uniq': X.sum(0)},
                                           index=pd.Index(list("abcd"), name="GeneID")))
    for k in SCORE_KEYS:
        ad.varm[k] = rng.uniform(size=(4, 2))
    ad.uns['brie_param'] = {'LRT_index': [], 'score': 2}
    ad.uns['score_ids'] = np.array(['RBFOX2', 'rs123'])
    return ad


def test_score_table_and_container_round_trip(tmp_path):
    from brie_b200.utils.anndata_lite import AnnDataLite
    from brie_b200.utils.io_utils import score_table
    ad = _score_adata()
    t = score_table(ad)
    assert list(t.columns) == ['RBFOX2_score_z', 'RBFOX2_pval_score', 'RBFOX2_FDR_score',
                               'rs123_score_z', 'rs123_pval_score', 'rs123_FDR_score']
    assert list(t.index) == list("abcd")
    assert np.array_equal(t['rs123_FDR_score'].values, ad.varm['fdr_score'][:, 1])
    p = str(tmp_path / "out.npz")
    ad.write_npz(p)
    back = AnnDataLite.read_npz(p)
    for k in SCORE_KEYS:
        assert np.array_equal(back.varm[k], ad.varm[k]), k
    assert back.uns['brie_param']['score'] == 2 and list(back.uns['score_ids']) == ['RBFOX2', 'rs123']


def _cli_input(tmp_path, Nc=6, Ng=3):
    from brie_b200.utils import io_utils
    layers = {k: np.ones((Nc, Ng), np.float32) for k in ('isoform1', 'isoform2', 'ambiguous')}
    inp = str(tmp_path / "c.npz")
    cells = ["c%d" % i for i in range(Nc)]
    io_utils.write_npz_counts(inp, layers, np.ones((Ng, 2, 3), np.float32), cells, ["g%d" % i for i in range(Ng)])
    return inp, cells


def test_cli_score_file_parses_and_reaches_fitBRIE(tmp_path, monkeypatch):
    import brie_b200.models as models
    from brie_b200.bin import quant as q
    seen = {}

    class Stop(Exception):
        pass

    def spy_fit(adata, **kw):
        seen['fit'] = kw
        raise Stop()
    inp, cells = _cli_input(tmp_path)
    sf = tmp_path / "score.tsv"
    rows = ["cellID\tRBFOX2\trs123"] + ["%s\t%d\t%.1f" % (c, i, 0.5 * i) for i, c in enumerate(cells[::-1])]
    sf.write_text("\n".join(rows) + "\n")
    monkeypatch.setattr(q, "filter_genes", lambda adata, **kw: adata)
    monkeypatch.setattr(models, "fitBRIE", spy_fit)
    monkeypatch.setattr(sys, "argv", ["brie-quant", "-i", inp, "-o", str(tmp_path / "o.npz")])
    with pytest.raises(Stop):
        q.main()
    assert seen['fit']['score_X'] is None
    monkeypatch.setattr(sys, "argv", ["brie-quant", "-i", inp, "-o", str(tmp_path / "o.npz"), "--scoreFile", str(sf)])
    with pytest.raises(Stop):
        q.main()
    X = seen['fit']['score_X']
    assert X.dtype == np.float32 and X.shape == (6, 2)
    assert np.array_equal(X[:, 0], np.arange(6)[::-1]) and np.array_equal(X[:, 1], 0.5 * np.arange(6)[::-1])
    # a fitted cell missing from the file
    sf.write_text("\n".join(rows[:-1]) + "\n")
    with pytest.raises(SystemExit) as e:
        q.main()
    assert e.value.code == 1 and 'fit' in seen
    out = __import__('subprocess').run([sys.executable, "-m", "brie_b200.bin.quant", "--help"], capture_output=True,
                                       text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0 and "--scoreFile" in out.stdout


def _bind_fake(lib, target=0, **buffers):
    """A narrow fit (Kc = 1, gene intercept) bound to fake aligned addresses: brie_fit_bind reads no memory of such a
    fit, so the argument checks run without a device.  None of these addresses may reach a launch."""
    from brie_b200 import _lib
    d = _lib.FitDesc()
    d.n_cells, d.n_events, d.ld, d.event_offset, d.seed = 100, 50, 64, 0, 1
    d.n_models, d.Kc, d.Kg, d.mc_size, d.n_layers = 1, 1, 0, 3, 3
    d.has_efflen, d.cell_mode, d.train_intercept, d.train_sigma, d.trace_cap = 0, 0, 1, 1, 8
    d.xc_mask[0], d.target = 1, target
    h = C.c_void_p()
    assert lib.brie_fit_create(C.byref(d), C.byref(h)) == 0
    b = _lib.FitBuffers()
    fake = iter(range(0x10000, 0x1000000, 0x1000))
    for name in ("Xc", "Z_loc", "Z_std_log", "adam_Z", "Wc", "intercept", "sigma_log", "adam_small", "active",
                 "loss_trace", "scratch"):
        setattr(b, name, next(fake))
    for i in range(3):
        b.counts[i] = next(fake)
    for name, v in buffers.items():
        setattr(b, name, v)
    assert lib.brie_fit_bind(h, C.byref(b)) == 0, lib.brie_last_error()
    return h


def test_abi_refusals_on_fake_addresses():
    """brie_fit_score_sizes / brie_fit_score_parts refuse a null or unbound fit, a model out of range, a gathered
    sub-fit, target marginLik, n_cand <= 0, ldx < n_cand and null or misaligned outputs or scratch, before any
    launch."""
    import torch
    from brie_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("a refusal missed here would launch on fake addresses")
    lib = _lib.load()
    ARG, UNSUP = -1, -3
    sz, kt = C.c_size_t(), C.c_int32()
    good = (0x10000000, 4, 4, 0x20000000, 0x30000000, 0x40000000, 0x50000000, 0x60000000)
    assert lib.brie_fit_score_sizes(None, 0, 4, C.byref(sz), C.byref(kt)) == ARG
    assert lib.brie_fit_score_parts(None, 0, *good, None) == ARG
    h = C.c_void_p()
    assert lib.brie_fit_create(C.byref(_lib.FitDesc(n_cells=10, n_events=4, ld=32, n_models=1, n_layers=2,
                                                    mc_size=1, trace_cap=1)), C.byref(h)) == 0
    assert lib.brie_fit_score_sizes(h, 0, 4, C.byref(sz), C.byref(kt)) == ARG             # not bound
    assert b"not bound" in lib.brie_last_error()
    lib.brie_fit_destroy(h)
    h = _bind_fake(lib)
    try:
        assert lib.brie_fit_score_sizes(h, 0, 4, C.byref(sz), C.byref(kt)) == 0
        assert kt.value == 2 and sz.value > 0                                            # x1 and the intercept
        assert lib.brie_fit_score_sizes(h, 0, 4, None, C.byref(kt)) == ARG
        for m, n in ((-1, 4), (1, 4), (0, 0), (0, -3)):                                 # model range, n_cand <= 0
            assert lib.brie_fit_score_sizes(h, m, n, C.byref(sz), C.byref(kt)) == ARG
        call = lambda *a: lib.brie_fit_score_parts(h, 0, *a, None)
        assert call(0, *good[1:]) == ARG                                                 # no X
        assert call(good[0], 4, 3, *good[3:]) == ARG                                     # ldx < n_cand
        assert call(good[0], 0, 4, *good[3:]) == ARG                                     # n_cand <= 0
        for i in range(5):                                                               # U, A, B, Ut, scratch
            for bad in (0, good[3 + i] + 4):
                args = list(good)
                args[3 + i] = bad
                assert call(*args) == ARG, (i, bad)
        assert lib.brie_fit_score_parts(h, 1, *good, None) == ARG
        assert lib.brie_fit_launch_count(h) == 0
    finally:
        lib.brie_fit_destroy(h)
    for kw, what in ((dict(target=1), b"target ELBO"), (dict(counts_model_stride=100 * 64), b"parent")):
        h = _bind_fake(lib, **kw)
        assert lib.brie_fit_score_sizes(h, 0, 4, C.byref(sz), C.byref(kt)) == UNSUP and what in lib.brie_last_error()
        assert lib.brie_fit_score_parts(h, 0, *good, None) == UNSUP
        assert lib.brie_fit_launch_count(h) == 0
        lib.brie_fit_destroy(h)
