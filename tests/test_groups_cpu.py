"""Joint tests of groups of covariates (LRT_groups, wald_groups, score_groups / brie-quant --LRTgroups, --waldGroups,
--scoreGroups): the host side -- known answers on a conjugate model, the k x k algebra and its degenerate rules, the
refusals, the engine plan, merges, the tables, the container, the CLI and the ABI refusals.  No GPU needed."""
import ctypes as C
import sys

import numpy as np
import pytest
from scipy.stats import chi2

import groups_ref
import score_ref
import wald_ref
from brie_b200.engine import (group_pairs, score_from_parts, score_groups_from_parts, wald_from_info,
                              wald_groups_from_info)
from brie_b200.models.model_wrap import (BRIE_RV, GROUP_KEYS, _engine_plan, _merge_shared, _set_fdr_groups, fdr_bh,
                                         fit_BRIE_matrix, fitBRIE, group_model_id, perm_model_id)
from test_score_cpu import _bind_fake, _cli_input


def _conjugate(theta_shift=0.0, seed=0):
    """Z ~ N(x~ theta + X beta, sigma^2), y | Z ~ N(Z, tau^2), 400 cells, 3 events, a group of 3 candidates X
    correlated with the fitted column and with each other.  Returns the null model's exact posterior at theta_hat +
    theta_shift, and the full model's fit (coefficients, exact posterior, joint 2 delta loglik of the group)."""
    rng = np.random.default_rng(seed)
    Nc, Ng = 400, 3
    x1 = rng.normal(size=Nc)
    Xt = np.stack([x1, np.ones(Nc)], axis=1)                       # a covariate and the per-event intercept
    X = np.stack([0.6 * x1 + rng.normal(size=Nc), rng.binomial(1, 0.3, Nc), rng.binomial(1, 0.4, Nc)], axis=1)
    X[:, 2] -= 0.5 * X[:, 1] * X[:, 2]
    sig, tau = np.array([0.8, 1.1, 0.5]), 0.7
    v = sig ** 2 + tau ** 2                                         # marginal variance of y
    beta = np.array([[0.3, 0.0, -0.2], [0.2, 0.0, 0.1], [-0.4, 0.1, 0.0]])
    y = Xt @ rng.normal(size=(2, Ng)) + X @ beta + rng.normal(size=(Nc, Ng)) * np.sqrt(v)
    theta = np.linalg.lstsq(Xt, y, rcond=None)[0] + theta_shift     # null MLE (known variance)
    s2 = 1.0 / (1.0 / sig ** 2 + 1.0 / tau ** 2)
    post = lambda m: s2 * (m / sig ** 2 + y / tau ** 2)             # exact posterior mean of Z given y
    Xf = np.concatenate([Xt, X], axis=1)
    coef = np.linalg.lstsq(Xf, y, rcond=None)[0]
    rss0 = ((y - Xt @ (theta - theta_shift)) ** 2).sum(0)
    rss1 = ((y - Xf @ coef) ** 2).sum(0)
    lam = np.broadcast_to(0.5 * np.log(s2), (Nc, Ng))
    return dict(Z_loc=post(Xt @ theta), Z_std_log=lam, sigma_log=np.log(sig), prior_mean=Xt @ theta, Xt=Xt, X=X,
                Xf=Xf, coef=coef.T, lrt=(rss0 - rss1) / v)


def _score_groups(c, groups, X=None, info=None):
    X = c['X'] if X is None else X
    parts = score_ref.parts(c['Z_loc'], c['Z_std_log'], c['sigma_log'], c['prior_mean'], c['Xt'], X)
    pairs = group_pairs(groups)
    info = wald_ref.info(c['Z_std_log'], c['sigma_log'], c['Xt']) if info is None else info
    cross = groups_ref.cross(c['Z_std_log'], c['sigma_log'], X, pairs)
    return parts, info, score_groups_from_parts(parts, cross, pairs, info, groups)


def test_conjugate_known_answers():
    c = _conjugate()
    _, _, (stat, p) = _score_groups(c, [[0, 1, 2]])
    # the full fit's joint Wald statistic of the group (its posterior: the information is Xf^T Xf / v exactly)
    wstat, wp = wald_groups_from_info(c['coef'], wald_ref.info(c['Z_std_log'], c['sigma_log'], c['Xf']), [[2, 3, 4]])
    assert np.allclose(stat[:, 0], c['lrt'], rtol=1e-9, atol=0)
    assert np.allclose(wstat[:, 0], c['lrt'], rtol=1e-9, atol=0)
    assert np.allclose(p[:, 0], chi2.sf(c['lrt'], 3), rtol=1e-9) and np.allclose(wp, p, rtol=1e-9)


def test_conjugate_statistic_is_invariant_to_an_unconverged_theta():
    _, _, (s0, _) = _score_groups(_conjugate(), [[0, 1, 2], [1, 2]])
    _, _, (s1, _) = _score_groups(_conjugate(theta_shift=np.array([[0.05, -0.02, 0.1], [0.1, 0.03, -0.05]])),
                                  [[0, 1, 2], [1, 2]])
    assert np.allclose(s1, s0, rtol=1e-9, atol=0)


def test_singleton_groups_equal_the_one_column_tests():
    c = _conjugate()
    parts, info, (stat, p) = _score_groups(c, [[0], [2], [1]])
    z, _, p1 = score_from_parts(parts, info)
    assert np.allclose(stat, z[:, [0, 2, 1]] ** 2, rtol=1e-12, atol=0)
    assert np.allclose(p, p1[:, [0, 2, 1]], rtol=1e-10)
    info_f = wald_ref.info(c['Z_std_log'], c['sigma_log'], c['Xf'])
    se, _ = wald_from_info(c['coef'], info_f)
    wstat, _ = wald_groups_from_info(c['coef'], info_f, [[k] for k in range(5)])
    assert np.allclose(wstat, (c['coef'] / se) ** 2, rtol=1e-12, atol=0)


def _random_pd(rng, Ng, K):
    Xt = rng.normal(size=(60, K))
    w = rng.uniform(0.2, 1.0, size=(60, Ng))
    return np.einsum('cg,ck,cl->gkl', w, Xt, Xt)


def test_wald_groups_match_a_direct_inverse():
    rng = np.random.default_rng(1)
    info, coef = _random_pd(rng, 6, 5), rng.normal(size=(6, 5))
    groups = [[0, 3], [4, 1, 2], [2]]
    stat, p = wald_groups_from_info(coef, info, groups)
    for g in range(6):
        Ii = np.linalg.inv(info[g])
        for h, G in enumerate(groups):
            want = coef[g, G] @ np.linalg.solve(Ii[np.ix_(G, G)], coef[g, G])
            assert np.isclose(stat[g, h], want, rtol=1e-10)
            assert np.isclose(p[g, h], chi2.sf(want, len(G)), rtol=1e-8)


def test_score_groups_match_a_direct_inverse():
    rng = np.random.default_rng(2)
    Ng, J, K = 7, 6, 3
    Xt, X = rng.normal(size=(50, K)), rng.normal(size=(50, J))
    w, r = rng.uniform(0.2, 1.0, size=(50, Ng)), rng.normal(size=(50, Ng))
    info = np.einsum('cg,ck,cl->gkl', w, Xt, Xt)
    parts = (r.T @ X, w.T @ X ** 2, np.einsum('cg,cj,ck->gjk', w, X, Xt), r.T @ Xt)
    groups = [[0, 1, 2], [5, 3], [4]]
    pairs = group_pairs(groups)
    assert pairs.tolist() == [[0, 1], [0, 2], [1, 2], [3, 5]]
    full = np.einsum('cg,cj,ck->gjk', w, X, X)
    stat, p = score_groups_from_parts(parts, full[:, pairs[:, 0], pairs[:, 1]], pairs, info, groups)
    for g in range(Ng):
        Ii = np.linalg.inv(info[g])
        for h, G in enumerate(groups):
            V = full[g][np.ix_(G, G)] - parts[2][g, G] @ Ii @ parts[2][g, G].T
            Ue = parts[0][g, G] - parts[2][g, G] @ Ii @ parts[3][g]
            want = Ue @ np.linalg.inv(V) @ Ue
            assert np.isclose(stat[g, h], want, rtol=1e-10)
            assert np.isclose(p[g, h], chi2.sf(want, len(G)), rtol=1e-8)


def test_degenerate_groups_and_information():
    c = _conjugate()
    Nc = c['X'].shape[0]
    X = np.stack([c['X'][:, 0], c['X'][:, 0], c['Xt'][:, 0] * 2.0, c['X'][:, 1], c['X'][:, 2], np.zeros(Nc)], axis=1)
    groups = [[0, 1], [3, 2], [3, 5], [3, 4], [0, 4, 3]]
    parts, info, (stat, p) = _score_groups(c, groups, X)
    # copies of each other, a member collinear with the fitted column, a member zero on every cell
    assert np.isnan(stat[:, :3]).all() and (p[:, :3] == 1).all()
    assert np.isfinite(stat[:, 3:]).all() and (p[:, 3:] < 1).all()
    # an information that is not positive definite: the whole event
    bad = info.copy()
    bad[1] = np.array([[1.0, 1.0], [1.0, 1.0]])
    _, _, (stat, p) = _score_groups(c, groups, X, info=bad)
    assert np.isnan(stat[1]).all() and (p[1] == 1).all() and np.isfinite(stat[[0, 2], 3:]).all()
    info_f = wald_ref.info(c['Z_std_log'], c['sigma_log'], c['Xf'])
    info_f[2] = 0.0
    wstat, wp = wald_groups_from_info(c['coef'], info_f, [[2, 3], [0]])
    assert np.isnan(wstat[2]).all() and (wp[2] == 1).all() and np.isfinite(wstat[:2]).all()


def _refusal_cases(Nc):
    sx = np.zeros((Nc, 3))
    return [
        (dict(LRT_groups=[[]]), 'empty'), (dict(LRT_groups=[]), 'at least one'), (dict(LRT_groups=[[0, 0]]), 'repeats'),
        (dict(LRT_groups=[[2]]), 'out of range'), (dict(LRT_groups=[[-1]]), 'out of range'),
        (dict(LRT_groups=[[0.5]]), 'not an integer'), (dict(LRT_groups=[[True]]), 'not an integer'),
        (dict(LRT_groups=[["0"]]), 'not an integer'), (dict(LRT_groups=3), 'list of groups'),
        (dict(LRT_groups=[[0]] * 4096), 'model ids'), (dict(LRT_groups=[[1]] * 4094, n_perm=1), 'model ids'),
        (dict(LRT_groups=[[0, 1]], base_mode='null', LRT_index=[1]), 'overlaps'),
        (dict(wald_groups=[[0, 1]], base_mode='null', LRT_index=[1]), 'does not fit'),
        (dict(wald_groups=[[0, 5]]), 'out of range'),
        (dict(wald_groups=[[0]], target='marginLik'), 'marginLik'),
        (dict(score_groups=[[0, 1]]), 'needs score_X'), (dict(score_groups=[[0]], target='marginLik'), 'marginLik'),
        (dict(score_groups=[[0, 3]], score_X=sx), 'out of range'), (dict(score_groups=[[1, 1]], score_X=sx), 'repeats'),
    ]


def test_refusals_before_any_device_work(monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: (_ for _ in ()).throw(AssertionError("device touched")))
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a: (_ for _ in ()).throw(AssertionError("device touched")))
    from brie_b200.utils.anndata_lite import AnnDataLite
    data = [np.ones((6, 3), np.float32) for _ in range(3)]
    Xc = np.zeros((6, 2), np.float32)
    for kw, msg in _refusal_cases(6):
        kw = dict(dict(LRT_index=[0]), **kw)
        with pytest.raises(ValueError, match=msg):
            fit_BRIE_matrix([d.copy() for d in data], Xc=Xc, **kw)
        ad = AnnDataLite(X=data[0], layers={'isoform1': data[0], 'isoform2': data[1], 'ambiguous': data[2]})
        with pytest.raises(ValueError, match=msg):
            fitBRIE(ad, Xc=Xc, **kw)


@pytest.mark.parametrize("T,cell,full,B", [(2, False, True, 0), (2, False, False, 0), (0, False, True, 0),
                                           (3, True, True, 2), (0, True, True, 0), (40, False, True, 1),
                                           (40, False, False, 0)])
def test_engine_plan_with_groups(T, cell, full, B):
    Kc = max(T, 1) + 3
    base = list(range(Kc)) if full else list(range(T, Kc))
    tested = list(range(T))
    tests = [[k for k in base if k != t] if full else base + [t] for t in tested]
    mode = 'cell' if cell else 'gene'
    plain = _engine_plan(base, tests, cell, mode, n_perm=B, tested=tested, n_cols=Kc, full=full)
    groups = [[0, 1], [2], [1, 0, 2]] * 12                                   # 36 groups
    gm = [[k for k in range(Kc) if k not in G] if full else base + G for G in groups]
    plan = _engine_plan(base, tests, cell, mode, n_perm=B, tested=tested, n_cols=Kc, full=full, group_masks=gm)
    assert plan[:len(plain)] == plain                                         # observed and permuted engines unchanged
    extra = plan[len(plain):]
    size = min(max(len(ids) for _, ids, _ in plain if max(ids) <= T), 32)       # the largest observed engine
    assert all(len(ids) <= size for _, ids, _ in extra) and all(len(ids) == size for _, ids, _ in extra[:-1])
    assert [m for ms, _, _ in extra for m in ms] == gm
    assert [i for _, ids, _ in extra for i in ids] == [group_model_id(i, T, B) for i in range(len(groups))]
    assert all(mode_e == 'gene' for _, _, mode_e in extra)
    assert group_model_id(0, T, B) == 1 + T * (1 + B) and (B == 0 or group_model_id(0, T, B) == perm_model_id(T - 1, B - 1, T, B) + 1)


def _rv(rng, Ng):
    r = BRIE_RV()
    r.Nc, r.Ng, r.intercept_mode = 5, Ng, 'gene'
    r.losses = np.zeros(3)
    r.loss_gene = rng.normal(size=Ng)
    for k, shape in (('sigma', (1, Ng)), ('intercept', (1, Ng)), ('cell_coeff', (2, Ng)), ('Psi', (5, Ng)),
                     ('Psi95CI', (5, Ng)), ('Z_std', (5, Ng)), ('Z_loc', (5, Ng))):
        setattr(r, k, rng.normal(size=shape))
    for (sk, pk, _), H in zip(GROUP_KEYS, (2, 3, 1)):
        setattr(r, sk, rng.normal(size=(Ng, H)))
        setattr(r, pk, rng.uniform(size=(Ng, H)))
    _set_fdr_groups(r)
    return r


@pytest.mark.parametrize("merge", ["concate", "shared"])
def test_chunks_and_ranks_carry_the_group_outputs(merge):
    rng = np.random.default_rng(5)
    a, b = _rv(rng, 4), _rv(rng, 3)
    want = {k: np.concatenate([getattr(a, k), getattr(b, k)]) for sk, pk, _ in GROUP_KEYS for k in (sk, pk)}
    if merge == "concate":
        a.concate(b)
        out = a
    else:
        out = _merge_shared([a, b])
    _set_fdr_groups(out)
    for k, v in want.items():
        assert np.array_equal(getattr(out, k), v), k
    for _, pk, fk in GROUP_KEYS:
        for j in range(want[pk].shape[1]):
            assert np.array_equal(getattr(out, fk)[:, j], fdr_bh(want[pk][:, j]))   # pooled over both parts


def _group_adata():
    import pandas as pd
    from brie_b200.utils.anndata_lite import AnnDataLite
    rng = np.random.default_rng(0)
    X = rng.poisson(0.3, (6, 4)).astype(np.float32)
    ad = AnnDataLite(X=X, var=pd.DataFrame({'n_counts': X.sum(0), 'n_counts_uniq': X.sum(0)},
                                           index=pd.Index(list("abcd"), name="GeneID")))
    for (sk, pk, fk), H in zip(GROUP_KEYS, (2, 1, 1)):
        for k in (sk, pk, fk):
            ad.varm[k] = rng.uniform(size=(4, H))
    ad.varm['score_z'] = ad.varm['pval_score'] = ad.varm['fdr_score'] = rng.uniform(size=(4, 3))
    ad.uns['brie_param'] = {'LRT_index': [], 'LRT_groups': [[1, 2], [0]], 'wald_groups': [[2, 0]],
                            'score_groups': [[0, 2]], 'score': 3}
    ad.uns['Xc_ids'] = np.array(['sex', 'clusterB', 'clusterC'])
    ad.uns['score_ids'] = np.array(['RBFOX2', 'rs1', 'rs2'])
    return ad


def test_tables_and_container_round_trip(tmp_path):
    from brie_b200.utils.anndata_lite import AnnDataLite
    from brie_b200.utils.io_utils import dump_results, score_table
    ad = _group_adata()
    t = dump_results(ad)
    assert list(t.columns)[-8:] == ['clusterB+clusterC_ELBO_gain_group', 'clusterB+clusterC_pval_group',
                                    'clusterB+clusterC_FDR_group', 'sex_ELBO_gain_group', 'sex_pval_group',
                                    'sex_FDR_group', 'clusterC+sex_pval_wald_group', 'clusterC+sex_FDR_wald_group']
    assert np.array_equal(t['sex_FDR_group'].values, ad.varm['fdr_group'][:, 1])
    s = score_table(ad)
    assert list(s.columns)[-3:] == ['RBFOX2+rs2_score_stat_group', 'RBFOX2+rs2_pval_score_group',
                                    'RBFOX2+rs2_FDR_score_group']
    assert np.array_equal(s['RBFOX2+rs2_score_stat_group'].values, ad.varm['score_stat_group'][:, 0])
    p = str(tmp_path / "out.npz")
    ad.write_npz(p)
    back = AnnDataLite.read_npz(p)
    for keys in GROUP_KEYS:
        for k in keys:
            assert np.array_equal(back.varm[k], ad.varm[k]), k
    for k in ('LRT_groups', 'wald_groups', 'score_groups'):
        assert back.uns['brie_param'][k] == ad.uns['brie_param'][k]


def test_cli_group_options_parse_and_reach_fitBRIE(tmp_path, monkeypatch, capsys):
    import brie_b200.models as models
    from brie_b200.bin import quant as q
    seen = {}

    class Stop(Exception):
        pass

    def spy_fit(adata, **kw):
        seen['fit'] = kw
        raise Stop()
    inp, cells = _cli_input(tmp_path)
    cf, sf = tmp_path / "cell.tsv", tmp_path / "score.tsv"
    cf.write_text("\n".join(["cellID\ta\tb\tc"] + ["%s\t%d\t%d\t%d" % (c, i % 2, i % 3 == 1, i % 3 == 2)
                                                   for i, c in enumerate(cells)]) + "\n")
    sf.write_text("\n".join(["cellID\tx\ty"] + ["%s\t%d\t%.1f" % (c, i, 0.5 * i) for i, c in enumerate(cells)]) + "\n")
    monkeypatch.setattr(q, "filter_genes", lambda adata, **kw: adata)
    monkeypatch.setattr(models, "fitBRIE", spy_fit)
    base = ["brie-quant", "-i", inp, "-o", str(tmp_path / "o.npz"), "-c", str(cf)]
    monkeypatch.setattr(sys, "argv", base)
    with pytest.raises(Stop):
        q.main()
    assert not any(k in seen['fit'] for k in ('LRT_groups', 'wald_groups', 'score_groups'))
    monkeypatch.setattr(sys, "argv", base + ["--LRTgroups", "1,2;0", "--waldGroups", "2,1", "--scoreFile", str(sf),
                                             "--scoreGroups", "0,1"])
    with pytest.raises(Stop):
        q.main()
    f = seen['fit']
    assert f['LRT_groups'] == [[1, 2], [0]] and f['wald_groups'] == [[2, 1]] and f['score_groups'] == [[0, 1]]
    for extra, msg in ((["--LRTgroups", "1,x"], "--LRTgroups needs"), (["--waldGroups", "1;;2"], "--waldGroups needs"),
                       (["--scoreGroups", "0,1"], "--scoreGroups needs --scoreFile"),
                       (["--LRTgroups", "1,3"], "out of range"), (["--LRTgroups", "1,1"], "repeats"),
                       (["--scoreFile", str(sf), "--scoreGroups", "0,2"], "out of range")):
        monkeypatch.setattr(sys, "argv", base + extra)
        with pytest.raises(SystemExit) as e:
            q.main()
        assert e.value.code == 1 and msg in capsys.readouterr().out, extra
    out = __import__('subprocess').run([sys.executable, "-m", "brie_b200.bin.quant", "--help"], capture_output=True,
                                       text=True, timeout=300)
    assert out.returncode == 0 and all(o in out.stdout for o in ("--LRTgroups", "--waldGroups", "--scoreGroups"))


def test_abi_refusals_on_fake_addresses():
    """brie_fit_score_cross_sizes / brie_fit_score_cross refuse a null or unbound fit, a model out of range, a gathered
    sub-fit, target marginLik, n_pairs <= 0, pairs out of range and null or misaligned X, pairs, output or scratch,
    before any copy or launch."""
    import torch
    from brie_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("a refusal missed here would copy to fake addresses")
    lib = _lib.load()
    ARG, UNSUP = -1, -3
    sz = C.c_size_t()
    ok = np.array([[0, 1], [1, 3]], np.int32)
    P = lambda a: a.ctypes.data                                      # a: an int32 array kept alive by the caller
    X, out, scr = 0x10000000, 0x20000000, 0x30000000
    assert lib.brie_fit_score_cross_sizes(None, 0, 2, C.byref(sz)) == ARG
    assert lib.brie_fit_score_cross(None, 0, X, 4, P(ok), 2, out, scr, None) == ARG
    h = C.c_void_p()
    assert lib.brie_fit_create(C.byref(_lib.FitDesc(n_cells=10, n_events=4, ld=32, n_models=1, n_layers=2,
                                                    mc_size=1, trace_cap=1)), C.byref(h)) == 0
    assert lib.brie_fit_score_cross_sizes(h, 0, 2, C.byref(sz)) == ARG and b"not bound" in lib.brie_last_error()
    lib.brie_fit_destroy(h)
    h = _bind_fake(lib)
    try:
        assert lib.brie_fit_score_cross_sizes(h, 0, 2, C.byref(sz)) == 0 and sz.value > 0
        assert lib.brie_fit_score_cross_sizes(h, 0, 2, None) == ARG
        for m, n in ((-1, 2), (1, 2), (0, 0), (0, -3)):
            assert lib.brie_fit_score_cross_sizes(h, m, n, C.byref(sz)) == ARG
        call = lambda *a: lib.brie_fit_score_cross(h, *a, None)
        assert call(1, X, 4, P(ok), 2, out, scr) == ARG                                  # model out of range
        assert call(0, X, 4, P(ok), 0, out, scr) == ARG                                  # n_pairs <= 0
        assert call(0, 0, 4, P(ok), 2, out, scr) == ARG                                  # no X
        assert call(0, X, 4, None, 2, out, scr) == ARG                                   # no pairs
        for bad in ([[0, 1], [1, 4]], [[-1, 1]], [[2, 2]], [[3, 1]]):                    # j' >= ldx, j < 0, j >= j'
            bad = np.array(bad, np.int32)
            assert call(0, X, 4, bad.ctypes.data, len(bad), out, scr) == ARG, bad
            assert b"pair" in lib.brie_last_error()
        assert call(0, X, 3, P(ok), 2, out, scr) == ARG                                  # ldx too small
        for o, s in ((0, scr), (out + 4, scr), (out, 0), (out, scr + 4)):
            assert call(0, X, 4, P(ok), 2, o, s) == ARG
        assert lib.brie_fit_launch_count(h) == 0
    finally:
        lib.brie_fit_destroy(h)
    for kw, what in ((dict(target=1), b"target ELBO"), (dict(counts_model_stride=100 * 64), b"parent")):
        h = _bind_fake(lib, **kw)
        assert lib.brie_fit_score_cross_sizes(h, 0, 2, C.byref(sz)) == UNSUP and what in lib.brie_last_error()
        assert lib.brie_fit_score_cross(h, 0, X, 4, P(ok), 2, out, scr, None) == UNSUP
        assert lib.brie_fit_launch_count(h) == 0
        lib.brie_fit_destroy(h)
