"""Count-matrix loaders and the result table (semantics of brie/utils/io_utils.py).

`anndata` / `h5py` are used when importable; otherwise the AnnDataLite duck type and
its npz persistence stand in (the image has neither package).
"""
import numpy as np
import pandas as pd

try:  # pragma: no cover - not installable in the build image
    import anndata as _anndata
except ImportError:
    _anndata = None

from .anndata_lite import AnnDataLite


def _make_adata(**kw):
    if _anndata is not None:
        return _anndata.AnnData(**kw)
    return AnnDataLite(**kw)


def read_h5ad(path):
    if _anndata is not None:
        return _anndata.read_h5ad(path)
    if str(path).endswith(".npz"):
        return AnnDataLite.read_npz(path)
    raise RuntimeError("brie_b200: reading .h5ad needs the `anndata` package; "
                       "use the brie .npz count format (read_npz) in this environment")


def convert_to_annData(Rmat_dict, effLen_tensor, cell_note, gene_note, fill_missing=True):
    """Count matrices keyed '0'..'3' + effective-length tensor (Ng, 2, 3) -> AnnData with layers
    isoform1/isoform2/ambiguous/poorQual, X = 1+2+3, varm['effLen'] (Ng, 6) = [iso1 | iso2],
    varm['p_ambiguous'] (io_utils.py:12-52)."""
    Rmat = {k: v.astype(np.float32) for k, v in Rmat_dict.items()}
    if fill_missing:
        shape = next(iter(Rmat.values())).shape
        for k in ['0', '1', '2', '3']:
            if k not in Rmat:
                print("key %s not exist in .mtx file, fill with zeros." % (k))
                Rmat[k] = np.zeros(shape, dtype=np.float32)
    layers = {'isoform1': Rmat['1'], 'isoform2': Rmat['2'], 'ambiguous': Rmat['3'], 'poorQual': Rmat['0']}
    obs = pd.DataFrame(cell_note[1:, :], index=cell_note[1:, 0], columns=cell_note[0, :])
    var = pd.DataFrame(gene_note[1:, :], index=gene_note[1:, 0], columns=gene_note[0, :])
    prob = effLen_tensor / effLen_tensor.sum(2, keepdims=True)
    varm = {'effLen': np.append(effLen_tensor[:, 0, :], effLen_tensor[:, 1, :], axis=1),
            'p_ambiguous': prob[:, :, 2]}
    return _make_adata(X=Rmat['1'] + Rmat['2'] + Rmat['3'], obs=obs, var=var, varm=varm, layers=layers)


def read_npz(path):
    """brie-count's npz (keys cell_note, gene_note, Rmat_dict, effLen_tensor; io_utils.py:55-65)."""
    dat = np.load(path, allow_pickle=True)
    return convert_to_annData(dat['Rmat_dict'].item(), dat['effLen_tensor'], dat['cell_note'], dat['gene_note'])


def write_npz_counts(path, layers, effLen_tensor, cell_ids, gene_ids):
    """Writer for the same npz format (used by tests and the synthetic-data tools)."""
    from scipy.sparse import csc_matrix
    keys = {'isoform1': '1', 'isoform2': '2', 'ambiguous': '3'}
    Rmat = {keys[k]: csc_matrix(v) for k, v in layers.items()}
    cell_note = np.array([["cellID"]] + [[c] for c in cell_ids], dtype=object)
    gene_note = np.array([["GeneID"]] + [[g] for g in gene_ids], dtype=object)
    np.savez(path, Rmat_dict=np.array(Rmat, dtype=object), effLen_tensor=effLen_tensor,
             cell_note=cell_note, gene_note=gene_note)


def dump_results(adata):
    """Per-event result table of the detected splicing phenotypes, the table brie-quant writes as
    <out>.brie_ident.tsv (io_utils.py:163-199; header pinned on the published tables in
    tests/golden/published_lrt.npz).  Keeps the reference's `_ceoff` spelling and its indexing of
    cell_coeff by loop position rather than by LRT_index (SURVEY appendix B.2)."""
    n_events = adata.shape[1]
    table = adata.var[['n_counts', 'n_counts_uniq']].astype(int)
    # cell detection rate per event; a caller that no longer holds the counts may supply var['cdr']
    table['cdr'] = (np.asarray(adata.var['cdr']) if 'cdr' in adata.var
                    else np.asarray((adata.X > 0).mean(0)).reshape(-1))
    for key in ('intercept', 'sigma'):
        table[key] = adata.varm[key][:, 0] if key in adata.varm else [None] * n_events
    tested = adata.uns['brie_param']['LRT_index'] if 'brie_param' in adata.uns else []
    names = adata.uns['Xc_ids'] if 'Xc_ids' in adata.uns else None
    for pos, feature in enumerate(tested):
        label = names[feature] if names is not None else 'X%d' % pos
        for suffix, source in (('_ceoff', 'cell_coeff'), ('_ELBO_gain', 'ELBO_gain'),
                               ('_pval', 'pval'), ('_FDR', 'fdr')):
            table[label + suffix] = adata.varm[source][:, pos]
    if 'pval_perm' in adata.varm:          # permutation null (brie-quant --nPerm): after all the reference's columns
        for pos, feature in enumerate(tested):
            label = names[feature] if names is not None else 'X%d' % pos
            table[label + '_pval_perm'] = adata.varm['pval_perm'][:, pos]
            table[label + '_FDR_perm'] = adata.varm['fdr_perm'][:, pos]
    if 'pval_wald' in adata.varm:          # Wald tests (brie-quant --wald): one set per cell_coeff row, labelled by
        for j, feature in enumerate(adata.uns['brie_param']['wald_columns']):    # its covariate, after all others
            label = names[feature] if names is not None else 'X%d' % feature
            table[label + '_se'] = adata.varm['cell_coeff_se'][:, j]
            table[label + '_pval_wald'] = adata.varm['pval_wald'][:, j]
            table[label + '_FDR_wald'] = adata.varm['fdr_wald'][:, j]
    param = adata.uns['brie_param'] if 'brie_param' in adata.uns else {}
    label = lambda G: '+'.join(str(names[k]) if names is not None else 'X%d' % k for k in G)
    if 'LRT_groups' in param:              # joint tests of groups of covariates, labelled <id>+<id>+..., after all others
        for i, G in enumerate(param['LRT_groups']):
            table[label(G) + '_ELBO_gain_group'] = adata.varm['ELBO_gain_group'][:, i]
            table[label(G) + '_pval_group'] = adata.varm['pval_group'][:, i]
            table[label(G) + '_FDR_group'] = adata.varm['fdr_group'][:, i]
    if 'wald_groups' in param:
        for i, G in enumerate(param['wald_groups']):
            table[label(G) + '_pval_wald_group'] = adata.varm['pval_wald_group'][:, i]
            table[label(G) + '_FDR_wald_group'] = adata.varm['fdr_wald_group'][:, i]
    return table


def score_table(adata):
    """Per-event table of the score tests of candidate cell covariates (brie-quant --scoreFile), written as
    <out>.brie_score.tsv: per candidate, in uns['score_ids'] order, <id>_score_z, <id>_pval_score, <id>_FDR_score;
    then per group of candidates (--scoreGroups) <id>+<id>..._score_stat_group, _pval_score_group, _FDR_score_group."""
    table = pd.DataFrame(index=adata.var.index)
    for j, cid in enumerate(adata.uns['score_ids']):
        table[str(cid) + '_score_z'] = adata.varm['score_z'][:, j]
        table[str(cid) + '_pval_score'] = adata.varm['pval_score'][:, j]
        table[str(cid) + '_FDR_score'] = adata.varm['fdr_score'][:, j]
    ids = adata.uns['score_ids']
    for i, G in enumerate(adata.uns['brie_param'].get('score_groups', [])):    # then per group of candidates
        label = '+'.join(str(ids[j]) for j in G)
        table[label + '_score_stat_group'] = adata.varm['score_stat_group'][:, i]
        table[label + '_pval_score_group'] = adata.varm['pval_score_group'][:, i]
        table[label + '_FDR_score_group'] = adata.varm['fdr_score_group'][:, i]
    return table
