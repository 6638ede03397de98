"""CPU tests of the host-side product code: the C-ABI library loads and exports every
declared symbol (no compute without a GPU), argument validation, host noise dump, the
reference-side helpers against golden vectors from the reference, sharding logic under
a 2-process gloo group."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import philox_np as px

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"), allow_pickle=True)


def test_library_exports_every_declared_symbol(lib):
    from brie_b200 import _lib
    header = open(os.path.join(ROOT, "include", "brie_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(brie_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), "missing export: " + name
    assert declared == set(_lib.SYMBOLS), "ctypes table and header disagree"
    assert lib.brie_abi_version() == _lib.ABI_VERSION


def test_struct_layout_matches_header():
    from brie_b200 import _lib
    assert C.sizeof(_lib.FitDesc) == 4 * 8 + 8 + 12 * 4 + 32 * 4 + 32 * 4 + 32 * 4
    assert C.sizeof(_lib.FitBuffers) == 20 * 8      # + event_ids, counts_model_stride, efflen_model_stride (ABI 4)
    assert C.sizeof(_lib.FitSizes) == 2 * 8 + 4 * 4


def _desc(**kw):
    from brie_b200 import _lib
    d = _lib.FitDesc()
    d.n_cells, d.n_events, d.ld, d.event_offset, d.seed = 100, 50, 64, 0, 1
    d.n_models, d.Kc, d.Kg, d.mc_size, d.n_layers = 1, 1, 0, 3, 3
    d.has_efflen, d.cell_mode, d.train_intercept, d.train_sigma, d.trace_cap = 1, 0, 1, 1, 8
    d.xc_mask[0] = 1
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def test_create_validates_arguments(lib):
    from brie_b200 import _lib
    h = C.c_void_p()
    assert lib.brie_fit_create(C.byref(_desc()), C.byref(h)) == 0
    sz = _lib.FitSizes()
    assert lib.brie_fit_get_sizes(h, C.byref(sz)) == 0
    assert sz.scratch_bytes > 0 and sz.n_col_tiles == 1 and sz.n_row_chunks * sz.rows_per_cta >= 100
    # not bound -> error code + message, no crash
    assert lib.brie_fit_run_steps(h, 1, -1, None) < 0
    assert b"not bound" in lib.brie_last_error()
    lib.brie_fit_destroy(h)
    for bad in (dict(ld=50), dict(ld=62), dict(Kc=3), dict(Kg=5), dict(Kc=5000), dict(Kg=-1), dict(n_models=0), dict(n_models=33),
                dict(mc_size=0), dict(n_layers=4), dict(n_cells=0), dict(event_offset=-1), dict(rows_per_cta=-1)):
        assert lib.brie_fit_create(C.byref(_desc(**bad)), C.byref(h)) < 0, bad
        assert len(lib.brie_last_error()) > 0
    d = _desc()
    d.xc_mask[0] = 2                      # bit beyond Kc
    assert lib.brie_fit_create(C.byref(d), C.byref(h)) < 0
    # widths beyond the register-resident instantiations select the wide (GEMM) form: accepted, scratch grows
    # by the prior-mean / residual planes and the Wc gradient
    dw = _desc(Kc=24)
    dw.xc_mask[0] = 0
    dw.xc_width[0] = 24
    assert lib.brie_fit_create(C.byref(dw), C.byref(h)) == 0
    szw = _lib.FitSizes()
    assert lib.brie_fit_get_sizes(h, C.byref(szw)) == 0
    assert szw.scratch_bytes >= (2 * 100 * 64 + 24 * 64) * 4 and szw.n_col_tiles == 1
    lib.brie_fit_destroy(h)
    assert lib.brie_fit_create(C.byref(_desc(Kc=24, target=1)), C.byref(h)) < 0     # marginLik: narrow designs only
    # a caller-fixed rows_per_cta (gathered sub-fits keep their parent's) is honoured
    assert lib.brie_fit_create(C.byref(_desc(rows_per_cta=16)), C.byref(h)) == 0
    assert lib.brie_fit_get_sizes(h, C.byref(sz)) == 0 and sz.rows_per_cta == 16 and sz.n_row_chunks == 7
    assert lib.brie_fit_resume_stage(h, 0.01, 5, 7) < 0 and b"not bound" in lib.brie_last_error()
    lib.brie_fit_destroy(h)


def _bind_fake(lib, counts, **buffers):
    """A narrow fit (Kc = 1, no lengths) bound to fake 16-byte-aligned addresses: brie_fit_bind reads no memory of
    such a fit, so the argument checks run without a device.  None of these addresses may reach a launch."""
    from brie_b200 import _lib
    h = C.c_void_p()
    assert lib.brie_fit_create(C.byref(_desc(has_efflen=0)), C.byref(h)) == 0
    b = _lib.FitBuffers()
    fake = iter(range(0x10000, 0x1000000, 0x1000))
    for name in ("Xc", "Z_loc", "Z_std_log", "adam_Z", "Wc", "intercept", "sigma_log", "adam_small", "active",
                 "loss_trace", "scratch"):
        setattr(b, name, next(fake))
    for i in range(3 if counts else 0):
        b.counts[i] = next(fake)
    for name, v in buffers.items():
        setattr(b, name, next(fake) if v is True else v)
    assert lib.brie_fit_bind(h, C.byref(b)) == 0, lib.brie_last_error()
    return h, b


def test_refused_step_leaves_the_adam_step_alone(lib):
    """A step that phase 0 refuses (here: a sub-fit with neither count tiles nor count codes) changes no state."""
    h, _ = _bind_fake(lib, counts=False, event_ids=True)
    assert lib.brie_fit_resume_stage(h, 0.01, 0, 0) == 0
    assert lib.brie_fit_run_steps(h, 1, -1, None) == -1
    assert b"neither count tiles nor count codes" in lib.brie_last_error()
    t, step = C.c_int64(-1), C.c_uint32(7)
    assert lib.brie_fit_get_step(h, C.byref(t), C.byref(step)) == 0
    assert (t.value, step.value) == (0, 0)
    assert lib.brie_fit_launch_count(h) == 0
    lib.brie_fit_destroy(h)


def test_subfit_is_refused_by_every_entry_but_the_step(lib):
    """A per-model count stride alone makes a sub-fit (brie_fit_buffers): loss_gene, element terms, Wald and the group
    trace work on the parent fit only and refuse it before any launch."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a refusal missed here would launch on fake addresses")
    h, b = _bind_fake(lib, counts=True, counts_model_stride=100 * 64)
    out = 0x2000000
    nbytes, kt = C.c_size_t(), C.c_int32()
    calls = {
        "eval_loss_gene": lambda: lib.brie_fit_eval_loss_gene(h, 1, 1, out, None),
        "element_terms": lambda: lib.brie_fit_element_terms(h, 0, b.counts[0], b.counts[1], b.counts[2], 1, 0, 0,
                                                            out, None, None, None),
        "wald_sizes": lambda: lib.brie_fit_wald_sizes(h, 0, C.byref(nbytes), C.byref(kt)),
        "group_trace": lambda: lib.brie_fit_group_trace(h, 1, 1, 1, out, None),
    }
    for name, call in calls.items():
        assert call() == -3, name
        assert b"parent" in lib.brie_last_error(), name
    assert lib.brie_fit_launch_count(h) == 0
    lib.brie_fit_destroy(h)


def test_host_normals_match_numpy_spec(lib):
    from brie_b200 import _lib
    S, R, Cn, off = 5, 7, 19, 4000
    out = np.empty((S, R, Cn), np.float32)
    _lib.check(lib.brie_philox_normals_host(1234567890123, 1, 9, 77, S, R, Cn, off, out.ctypes.data))
    ref = px.normal_field(R, Cn, 77, 1, 9, 1234567890123, S, col_offset=off)
    assert np.abs(out - ref).max() < 2e-6


def test_product_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from brie_b200.engine import FitEngine
    with pytest.raises(RuntimeError, match="no CUDA device"):
        FitEngine([np.zeros((4, 4), np.float32)] * 2)


def test_match_against_reference_golden():
    from brie_b200.utils.base_utils import match
    idx = match(GOLD['match_ref'], GOLD['match_new'])
    got = np.array([-1 if v is None else int(v) for v in idx])
    assert np.array_equal(got, GOLD['match_idx'])
    f = idx.astype(float)                 # quant.py:53-55 idiom
    assert np.array_equal(f == f, got >= 0)


def test_filter_genes_against_reference_golden():
    from brie_b200.utils.preprocessing import filter_genes
    from brie_b200.utils.anndata_lite import AnnDataLite
    from scipy.sparse import csc_matrix
    for wrap in (lambda x: x, csc_matrix):
        ad = AnnDataLite(X=GOLD['fg_l1'] + GOLD['fg_l2'] + GOLD['fg_l3'],
                         layers={'isoform1': wrap(GOLD['fg_l1']), 'isoform2': wrap(GOLD['fg_l2']),
                                 'ambiguous': wrap(GOLD['fg_l3'])})
        out = filter_genes(ad, min_counts=50, min_counts_uniq=10, min_cells_uniq=30, min_MIF_uniq=0.001, copy=True)
        assert out.shape == (80, int(GOLD['fg_subset'].sum()))
        assert np.array_equal(np.asarray(out.var['n_counts']), GOLD['fg_n_counts'])
        assert np.array_equal(np.asarray(out.var['n_counts_uniq']), GOLD['fg_n_counts_uniq'])
        l1 = out.layers['isoform1']
        l1 = l1.toarray() if hasattr(l1, 'toarray') else l1
        assert np.array_equal(l1, GOLD['fg_l1'][:, GOLD['fg_subset']])
        assert ad.shape == (80, 120)      # copy=True leaves the input alone


def test_fdr_bh_matches_oracle():
    from brie_b200.models.model_wrap import fdr_bh
    from oracle.brie2_oracle import fdr_bh as ofdr
    rng = np.random.default_rng(0)
    p = rng.uniform(size=200) ** 3
    p[:5] = p[5:10]                       # ties
    assert np.allclose(fdr_bh(p), ofdr(p))
    assert fdr_bh(np.array([])).size == 0


def test_event_shards_properties():
    from brie_b200.sharding import event_shards
    for n, w, g in [(5000, 8, 100), (5000, 3, 100), (20000, 8, 1), (17, 4, 5), (3, 8, 1), (1000, 1, 7)]:
        sh = event_shards(n, w, g)
        assert len(sh) == w and sh[0][0] == 0 and sh[-1][1] == n
        for (a, b), (c, d) in zip(sh[:-1], sh[1:]):
            assert b == c and a <= b
        assert all(a % g == 0 for a, _ in sh if a < n)
        sizes = [-(-(b - a) // g) for a, b in sh]
        assert max(sizes) - min(sizes) <= 1


def test_sharded_gather_two_process_gloo(tmp_path):
    """world_size 2 on CPU (gloo): each rank owns an aligned event shard, results are gathered
    along the event axis and equal the un-sharded array."""
    script = tmp_path / "w.py"
    script.write_text('''
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch.distributed as dist
from brie_b200.sharding import event_shards, gather_event_axis
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
Nc, Ng, gs = 7, 53, 5
full = np.arange(Nc * Ng, dtype=np.float32).reshape(Nc, Ng)
a, b = event_shards(Ng, w, gs)[r]
got = gather_event_axis(full[:, a:b].copy(), 1)
lg = gather_event_axis(full[0, a:b].copy(), 0)
assert np.array_equal(got, full) and np.array_equal(lg, full[0])
dist.destroy_process_group()
print("rank", r, "ok")
''' % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29631", str(script)],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


def test_layer_store_ram_and_memmap(tmp_path):
    from brie_b200.utils.layer_store import LayerStore, BIG_KEYS
    from brie_b200.models.model_wrap import BRIE_RV
    rng = np.random.default_rng(0)
    Nc, Ng = 9, 41
    full = {k: rng.standard_normal((Nc, Ng)).astype(np.float32) for k in BIG_KEYS}
    for out_dir in (None, str(tmp_path / "layers")):
        st = LayerStore(Nc, Ng, out_dir)
        for e0, e1 in [(0, 16), (16, 17), (17, 41)]:            # ragged chunks
            rv = BRIE_RV()
            rv.Nc, rv.Ng = Nc, e1 - e0
            for k in BIG_KEYS:
                setattr(rv, k, full[k][:, e0:e1].copy())
            st.put(e0, rv)
            assert rv.Psi.shape == (Nc, 0)                      # stub left behind for concate()
        got = st.finish()
        for k in BIG_KEYS:
            assert np.array_equal(np.asarray(got[k]), full[k])
        if out_dir:
            assert np.array_equal(np.load(os.path.join(out_dir, "Psi.npy")), full['Psi'])


def test_layer_store_checkpoint_and_resume(tmp_path):
    """Finished chunks leave a checkpoint; a resumed store with the same signature hands them back
    and keeps the big arrays, a different signature (or resume=False) starts from scratch."""
    from brie_b200.utils.layer_store import LayerStore, BIG_KEYS
    from brie_b200.models.model_wrap import BRIE_RV
    rng = np.random.default_rng(1)
    Nc, Ng = 7, 30
    full = {k: rng.standard_normal((Nc, Ng)).astype(np.float32) for k in BIG_KEYS}
    out_dir = str(tmp_path / "ckpt")
    sig = dict(n_cells=Nc, n_events=Ng, fit=dict(seed=3, min_iter=600), LRT_index=[0])

    def chunk(e0, e1):
        rv = BRIE_RV()
        rv.Nc, rv.Ng = Nc, e1 - e0
        rv.loss_gene = np.arange(e0, e1, dtype=np.float32)
        for k in BIG_KEYS:
            setattr(rv, k, full[k][:, e0:e1].copy())
        return rv

    st = LayerStore(Nc, Ng, out_dir, signature=sig, resume=True)      # nothing to resume yet
    assert not st.resumed and st.load_chunk(0, 10) is None
    st.put(0, chunk(0, 10))
    st.put(10, chunk(10, 20))                                         # ... and the job dies here
    del st
    st = LayerStore(Nc, Ng, out_dir, signature=sig, resume=True)
    assert st.resumed
    done = [st.load_chunk(0, 10), st.load_chunk(10, 20)]
    assert all(d is not None for d in done) and st.load_chunk(20, 30) is None
    assert np.array_equal(done[1].loss_gene, np.arange(10, 20, dtype=np.float32)) and done[1].Psi.shape == (Nc, 0)
    st.put(20, chunk(20, 30))
    got = st.finish()
    for k in BIG_KEYS:
        assert np.array_equal(np.asarray(got[k]), full[k])
    # another fit in the same directory does not pick these chunks up
    st = LayerStore(Nc, Ng, out_dir, signature=dict(sig, fit=dict(seed=4, min_iter=600)), resume=True)
    assert not st.resumed and st.load_chunk(0, 10) is None
    assert not any(f.startswith("chunk_") for f in os.listdir(out_dir))
    st = LayerStore(Nc, Ng, out_dir, signature=sig, resume=False)
    assert not st.resumed


def test_layer_store_two_process_gloo(tmp_path):
    """world_size 2 (gloo): both ranks write their event ranges; RAM mode exchanges blocks,
    memmap mode shares the files -- every rank ends with the full arrays."""
    script = tmp_path / "w.py"
    script.write_text('''
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch.distributed as dist
from brie_b200.sharding import event_shards
from brie_b200.utils.layer_store import LayerStore
from brie_b200.models.model_wrap import BRIE_RV
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
Nc, Ng = 5, 37
full = np.arange(Nc * Ng, dtype=np.float32).reshape(Nc, Ng)
a, b = event_shards(Ng, w, 4)[r]
for out_dir in (None, %r):
    st = LayerStore(Nc, Ng, out_dir, r, w, dist, keys=("Psi",))
    for e0 in range(a, b, 6):
        rv = BRIE_RV(); rv.Nc = Nc; rv.Ng = min(e0 + 6, b) - e0
        rv.Psi = full[:, e0:e0 + rv.Ng].copy()
        st.put(e0, rv)
    got = st.finish()
    assert np.array_equal(np.asarray(got["Psi"]), full), (r, out_dir)
dist.destroy_process_group()
print("rank", r, "ok")
''' % (ROOT, str(tmp_path / "shared")))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29633", str(script)],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.count("ok") == 2

@pytest.mark.parametrize("table", ["msEAE", "scNT", "dentate"])
def test_fdr_by_group_reproduces_published_reference_tables(table):
    """The product's multiple-testing scope (fdr_by_group over convergence groups of
    ceil(batch_size / n_cells) events, any chunking / sharding of the events) reproduces the FDR
    columns of the reference's published result tables (tests/golden/published_lrt.npz)."""
    from brie_b200.models.model_wrap import fdr_by_group
    from brie_b200.sharding import event_shards
    pub = np.load(os.path.join(ROOT, "tests", "golden", "published_lrt.npz"), allow_pickle=True)
    pval, fdr = pub[table + "_pval"], pub[table + "_fdr"]
    n_gene = int(np.ceil(int(pub[table + "_batch_size"]) / int(pub[table + "_n_cells"])))
    Ng = len(pval)
    got = fdr_by_group(pval, n_gene, 0)
    assert np.all(np.abs(got - fdr) <= 2e-3 * fdr)
    # fitted as 3 rank shards (group-aligned), each in chunks of 4 groups, as fitBRIE does
    parts = []
    for lo, hi in event_shards(Ng, 3, n_gene):
        for e0 in range(lo, hi, 4 * n_gene):
            e1 = min(e0 + 4 * n_gene, hi)
            parts.append(fdr_by_group(pval[e0:e1], n_gene, e0))
    assert np.array_equal(np.concatenate(parts, 0), got)
    assert not np.allclose(fdr_by_group(pval, None), fdr, rtol=1e-2)


def test_dump_results_header_matches_published_table():
    """Column names and order of the result table (io_utils.py:163-199) against the header of the
    reference's published msEAE table, including the '_ceoff' spelling."""
    import pandas as pd
    from brie_b200.utils.anndata_lite import AnnDataLite
    from brie_b200.utils.io_utils import dump_results
    pub = np.load(os.path.join(ROOT, "tests", "golden", "published_lrt.npz"), allow_pickle=True)
    rng = np.random.default_rng(0)
    X = rng.poisson(0.3, (6, 4)).astype(np.float32)
    ad = AnnDataLite(X=X, var=pd.DataFrame({'n_counts': X.sum(0), 'n_counts_uniq': X.sum(0)},
                                           index=pd.Index(list("abcd"), name="GeneID")))
    ad.varm['intercept'] = rng.normal(size=(4, 1))
    ad.varm['sigma'] = rng.uniform(size=(4, 1))
    for k in ('cell_coeff', 'ELBO_gain', 'pval', 'fdr'):
        ad.varm[k] = rng.uniform(size=(4, 2 if k == 'cell_coeff' else 1))
    ad.uns['brie_param'] = {'LRT_index': [0]}
    ad.uns['Xc_ids'] = ['isEAE', 'isCD1']
    df = dump_results(ad)
    assert [df.index.name] + list(df.columns) == list(pub['msEAE_columns'])
    line = df.to_csv(sep='\t', float_format='%.3e').splitlines()[1].split('\t')
    assert len(line) == 10 and all('e' in v for v in line[3:])       # quant.py:129-130 format
    assert np.allclose(df['cdr'].values, (X > 0).mean(0))


def test_gathered_vs_in_place_cost_model():
    """Which form an extension round takes (engine.gathered_round_is_cheaper): --batchSize 500000 batches are
    100 events at 5k cells (whole 8-event blocks: in place, counts shared by the models), 5 events at 100k
    cells and 1 event at 1M cells (finer than a 32-byte sector: gathered), whatever fraction is still active."""
    from brie_b200.engine import gathered_round_is_cheaper

    def cols(Ng, M, group, p, seed=0):
        act = np.random.default_rng(seed).random((M, -(-Ng // group))) < p
        g = np.arange(Ng) // group
        return [np.flatnonzero(act[m, g]) for m in range(M)]

    for p in (0.6, 0.3, 0.1, 0.03):
        assert not gathered_round_is_cheaper(cols(5000, 2, 100, p), 5000, 5000, 3, 500)          # C2
        assert gathered_round_is_cheaper(cols(2500, 4, 5, p), 2500, 100000, 3, 500)              # C3 share
        assert gathered_round_is_cheaper(cols(1250, 2, 1, p), 1250, 1000000, 3, 500)             # C5 share
    # tiny problems: the fixed set-up cost of a gathered round dominates
    assert not gathered_round_is_cheaper(cols(64, 1, 1, 0.3), 64, 50, 3, 500)
    # nothing active in one model, a few batches in the other
    c = cols(2500, 2, 5, 0.1)
    c[0] = c[0][:0]
    assert gathered_round_is_cheaper(c, 2500, 100000, 3, 500)


def test_npz_container_references_memmapped_layers(tmp_path):
    """brie-quant --outDir: the dense output layers are .npy memory maps; the output container stores their
    paths instead of embedding 80 GB arrays, and reading it maps them again."""
    from brie_b200.utils.anndata_lite import AnnDataLite
    rng = np.random.default_rng(0)
    X = rng.poisson(1.0, (6, 9)).astype(np.float32)
    ad = AnnDataLite(X=X, layers={'isoform1': X.copy()})
    p = str(tmp_path / "Psi.npy")
    mm = np.lib.format.open_memmap(p, mode='w+', dtype=np.float32, shape=X.shape)
    mm[:] = rng.uniform(size=X.shape)
    mm.flush()
    ad.layers['Psi'] = np.load(p, mmap_mode='r+')
    out = str(tmp_path / "out.npz")
    ad.write_npz(out)
    assert os.path.getsize(out) < 4096                                   # the map is referenced, not embedded
    z = np.load(out, allow_pickle=True)
    assert 'layers/Psi@memmap' in z.files and 'layers/Psi' not in z.files
    back = AnnDataLite.read_npz(out)
    assert isinstance(back.layers['Psi'], np.memmap)
    assert np.array_equal(np.asarray(back.layers['Psi']), np.asarray(mm))
    assert np.array_equal(back.layers['isoform1'], X)
    # sparse matrices stay sparse in the container (a 1M x 20k count matrix is 80 GB dense)
    from scipy.sparse import csc_matrix, issparse
    ads = AnnDataLite(X=csc_matrix(X), layers={'isoform1': csc_matrix(X), 'dense': X.copy()})
    outs = str(tmp_path / "sparse.npz")
    ads.write_npz(outs)
    backs = AnnDataLite.read_npz(outs)
    assert issparse(backs.X) and issparse(backs.layers['isoform1']) and not issparse(backs.layers['dense'])
    assert np.array_equal(backs.X.toarray(), X) and np.array_equal(backs.layers['isoform1'].toarray(), X)


def test_host_pseudo_count_side_effect_semantics():
    """model_wrap.py:113-117 mutates the caller's dense arrays; read-only arrays raise (numpy's own error in the
    reference) and are never written through another view; fitBRIE's batch slices are left alone."""
    from brie_b200.models.model_wrap import _host_pseudo_count_inplace
    a = np.array([[0, 2, 0], [1, 0, 0]], np.float32)
    b = np.array([[0, 0, 0], [3, 0, 1]], np.float32)
    _host_pseudo_count_inplace([a, b, None], 0.01)
    assert np.allclose(a, [[0, 2.01, 0], [1.01, 0, 0.01]]) and np.allclose(b, [[0, 0.01, 0], [3.01, 0, 1.01]])
    ro = a.copy()
    ro.flags.writeable = False
    keep = ro.copy()
    with pytest.raises(ValueError, match="read-only"):
        _host_pseudo_count_inplace([ro, b, None], 0.01)
    assert np.array_equal(ro, keep)


def test_cli_has_outdir_and_resume_flags():
    import subprocess
    out = subprocess.run([sys.executable, "-m", "brie_b200.bin.quant", "--help"], capture_output=True, text=True,
                         cwd=ROOT, timeout=120)
    assert out.returncode == 0
    for flag in ("--outDir", "--resume", "--LRTindex", "--testBase", "--interceptMode", "--MCsize", "--batchSize"):
        assert flag in out.stdout, flag


def test_engine_plan_splits_long_lrt_lists():
    """fit_BRIE_matrix batches the base model and the LRT refits into FitEngines of at most 32 models; a one-vs-rest
    LRT over more covariates runs the remaining refits in further engines (the reference loops over any number of
    tests, model_wrap.py:156-187); a cell-mode base model sits alone (refits use the per-event layout, :174-178)."""
    from brie_b200.models.model_wrap import _engine_plan
    tests = [[k for k in range(40) if k != i] for i in range(40)]
    plan = _engine_plan(list(range(40)), tests, False, 'gene')
    assert [len(p[0]) for p in plan] == [32, 9]
    assert plan[0][1] == list(range(32)) and plan[1][1] == list(range(32, 41))
    assert plan[0][0][0] == list(range(40)) and plan[0][0][1] == tests[0] and plan[1][0][0] == tests[31]
    assert sorted(i for p in plan for i in p[1]) == list(range(41))              # every model exactly once
    plan = _engine_plan([0], [[0, 1], [0, 2]], True, 'cell')
    assert [(p[1], p[2]) for p in plan] == [([0], 'cell'), ([1, 2], 'gene')]
    plan = _engine_plan([0, 1], [], True, 'cell')
    assert plan == [([[0, 1]], [0], 'cell')]
    plan = _engine_plan([], [[0]], False, 'None', max_models=2)
    assert [(p[0], p[1]) for p in plan] == [([[], [0]], [0, 1])]
    plan = _engine_plan([], [[0], [1], [2]], False, 'gene', max_models=2)
    assert [p[1] for p in plan] == [[0, 1], [2, 3]]


def test_product_path_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under brie_b200/ may import, load or execute it (a product path
    routed through the oracle or any CPU fallback would void every parity claim)."""
    import glob
    bad = []
    for path in glob.glob(os.path.join(ROOT, "brie_b200", "**", "*"), recursive=True):
        if not path.endswith((".py", ".cu", ".cuh", ".h")):
            continue
        txt = open(path, errors="ignore").read()
        if re.search(r"^\s*(from|import)\s+oracle\b|oracle[./]brie2|oracle/_ref|philox_np", txt, flags=re.M):
            bad.append(path)
    assert not bad, bad
    # and the fit refuses to run without a CUDA device instead of falling back
    import torch
    if not torch.cuda.is_available():
        from brie_b200.models import fit_BRIE_matrix
        with pytest.raises(RuntimeError, match="no CUDA device"):
            fit_BRIE_matrix([np.ones((3, 4), np.float32), np.ones((3, 4), np.float32)])


def test_bench_reference_arm_runs_and_mirrors_the_config():
    """`bench.py --impl reference` (the restated reference on the host cores; only rank 0 works) prints one JSON line
    with the contract's keys and the same `config` dict the GPU arm prints."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 2
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.config_dict(2) and line["unit"] == bench.UNIT and line["metric"] == bench.METRIC
    other = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                           capture_output=True, text=True, timeout=60, cwd=ROOT, env=dict(os.environ, RANK="1"))
    assert other.returncode == 0 and other.stdout.strip() == ""            # ranks other than 0 exit without work


def test_bench_rejects_zero_steps_and_a_dump_of_the_reference_arm():
    """--steps is the number of timed steps, so 0 is an error rather than a silent 1; --dump-outputs writes the GPU
    arm's outputs and is refused with --impl reference.  Both are refused before any work."""
    for extra, msg in ((["--steps", "0"], "--steps must be at least 1"),
                       (["--impl", "reference", "--dump-outputs", "unused"], "--dump-outputs applies to the GPU arm")):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "" and msg in out.stderr, (extra, out.stderr[-2000:])
