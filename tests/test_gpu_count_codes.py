"""GPU tests of the packed count codes of the fused step kernel (brie_encode_counts, brie_fit_set_count_codes): the
codes decode to the float32 tiles, their non-zero test is the kernel's read test, and a fit that steps on codes is
bit-identical to one that steps on the float32 tiles -- every instantiation family, in-place and gathered extension
rounds, and a whole fit_BRIE_matrix with LRT refits and permutations.  A layer with too many distinct values falls
back to the float32 tiles."""
import numpy as np
import pytest

from oracle.brie2_oracle import add_pseudo_count
from util import make_lrt_problem, make_problem

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _state(eng):
    torch.cuda.synchronize()
    return dict(Z_loc=eng.Z_loc.clone(), Z_std_log=eng.Z_std_log.clone(), adam_Z=eng.adam_Z.clone(),
                Wc=eng.Wc.clone(), intercept=eng.intercept.clone(), sigma_log=eng.sigma_log.clone(),
                Wg=eng.Wg.clone(), adam_small=eng.adam_small.clone(), loss_trace=eng.loss_trace.clone())


def _assert_same(a, b):
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_codes_decode_to_the_tiles_and_mark_the_elements_with_reads():
    from brie_b200 import _lib
    from brie_b200.engine import encode_counts
    lib = _lib.load()
    rng = np.random.default_rng(0)
    Nc, ld = 257, 384
    tiles = [rng.poisson(0.4, (Nc, ld)).astype(np.float32) for _ in range(3)]
    tiles[2][rng.random((Nc, ld)) < 0.9] = 0
    add_pseudo_count(tiles, np.float32(0.01))        # values k + 0.01 next to plain integers
    tiles[0][3, :7] = -0.0
    tiles[2][5, 9] = 1e-40                           # a denormal is a value like any other
    dev = [torch.from_numpy(t).cuda() for t in tiles]
    codes, dct = encode_counts(lib, dev, torch.device("cuda"))
    w = codes.cpu().numpy().view(np.uint32)
    d = dct.cpu().numpy()
    assert (w >> 24 == 0).all() and (d[:, 0] == 0).all() and not np.signbit(d[:, 0]).any()
    for l in range(3):
        dec = d[l][(w >> (8 * l)) & 255]
        nz = tiles[l] != 0
        assert np.array_equal(dec.view(np.uint32)[nz], tiles[l].view(np.uint32)[nz]), l   # bit for bit
        assert (dec[~nz] == 0).all()                                                     # +0 and -0: code 0
        vals = np.unique(tiles[l][nz])
        assert np.array_equal(d[l, 1:1 + len(vals)], vals) and (d[l, 1 + len(vals):] == 0).all()
    reads = (tiles[0] + tiles[1] + tiles[2]) > np.float32(0)
    assert np.array_equal(w != 0, reads)
    # two layers: the third byte stays 0
    codes2, _ = encode_counts(lib, dev[:2], torch.device("cuda"))
    assert (codes2.cpu().numpy().view(np.uint32) >> 16 == 0).all()


def test_encoder_refuses_what_it_cannot_code():
    from brie_b200 import _lib
    from brie_b200.engine import encode_counts
    lib = _lib.load()
    base = np.zeros((64, 128), np.float32)
    base[:10, :30] = np.arange(300, dtype=np.float32).reshape(10, 30) + 1        # 300 distinct values
    z = torch.zeros((64, 128), device="cuda")
    assert encode_counts(lib, [z, torch.from_numpy(base).cuda()], torch.device("cuda")) is None
    base[:] = 0
    base[0, 0] = np.nan
    assert encode_counts(lib, [torch.from_numpy(base).cuda(), z], torch.device("cuda")) is None
    base[0, 0] = -1.0
    assert encode_counts(lib, [torch.from_numpy(base).cuda(), z], torch.device("cuda")) is None
    base[0, 0] = 7.0
    assert encode_counts(lib, [torch.from_numpy(base).cuda(), z], torch.device("cuda")) is not None


# name -> (Nc, Ng, Kc, Kg, effLen, layers, intercept mode, masks)
CONFIGS = {
    "C2": (300, 500, 1, 0, True, 3, 'gene', [[0], []]),
    "C3": (260, 400, 3, 0, True, 3, 'gene', [[0, 1, 2], [1, 2], [0, 2], [0, 1]]),
    "C4": (300, 333, 0, 8, False, 2, 'cell', [[]]),
    "Kc16": (200, 300, 16, 0, True, 3, 'gene', [list(range(16))]),          # 2 events per lane, 2 rows per iteration
    "Kc8Kg4": (150, 260, 8, 4, True, 3, 'gene', [list(range(8))]),
    "wide": (180, 300, 20, 0, True, 3, 'gene', [list(range(20)), list(range(19))]),   # EXT: GEMMs around the kernel
}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_code8_steps_are_bit_identical_to_f32(name):
    from brie_b200.engine import FitEngine
    Nc, Ng, Kc, Kg, eff, nl, mode, masks = CONFIGS[name]
    data, effLen, Xc, Xg = make_problem(Nc, Ng, Kc, Kg, eff, nl, seed=5)
    add_pseudo_count(data, np.float32(0.01))
    out = {}
    for fmt in (None, 'f32'):
        eng = FitEngine(data, effLen=effLen if eff else None, Xc=Xc, Xg=Xg if Kg else None, masks=masks,
                        intercept_mode=mode, MC_size=3, seed=9, trace_cap=40, count_format=fmt)
        assert eng.count_format == ('code8' if fmt is None else 'f32')
        eng.init_params()
        eng.begin_stage(0.01)
        eng.run_steps(25)                 # without the loss trace
        eng.begin_stage(0.02)
        eng.run_steps(35, 0)              # with it
        out[fmt] = _state(eng)
    _assert_same(out[None], out['f32'])
    assert float(out[None]['loss_trace'][:, 34, :Ng].abs().sum()) > 0


def test_layer_with_300_values_falls_back_to_f32():
    from brie_b200.engine import FitEngine
    data, effLen, Xc, _ = make_problem(120, 200, 1, 0, True, 3, seed=6)
    add_pseudo_count(data, np.float32(0.01))
    data[2][data[2] > 0] = np.random.default_rng(1).integers(1, 301, int((data[2] > 0).sum())).astype(np.float32)
    data[2][:30, :10] = np.arange(300, dtype=np.float32).reshape(30, 10) + 1     # 300 distinct values for sure
    out = []
    for fmt in (None, 'f32'):
        eng = FitEngine(data, effLen=effLen, Xc=Xc, masks=[[0], []], MC_size=3, seed=2, trace_cap=20, count_format=fmt)
        assert eng.count_format == 'f32' and eng.count_codes is None
        eng.init_params(); eng.begin_stage(0.01); eng.run_steps(20, 0)
        out.append(_state(eng))
    _assert_same(*out)


@pytest.mark.parametrize("gathered", [False, True])
def test_extension_rounds_bit_identical(gathered, monkeypatch):
    """In-place rounds over the active 8-event blocks and gathered sub-fits (which move code words, not layers)."""
    from brie_b200.engine import FitEngine
    Nc, Ng, group = 300, 700, 3
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=8)
    add_pseudo_count(data, np.float32(0.01))
    out = {}
    for fmt in (None, 'f32'):
        eng = FitEngine(data, effLen=effLen, Xc=Xc, masks=[[0, 1], [1]], model_ids=[0, 1], MC_size=3, seed=12,
                        trace_cap=8, group_size=group, count_format=fmt)
        eng.init_params(); eng.begin_stage(0.01); eng.run_steps(4)
        for frac in (0.3, 0.05):
            act = np.random.default_rng(int(frac * 100)).random((2, eng.n_groups)) < frac
            act[1, 0] = True
            if gathered:
                assert eng.run_steps_gathered(act, 3, force=True)
            else:
                eng.set_active_groups(act)
                eng.run_steps(3, 0)
        eng.set_active_groups(np.ones((2, eng.n_groups), bool))
        eng.run_steps(2, 0)
        out[fmt] = _state(eng)
        assert eng.gather_rounds == (2 if gathered else 0)
    _assert_same(out[None], out['f32'])


def test_fit_matrix_with_lrt_and_permutations_bit_identical(monkeypatch):
    from brie_b200 import engine
    from brie_b200.models import fit_BRIE_matrix
    data, effLen, Xc, _ = make_lrt_problem(Nc=140, Ng=40, seed=3)
    Xc = np.concatenate([Xc, np.random.default_rng(2).standard_normal((140, 1)).astype(np.float32)], axis=1)
    add_pseudo_count(data, np.float32(0.01))
    kw = dict(Xc=Xc, effLen=effLen, LRT_index=[0, 1], intercept_mode='gene', min_iter=240, max_iter=740, MC_size=2,
              n_eval=10, seed=3, n_perm=2)
    calls = []
    real = engine.encode_counts

    def counted(*a):
        calls.append(1)
        return real(*a)

    monkeypatch.setattr(engine, "encode_counts", counted)
    r_code = fit_BRIE_matrix([x.copy() for x in data], **kw)
    assert len(calls) == 1                           # one code tile for every engine of the chunk
    monkeypatch.setattr(engine, "encode_counts", lambda *a: None)
    r_f32 = fit_BRIE_matrix([x.copy() for x in data], **kw)
    for k in ('Psi', 'Psi95CI', 'Z_std', 'loss_gene', 'ELBO_gain', 'pval', 'fdr', 'n_iter', 'cell_coeff',
              'ELBO_gain_perm', 'pval_perm'):
        assert np.array_equal(np.asarray(getattr(r_code, k)), np.asarray(getattr(r_f32, k))), k
