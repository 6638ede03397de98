"""Two steps per pass: run_steps(K) of a fit with per-event parameters only (gene mode, Kg = 0, Kc <= 4) takes its
steps in pairs over one read and write of the state, with a sums-only pre-pass and the next pair's parameters formed
from statistics of the state.  It must end where K single steps end: same Adam step and RNG word, the same state,
parameters and loss trace up to float32 summation order, and no further from the float64 oracle than single steps."""
import numpy as np
import pytest

from oracle import philox_np as px
from oracle.brie2_oracle import OracleBRIE2, _Adam, add_pseudo_count

from util import device_eps_provider, make_problem

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _engines(data, effLen, Xc, n=2, **kw):
    from brie_b200.engine import FitEngine
    out = []
    for _ in range(n):
        e = FitEngine(data, effLen=effLen, Xc=Xc, Xg=None, **kw)
        e.init_params()
        out.append(e)
    return out


def _state(e):
    Ng = e.Ng
    return {"Z_loc": e.Z_loc[:, :, :Ng], "Z_std_log": e.Z_std_log[:, :, :Ng], "Wc": e.Wc[:, :, :Ng],
            "intercept": e.intercept[:, :Ng], "sigma_log": e.sigma_log[:, :Ng], "trace": e.loss_trace[:, :, :Ng]}


def _max_diff(a, b):
    return (a - b).abs().max().item() if a.numel() else 0.0


CASES = [
    # Nc, Ng, Kc, masks, count_format, sigma_log0, frozen
    (157, 203, 3, [[0, 1, 2], [0, 1]], None, None, False),      # LRT full + null, packed codes, odd cells
    (157, 203, 3, [[0, 1, 2], [0, 1]], 'f32', None, False),     # float32 count tiles
    (96, 130, 1, [[0], []], None, 2.5, False),                  # tau far from 0
    (96, 130, 2, [[0, 1]], None, -2.0, True),                   # frozen events
    (150, 77, 0, [[]], 'f32', None, True),                      # no covariates
]


@pytest.mark.parametrize("K", [2, 3, 6, 7])
@pytest.mark.parametrize("trace", [False, True])
@pytest.mark.parametrize("Nc,Ng,Kc,masks,count_format,sigma_log0,frozen", CASES)
def test_run_steps_equals_single_steps(K, trace, Nc, Ng, Kc, masks, count_format, sigma_log0, frozen):
    data, effLen, Xc, _ = make_problem(Nc, Ng, Kc, 0, True, 3)
    add_pseudo_count(data, np.float32(0.01))
    a, b, init = _engines(data, effLen, Xc, n=3, masks=masks, MC_size=3, seed=5, trace_cap=16,
                          count_format=count_format)
    for e in (a, b, init):
        if sigma_log0 is not None:
            e.sigma_log[:, :Ng] = sigma_log0
        if frozen:
            e.active[:, 1:Ng:3] = 0
        e.begin_stage(0.05)
    a.run_steps(K, 0 if trace else -1)
    for i in range(K):
        b.run_steps(1, i if trace else -1)
    torch.cuda.synchronize()
    assert a.step_counters() == b.step_counters()
    sa, sb = _state(a), _state(b)
    for name in ("Z_loc", "Z_std_log", "Wc", "intercept", "sigma_log"):
        d = _max_diff(sa[name], sb[name])
        print("K=%d %s max |pairs - singles| %.2e" % (K, name, d))
        assert d < 2e-3, name
    if frozen:   # frozen events do not move
        for name in ("Z_loc", "intercept", "sigma_log"):
            assert torch.equal(_state(init)[name][..., 1:Ng:3], sa[name][..., 1:Ng:3]), name
    if trace:
        ta, tb = sa["trace"][:, :K].double(), sb["trace"][:, :K].double()
        rel = ((ta - tb).abs() / tb.abs().clamp_min(1.0)).max().item()
        print("K=%d loss trace max relative difference %.2e" % (K, rel))
        assert rel < 1e-4


@pytest.mark.parametrize("Kc,sigma_log0", [(3, None), (1, 2.5), (4, -1.5)])
@pytest.mark.parametrize("K", [8, 9])
def test_pairs_no_further_from_oracle_than_single_steps(Kc, sigma_log0, K):
    """The look-ahead update forms its sums from statistics, not from the elements: over K steps its parameters and
    state must stay as close to the float64 oracle (same init, same device noise) as single steps do."""
    Nc, Ng, S, seed, lr = 111, 97, 3, 7, 0.05
    data, effLen, Xc, _ = make_problem(Nc, Ng, Kc, 0, True, 3, seed=4)
    add_pseudo_count(data, np.float32(0.01))
    a, b = _engines(data, effLen, Xc, MC_size=S, seed=seed, trace_cap=16)
    om = OracleBRIE2(Nc, Ng, Kc, 0, effLen, None, 'gene', None, dtype=np.float64, seed=seed)
    om.Xc = Xc.astype(np.float64)
    for e in (a, b):
        if sigma_log0 is not None:
            e.sigma_log[:, :Ng] = sigma_log0
        e.begin_stage(lr)
    if sigma_log0 is not None:
        om.p['sigma_log'][...] = sigma_log0
    a.run_steps(K, 0)
    for i in range(K):
        b.run_steps(1, i)
    names = om.trainable()
    adam = _Adam(lr, {k: om.p[k] for k in names}, np.float64)
    epsf = device_eps_provider(seed, 0, Nc, Ng)
    ref_losses = []
    for step in range(K):
        loss, _, grads = om.loss_and_grads(data, epsf(px.PHASE_TRAIN, step, S))
        ref_losses.append(loss)
        adam.apply(om.p, {k: grads[k] for k in names})
        np.clip(om.p['Z_loc'], -9, 9, out=om.p['Z_loc'])
        np.clip(om.p['intercept'], -9, 9, out=om.p['intercept'])
    torch.cuda.synchronize()
    ref = {"Z_loc": om.p['Z_loc'], "Z_std_log": om.p['Z_std_log'], "Wc": om.p['Wc_loc'].reshape(Kc, Ng),
           "intercept": om.p['intercept'].reshape(-1), "sigma_log": om.p['sigma_log'].reshape(-1)}
    for name, r in ref.items():
        if r.size == 0:
            continue
        dev = {e: _state(e)[name][0].cpu().numpy().astype(np.float64) for e in (a, b)}
        if name == "Wc":
            dev = {e: v[:Kc] for e, v in dev.items()}
        err_pair, err_single = np.abs(dev[a] - r).max(), np.abs(dev[b] - r).max()
        print("K=%d %s max |x - oracle|: pairs %.2e, single steps %.2e" % (K, name, err_pair, err_single))
        assert err_pair <= 1.5 * err_single + 1e-6, name
    tr = _state(a)["trace"][0, :K].double().sum(dim=1).cpu().numpy()
    ts = _state(b)["trace"][0, :K].double().sum(dim=1).cpu().numpy()
    ref_losses = np.array(ref_losses)
    assert np.abs(tr - ref_losses).max() <= max(1.5 * np.abs(ts - ref_losses).max(), 1e-6 * np.abs(ref_losses).max())


@pytest.mark.parametrize("gathered", [False, True])
def test_pairs_on_active_blocks_and_gathered_subfits(gathered):
    """Extension rounds in pairs: over the 8-event blocks that still hold an active event (column compaction) or on
    a gathered sub-fit, against single steps over the whole shard with the same events frozen."""
    Nc, Ng, group, K = 130, 300, 3, 6
    data, effLen, Xc, _ = make_problem(Nc, Ng, 2, 0, True, 3, seed=8)
    add_pseudo_count(data, np.float32(0.01))
    a, b = _engines(data, effLen, Xc, masks=[[0, 1], [1]], model_ids=[0, 1], MC_size=3, seed=12, trace_cap=8,
                    group_size=group)
    for e in (a, b):
        e.begin_stage(0.02)
        e.run_steps(4)
    act = np.random.default_rng(3).random((2, a.n_groups)) < 0.2
    act[1, 0] = True
    if gathered:
        assert a.run_steps_gathered(act, K, force=True)
    else:
        a.set_active_groups(act)
        assert a._blk_ids is not None
        a.run_steps(K, 0)
    b.set_active_groups(act)
    for i in range(K):
        b.run_steps(1, i)
    torch.cuda.synchronize()
    sa, sb = _state(a), _state(b)
    for name in ("Z_loc", "Z_std_log", "Wc", "intercept", "sigma_log"):
        d = _max_diff(sa[name], sb[name])
        print("%s max |pairs - singles| %.2e" % (name, d))
        assert d < 2e-3, name
