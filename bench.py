#!/usr/bin/env python
"""bench.py -- BRIE2 VI-fit hot path on B200.

Metric (BASELINE.json): cell x event x MC-sample ELBO fwd+bwd per second (+ brie-quant fit+LRT wall time).

Headline workload (every N): BASELINE config C3 "10x-scale DAS" -- 100 000 cells x 10 000 events, 3 cell
covariates + batched LRT (full model + 3 refits, M = 4), 3 count layers with effective lengths, MC_size 3,
--interceptMode gene -- the largest configuration that fits one B200 (108 GB resident) and the one BASELINE
lists for 1/2/4/8 GPUs.  STRONG scaling: the 10 000 events are sharded over the N ranks in contiguous ranges
aligned to the reference's event batches (model_wrap.py:241-260); per-event parameters are independent, so
this leg has no data-path collective.  One "step" = one fused ELBO forward+backward+Adam step of all four
models over the whole matrix.

  value    : device-resident throughput, CUDA events around K steps, max over ranks
  e2e      : the same metric through the public API `brie_b200.models.fitBRIE` on the same workload with HOST
             inputs (scipy CSC layers, what brie-count hands over): H2D ingest, the full default brie-quant
             schedule (--minIter 5000 --maxIter 20000 --MCsize 3 --batchSize 500000 convergence groups),
             500-sample loss_gene, LRT, p / FDR, D2H of Psi / Psi_95CI / Z_std / Z_loc into the output maps.
             `fit_lrt_wall_s` is BASELINE's second metric for this configuration.
  roofline : fused step kernel, algorithmic bytes (12 + 48 M per cell-event-step) / CUDA-event kernel time,
             against MEASURED_PEAKS.json hbm_gbs
  shapes   : the other named shapes, device-resident, K steps each: C2 (5k x 5k, the round-1 headline, strong-
             sharded), C5 (1M cells, a per-GPU event slab)
  c4       : BASELINE config C4 (200k cells x 20k genes, spliced/unspliced, Kg = 8 gene features,
             interceptMode cell), events strong-sharded: the ONE exchange step of the path -- the per-step NCCL
             all-reduce of d/dWg, d/db, d/dlog sigma per cell (8 MB), issued by the library in stream order -- with
             step time with / without the collective, the all-reduce alone, and a sharded-vs-unsharded parity check
  cpu_baseline : the restated reference (oracle/brie2_torch_eager.py, op-for-op PyTorch-CPU eager, not
             TensorFlow) on one reference batch of the headline workload on the box's host cores.

`--impl reference` times that restated reference alone (the real reference needs TensorFlow, which cannot
be installed here), on the same config / metric / unit.

`--dump-outputs DIR` writes the headline fit's state after its last timed step to DIR/<name>.npy (float32, about
42 MB): what a caller of the timed steps receives, for comparing two builds output for output.  The inputs are drawn
from fixed seeds, so two runs with the same arguments start from identical data.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S = 3
METRIC = "cell x event x MC-sample ELBO fwd+bwd per second"
UNIT = "cell*event*sample/s"
SHAPES = {
    "C2": dict(cells=5000, events=5000, design='binary1', layers=3, eff=True, Kg=0, mode='gene',
               masks=[[0], []], name="C2 Smart-seq2-scale DAS: 5000 cells x 5000 events, Kc=1, LRT full+null (M=2)"),
    "C3": dict(cells=100000, events=10000, design='mixed3', layers=3, eff=True, Kg=0, mode='gene',
               masks=[[0, 1, 2], [1, 2], [0, 2], [0, 1]],
               name="C3 10x-scale DAS: 100000 cells x 10000 events, 3 count layers + effLen, Kc=3, LRT full + 3 "
                    "refits batched (M=4), MC_size=3, interceptMode gene"),
    "C4": dict(cells=200000, events=20000, design='none', layers=2, eff=False, Kg=8, mode='cell', masks=[[]],
               name="C4 DMG: 200000 cells x 20000 genes, spliced/unspliced, Kg=8 gene features, interceptMode cell (M=1)"),
    "C5": dict(cells=1000000, events=20000, design='pseudotime', layers=3, eff=True, Kg=0, mode='gene',
               masks=[[0], []], name="C5 atlas DAS: 1M cells x 20000 events, pseudotime + LRT (M=2)"),
}
HEAD = "C3"


def config_dict(world):
    c = SHAPES[HEAD]
    return {"workload": c["name"], "cells": c["cells"], "events": c["events"], "models": len(c["masks"]),
            "mc_size": S, "scaling": "strong: events sharded over %d rank(s), aligned to --batchSize 500000 groups" % world,
            "l2": "inputs larger than L2: %.0f GB moved per step per GPU >> 126 MB L2" % (
                c["cells"] * c["events"] / world * (12 + 48 * len(c["masks"])) / 1e9),
            "parallelism": "events sharded x%d, no data-path collective on this leg (the C4 leg has the Wg all-reduce)" % world}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, period_ms=100):
        self.lines, self.proc = [], None
        self.index, self.period = index, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", str(self.period)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(self.period / 1000.0 * 1.5)
        self.proc.terminate()
        rows = [l for (t, l) in self.lines if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.15)]
        if len(rows) < 3:
            rows = [l for (_, l) in self.lines]
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[2])); smax.append(float(f[3])); power.append(float(f[4]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[5:9]):
                if v == "Active":
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_run(n_steps, warmup, threads, seed=1):
    """Restated reference (op-for-op torch-CPU eager + autograd + TF-form Adam) on ONE reference batch of the
    headline workload: 100 000 cells x 5 events = --batchSize 500000 (model_wrap.py:242), full model (Kc = 3)."""
    import torch
    from oracle.brie2_torch_eager import EagerBRIE2
    from oracle.brie2_oracle import OracleInit, add_pseudo_count
    from brie_b200.utils.synth import simulate_counts
    c = SHAPES[HEAD]
    Nc = c["cells"]
    n_events = int(np.ceil(500000 / Nc))
    Kc = len(c["masks"][0])
    torch.set_num_threads(threads)
    d = simulate_counts(Nc, n_events, design=c["design"], seed=seed)
    data = [x.copy() for x in d['layers']]
    add_pseudo_count(data, np.float32(0.01))
    init = OracleInit(Nc, n_events, Kc, 0, (1, n_events), (1, n_events), None, None, seed=seed)
    m = EagerBRIE2(Nc, n_events, Kc, 0, d['effLen'], None, 'gene', None, init, torch.float32)
    m.set_design(d['Xc'], None)
    cl = [torch.from_numpy(x) for x in data]
    st = {'t': 0, 'm': {}, 'v': {}}
    gen = torch.Generator().manual_seed(seed)
    times = []
    for i in range(warmup + n_steps):
        t0 = time.perf_counter()
        eps = torch.randn((S, Nc, n_events), generator=gen)      # tfd.Normal.sample cost is part of the step
        m.train_step(cl, eps, st, 0.01)
        times.append(time.perf_counter() - t0)
    dt = float(np.sum(times[warmup:]))
    sample = ("%d cells x %d events (one --batchSize 500000 reference batch of the workload, ONE of its %d models), "
              "%d steps, S=%d" % (Nc, n_events, len(c["masks"]), n_steps, S))
    return Nc * n_events * S * n_steps / dt, dt / n_steps * 1e3, sample


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    K, W = args.steps, max(args.warmup, 0)
    val, ms, sample = cpu_reference_run(K, W, threads)
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
           "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config_dict(args.gpus),
           "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                            "note": "restated reference (PyTorch-CPU eager, not TensorFlow: TF/TFP are not installable "
                                    "here); runs on rank 0's host cores whatever --gpus says"},
           "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# ----------------------------------------------------------------------------------------------- GPU arm
class Ctx:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = "cuda:%d" % self.local
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.dist is None:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def shard_of(ctx, name, events=None):
    """This rank's contiguous event range of a named shape: aligned to the reference's event batches."""
    from brie_b200.sharding import event_shards
    c = SHAPES[name]
    Ng = events if events is not None else c["events"]
    group = max(1, int(np.ceil(500000 / c["cells"])))
    return event_shards(Ng, ctx.world, group)[ctx.rank], group, Ng


def build_engine(ctx, name, lo, hi, Ng_total, group, seed=3, trace_cap=8, dist_group=None):
    """Device-resident engine over events [lo, hi) of a named shape, counts drawn on the device."""
    from brie_b200.engine import FitEngine
    from brie_b200.utils.synth import simulate_counts_device
    c = SHAPES[name]
    n = hi - lo
    sim = simulate_counts_device(c["cells"], n, design=c["design"], seed=seed + 17 * ctx.rank, with_efflen=c["eff"],
                                 n_layers=c["layers"], event_offset=lo, device=ctx.dev,
                                 Xc=__import__("brie_b200.utils.synth", fromlist=["make_design"]).make_design(
                                     c["cells"], c["design"], np.random.default_rng(0)))
    nz = float(((sim['layers'][0] + sim['layers'][1] + (sim['layers'][2] if c["layers"] > 2 else 0)) > 0).float().mean())
    Xg = np.random.default_rng(1).standard_normal((Ng_total, c["Kg"])).astype(np.float32)[lo:hi] if c["Kg"] else None
    eng = FitEngine(sim['layers'], effLen=sim['effLen'], Xc=sim['Xc'], Xg=Xg, masks=c["masks"],
                    intercept_mode=c["mode"], MC_size=S, seed=7, n_events=n, event_offset=lo, n_events_total=Ng_total,
                    trace_cap=trace_cap, group_size=group, device=ctx.dev, dist_group=dist_group)
    eng.init_params()
    eng.begin_stage(0.01)
    return eng, nz


def time_steps(ctx, eng, K, W, sampler=None):
    """W warm-up steps, then exactly K steps between barriers; CUDA events, max over ranks."""
    torch = ctx.torch
    eng.run_steps(W)
    torch.cuda.synchronize()
    eng.kernel_timing(K)
    ctx.barrier()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    eng.run_steps(K)
    e1.record()
    torch.cuda.synchronize()
    ctx.barrier()
    t1 = time.time()
    ms_local = e0.elapsed_time(e1)
    kms, kn = eng.kernel_time_ms()
    return dict(ms=ctx.max_over_ranks(ms_local), ms_local=ms_local, kernel_ms=kms / max(kn, 1), launches=eng.launch_count - l0,
                t0=t0, t1=t1)


def dump_outputs(ctx, eng, out_dir, n_cells=128, seed=0):
    """The engine state after its last step, gathered over the ranks' event shards, as float32 .npy files in
    out_dir: the per-event parameters (Wc, intercept, sigma_log: models x rows x events) whole, and the
    variational parameters (Z_loc, Z_std_log: models x cells x events) for a fixed, seeded sample of n_cells
    cells -- all of them would be 16 GB at the headline size."""
    from brie_b200.sharding import gather_event_axis
    torch = ctx.torch
    Ng = eng.Ng
    cells = np.sort(np.random.default_rng(seed).choice(eng.Nc, min(n_cells, eng.Nc), replace=False))
    rows = torch.from_numpy(cells).to(eng.device)
    arrays = {"Z_loc": eng.Z_loc.index_select(1, rows)[:, :, :Ng],
              "Z_std_log": eng.Z_std_log.index_select(1, rows)[:, :, :Ng],
              "Wc": eng.Wc[:, :max(len(mk) for mk in eng.masks), :Ng],
              "intercept": eng.intercept[:, :Ng], "sigma_log": eng.sigma_log[:, :Ng]}
    arrays = {k: gather_event_axis(v.cpu().numpy(), v.dim() - 1) for k, v in arrays.items()}
    if ctx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for k, v in arrays.items():
            np.save(os.path.join(out_dir, k + ".npy"), v)


def shape_leg(ctx, name, K, W, events=None, note=None):
    c = SHAPES[name]
    (lo, hi), group, Ng = shard_of(ctx, name, events)
    eng, nz = build_engine(ctx, name, lo, hi, Ng, group)
    r = time_steps(ctx, eng, K, W)
    M = len(c["masks"])
    peak, _ = hbm_peak()
    alg = c["cells"] * (hi - lo) * (4 * c["layers"] + 48 * M)
    out = {"workload": c["name"], "events_total": Ng, "events_this_rank": hi - lo, "steps": K,
           "ms_per_step": r["ms"] / K, "value": c["cells"] * Ng * S * M * K / (r["ms"] * 1e-3), "unit": UNIT,
           "kernel_ms": r["kernel_ms"], "frac_of_measured_hbm": alg / (r["kernel_ms"] * 1e-3) / 1e9 / peak,
           "nonzero_fraction": nz}
    if note:
        out["note"] = note
    del eng
    ctx.torch.cuda.empty_cache()
    return out


def c4_leg(ctx, K, W):
    """C4: the per-step all-reduce of the shared per-cell gradients."""
    torch = ctx.torch
    import ctypes as C
    from brie_b200 import _lib
    lib = _lib.load()
    c = SHAPES["C4"]
    (lo, hi), group, Ng = shard_of(ctx, "C4")
    eng, nz = build_engine(ctx, "C4", lo, hi, Ng, group, seed=40,
                           dist_group=ctx.dist.group.WORLD if ctx.dist is not None else None)
    with_c = time_steps(ctx, eng, K, W)
    M = len(c["masks"])
    peak, _ = hbm_peak()
    alg = c["cells"] * (hi - lo) * (4 * c["layers"] + 48 * M)
    out = {"workload": c["name"], "events_this_rank": hi - lo, "steps": K,
           "ms_per_step": with_c["ms"] / K, "value": c["cells"] * Ng * S * M * K / (with_c["ms"] * 1e-3), "unit": UNIT,
           "kernel_ms": with_c["kernel_ms"], "frac_of_measured_hbm": alg / (with_c["kernel_ms"] * 1e-3) / 1e9 / peak,
           "launches_per_step": with_c["launches"] / K, "nonzero_fraction": nz}
    n_G = M * c["cells"] * (c["Kg"] + 2)
    out["allreduce_bytes_per_step"] = n_G * 4
    if ctx.dist is not None and eng._comm is not None:
        out["collective"] = "ncclAllReduce(sum, f32) of (M, Nc, Kg+2) issued by libbrie_b200.so in stream order (NCCL %d)" % (
            lib.brie_comm_nccl_version())
        _lib.check(lib.brie_fit_set_comm(eng.h, None))          # same kernels, no exchange (results unused)
        without = time_steps(ctx, eng, K, W)
        _lib.check(lib.brie_fit_set_comm(eng.h, eng._comm.h))
        out["ms_per_step_without_collective"] = without["ms"] / K
        out["exposed_collective_ms_per_step"] = (with_c["ms"] - without["ms"]) / K
        out["exposed_collective_frac_of_step"] = (with_c["ms"] - without["ms"]) / with_c["ms"]
        G = torch.zeros(n_G, dtype=torch.float32, device=ctx.dev)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for _ in range(3):
            _lib.check(lib.brie_comm_allreduce_f32(eng._comm.h, G.data_ptr(), n_G, st))
        ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            _lib.check(lib.brie_comm_allreduce_f32(eng._comm.h, G.data_ptr(), n_G, st))
        e1.record()
        torch.cuda.synchronize()
        a_ms = ctx.max_over_ranks(e0.elapsed_time(e1)) / K
        out["allreduce_alone_ms"] = a_ms
        out["allreduce_alone_busbw_GBps"] = n_G * 4 * 2 * (ctx.world - 1) / ctx.world / (a_ms * 1e-3) / 1e9
    del eng
    torch.cuda.empty_cache()
    if ctx.dist is not None:
        out["sharded_vs_unsharded"] = sharded_parity(ctx)
    return out


def sharded_parity(ctx, steps=30):
    """A small C4-style fit (Kg = 8, cell mode) stepped (a) un-sharded on this GPU and (b) event-sharded over
    all ranks with the in-library all-reduce: shared parameters and this rank's Z columns must agree up to the
    float32 summation order of the per-cell gradient sums."""
    torch = ctx.torch
    from brie_b200.engine import FitEngine
    from brie_b200.sharding import event_shards
    from brie_b200.utils.synth import simulate_counts
    Nc, Ng, Kg = 3000, 1024, 8
    d = simulate_counts(Nc, Ng, design='none', seed=5, with_efflen=False, n_layers=2)
    data = d['layers']
    idx = data[0] + data[1] > 0
    for i in range(2):
        data[i][idx] += np.float32(0.01)
    Xg = np.random.default_rng(2).standard_normal((Ng, Kg)).astype(np.float32)
    lo, hi = event_shards(Ng, ctx.world, 1)[ctx.rank]
    kw = dict(effLen=None, masks=[[]], intercept_mode='cell', MC_size=S, seed=3, trace_cap=steps, device=ctx.dev)
    full = FitEngine(data, Xg=Xg, **kw)
    part = FitEngine([x[:, lo:hi] for x in data], Xg=Xg[lo:hi], event_offset=lo, n_events_total=Ng,
                     dist_group=ctx.dist.group.WORLD, **kw)
    for e in (full, part):
        e.init_params()
        e.begin_stage(0.01)
        e.run_steps(steps, 0)
    torch.cuda.synchronize()
    tr_full = full.group_trace(steps)[0, 0]
    tr_part = part.group_trace(steps)[0, 0]                      # all-reduced over ranks
    out = {"cells": Nc, "events": Ng, "Kg": Kg, "steps": steps,
           "max_abs_diff_Wg": float((full.Wg - part.Wg).abs().max()),
           "max_abs_diff_intercept": float((full.intercept - part.intercept).abs().max()),
           "max_abs_diff_sigma_log": float((full.sigma_log - part.sigma_log).abs().max()),
           "max_abs_diff_Z_loc": float((full.Z_loc[0, :, lo:hi] - part.Z_loc[0, :, :hi - lo]).abs().max()),
           "max_rel_diff_loss_trace": float(np.abs(tr_full - tr_part).max() / np.abs(tr_full).max())}
    for k in list(out):
        if k.startswith("max_"):
            out[k] = ctx.max_over_ranks(out[k])
    out["ok"] = bool(out["max_abs_diff_Wg"] < 1e-4 and out["max_abs_diff_Z_loc"] < 1e-4 and
                     out["max_rel_diff_loss_trace"] < 1e-5)
    del full, part
    torch.cuda.empty_cache()
    return out


def device_block_to_csc(t, n):
    """(Nc, ld) device tile -> host CSC of its first n columns."""
    import torch
    from scipy.sparse import csc_matrix
    tt = t[:, :n].t().contiguous()
    nz = tt != 0
    colrow = nz.nonzero()
    indptr = np.zeros(n + 1, np.int64)
    indptr[1:] = np.cumsum(nz.sum(1).cpu().numpy())
    return csc_matrix((tt[nz].cpu().numpy(), colrow[:, 1].to(torch.int32).cpu().numpy(), indptr), shape=(t.shape[0], n))


def e2e_leg(ctx, name, min_iter, out_root):
    """fitBRIE on the whole named workload from host CSC layers; every rank holds the AnnData with its own
    event shard's columns filled (the columns it reads), drawn on the device and brought to the host untimed."""
    torch = ctx.torch
    from scipy.sparse import csc_matrix, hstack
    from brie_b200.models import fitBRIE
    from brie_b200.utils.anndata_lite import AnnDataLite
    from brie_b200.utils.synth import make_design, simulate_counts_device
    c = SHAPES[name]
    Nc, Ng = c["cells"], c["events"]
    (lo, hi), group, _ = shard_of(ctx, name)
    Xc = make_design(Nc, c["design"], np.random.default_rng(0))
    keys = ('isoform1', 'isoform2', 'ambiguous')[:c["layers"]]
    blocks = {k: [csc_matrix((Nc, lo), dtype=np.float32)] for k in keys}
    eff = np.ones((Ng, 6), np.float32)
    for b0 in range(lo // 512 * 512, hi, 512):             # global 512-event blocks: the data do not depend on the sharding
        nb = min(512, Ng - b0)
        sim = simulate_counts_device(Nc, nb, design=c["design"], seed=100 + b0, with_efflen=c["eff"],
                                     n_layers=c["layers"], pseudo_count=0.0, event_offset=b0, Xc=Xc, device=ctx.dev)
        s0, s1 = max(lo, b0) - b0, min(hi, b0 + nb) - b0        # this rank's columns of the block
        for k, t in zip(keys, sim['layers']):
            blocks[k].append(device_block_to_csc(t[:, s0:s1], s1 - s0))
        if c["eff"]:
            eff[b0 + s0:b0 + s1] = sim['effLen'][s0:s1]
        del sim
    for k in keys:
        blocks[k].append(csc_matrix((Nc, Ng - hi), dtype=np.float32))
    layers = {k: hstack(v, format='csc') for k, v in blocks.items()}
    del blocks
    torch.cuda.empty_cache()
    h2d = sum(v.data.nbytes + v.indices.nbytes + (hi - lo + 1) * 8 for v in layers.values())
    ad = AnnDataLite(X=layers[keys[0]], layers=layers, varm={'effLen': eff} if c["eff"] else {})
    out_dir = os.path.join(out_root, "brie_bench_e2e_%s" % name)
    ctx.barrier()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        res = fitBRIE(ad, Xc=Xc, LRT_index=None, intercept_mode=c["mode"], layer_keys=list(keys),
                      min_iter=min_iter, max_iter=4 * min_iter, MC_size=S, seed=7, out_dir=out_dir)
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    n_stage = int(min_iter / 6)
    ran = (np.asarray(res.n_iter) - min_iter) + 6 * n_stage           # steps run per (model, batch); all batches, all ranks
    ev_per_group = np.minimum(group, Ng - np.arange(ran.shape[1]) * group)
    units = float((ran * ev_per_group[None, :]).sum()) * Nc * S
    steps_max = int(ran.max())
    d2h = 4 * Nc * (hi - lo) * 4 + 3 * (hi - lo) * 4
    psi_ok = bool(np.isfinite(np.asarray(ad.layers['Psi'][:, lo:min(lo + 8, hi)])).all())
    out = {"value": units / dt, "unit": UNIT, "h2d_bytes_per_step": ctx.sum_over_ranks(h2d) / steps_max,
           "d2h_bytes_per_step": ctx.sum_over_ranks(d2h) / steps_max, "wall_s": dt, "steps_max": steps_max,
           "steps_mean": float(ran.mean()), "min_iter": min_iter, "max_iter": 4 * min_iter, "workload": c["name"],
           "api": "brie_b200.models.fitBRIE(AnnData with host scipy CSC layers) -> device ingest, full schedule, "
                  "per-batch convergence extensions, loss_gene, LRT, p/FDR, D2H of 4 dense layers into .npy maps",
           "fdr05_calls": [int(v) for v in (np.asarray(res.fdr) < 0.05).sum(0)], "outputs_finite": psi_ok,
           "output_maps": out_dir + " (removed after the run)"}
    del res
    ad.layers.clear()
    ctx.barrier()
    if ctx.rank == 0:                              # 4 x (cells, events) float32 maps: do not leave them on the box
        import shutil
        shutil.rmtree(out_dir, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-shapes", action="store_true")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--e2e-min-iter", type=int, default=5000)
    ap.add_argument("--e2e-max-s", type=float, default=420.0,
                    help="run the end-to-end leg on the headline workload only if its predicted wall time is below this; "
                         "else on C2 (said in e2e.workload)")
    ap.add_argument("--out-root", default="/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline fit's state after its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
        return run_reference_arm(args)

    ctx = Ctx()
    torch = ctx.torch
    W, K = max(args.warmup, 3), args.steps
    c = SHAPES[HEAD]
    M = len(c["masks"])
    (lo, hi), group, Ng = shard_of(ctx, HEAD)

    # ---- the small shape first, from an idle GPU: C2 is a 25 ms burst whose clocks should not be those the long legs leave
    shapes = None
    if not args.no_shapes:
        shapes = {"C2": shape_leg(ctx, "C2", max(K, 50), W)}

    # ---- headline: C3, strong scaling, device-resident
    eng, nz = build_engine(ctx, HEAD, lo, hi, Ng, group)
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
        time.sleep(0.25)
    r = time_steps(ctx, eng, K, W)
    clocks = sampler.stop(r["t0"], r["t1"]) if ctx.rank == 0 else None
    if args.dump_outputs:
        dump_outputs(ctx, eng, args.dump_outputs)
    value = c["cells"] * Ng * S * M * K / (r["ms"] * 1e-3)
    peak, peak_src = hbm_peak()
    alg_bytes = c["cells"] * (hi - lo) * (4 * c["layers"] + 48 * M)        # this GPU's launch (SURVEY.md 8d)
    achieved = alg_bytes / (r["kernel_ms"] * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": "elbo_step_kernel<KC=4 (3 covariates padded),KG=0,gene,noloss>",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
            "peak_source": peak_src, "kernel_ms": r["kernel_ms"], "kernel_share_of_step": r["kernel_ms"] * K / r["ms_local"],
            "algorithmic_bytes_per_launch": alg_bytes, "per": "GPU (rank 0's launch over its event shard)"}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        ent = tj.get(HEAD) if isinstance(tj.get(HEAD), dict) else None
        if ent and ctx.world == 1:
            roof["traffic"] = ent.get("dram_bytes_per_launch")
            roof["traffic_source"] = ent.get("source")
    launches = r["launches"]
    state_gb = torch.cuda.memory_allocated() / 1e9
    del eng
    torch.cuda.empty_cache()

    if not args.no_shapes:
        ev5 = min(SHAPES["C5"]["events"] // ctx.world, 2048) * ctx.world
        shapes["C5"] = shape_leg(ctx, "C5", min(K, 10), 3, events=ev5,
                                 note="per-GPU slab of %d events (the full 20 000 need 8 GPUs: 150 GB per GPU)" % (ev5 // ctx.world))
    c4 = None if args.no_c4 else c4_leg(ctx, min(K, 20), 3)

    e2e = None
    if not args.no_e2e:
        predicted = r["ms"] / K * 1e-3 * (args.e2e_min_iter * 1.12) * 1.1 + 25
        name = HEAD if predicted <= args.e2e_max_s else "C2"
        e2e = e2e_leg(ctx, name, args.e2e_min_iter, args.out_root)
        e2e["predicted_wall_s"] = predicted

    cpu = None
    if ctx.rank == 0 and not args.no_cpu:
        threads = os.cpu_count() or 1
        v, cms, sample = cpu_reference_run(12, 2, threads)
        v6, _, _ = cpu_reference_run(6, 1, min(6, threads))      # the reference's own default, --nproc 6 (quant.py:183)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "ms_per_step": cms,
               "value_at_nproc_6": v6, "note": "restated reference, PyTorch-CPU eager -- not TensorFlow"}

    if ctx.rank == 0:
        cfg = config_dict(ctx.world)                 # identical to the reference arm's
        run_info = {"events_this_rank": hi - lo, "nonzero_fraction": nz, "resident_GB_per_gpu": state_gb}
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": K, "warmup": W,
               "ms_per_step": r["ms"] / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": cfg,
               "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof,
               "cpu_baseline": cpu, "fit_lrt_wall_s": e2e["wall_s"] if e2e else None, "shapes": shapes, "c4": c4,
               "run_info": run_info}
        print(json.dumps(out))
    if ctx.dist is not None:
        ctx.dist.barrier()
        from brie_b200 import comm
        comm.destroy_all()
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
