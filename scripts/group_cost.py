"""Cost of the joint group tests against the fit they read.

1. The cross-term pass (brie_fit_score_cross) against the fit: per shape (scripts/wald_cost.py SHAPES: C2 = 5 000 cells
   x 5 000 events, Kc 1; C3-slab = 100 000 x 2 500, Kc 3), one model fitted for --iters steps (host clock around
   FitEngine.fit with a device synchronise), then the pass over the pairs of one group of 2, 8 and 32 of 32
   standard-normal candidates (1, 28 and 496 pairs) in one call of the ABI entry point, timed with CUDA events
   around --reps calls after a warm-up call (device output only).  Bytes: the pass reads the model's Z_std_log plane
   once per 36-pair block.
2. Group LRT wall time against none on C2 with Kc 4: fit_BRIE_matrix(LRT_index=[]) with LRT_groups of G = 1 and 4
   groups of 2 columns, vs no groups, each the median of --runs alternating runs (host clock).  Byte model: with no
   LRT refits the observed engine holds one model, so each group refit is one more one-model engine, and each step of
   it streams the counts once plus that model's 48 B of state per element: about (1 + G) x the stepping bytes of the
   plain fit, plus one loss_gene evaluation per group.

Prints one JSON line per measurement and writes them to --out, with the card's name and power limit (read-only
nvidia-smi query).

    python scripts/group_cost.py [--iters 1200] [--reps 10] [--runs 3] [--out profiles/group_cost.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from wald_cost import SHAPES, card  # noqa: E402


def cross_vs_fit(name, iters, reps, sizes):
    import torch
    from brie_b200 import _lib
    from brie_b200.engine import FitEngine, group_pairs
    from brie_b200.utils.synth import simulate_counts_device
    sh = SHAPES[name]
    d = simulate_counts_device(sh['Nc'], sh['Ng'], design=sh['design'], seed=1)
    eng = FitEngine(d['layers'], effLen=d['effLen'], Xc=d['Xc'], MC_size=1, seed=7, n_events=sh['Ng'])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.fit(min_iter=iters, max_iter=iters, n_eval=500)
    torch.cuda.synchronize()
    fit_s = time.perf_counter() - t0
    lib = eng.lib
    X = torch.randn((eng.Nc, 32), generator=torch.Generator().manual_seed(3)).to(eng.device)
    out = []
    for k in sizes:
        pairs = group_pairs([list(range(k))])
        P = len(pairs)
        nbytes = C.c_size_t()
        _lib.check(lib.brie_fit_score_cross_sizes(eng.h, 0, P, C.byref(nbytes)))
        res = torch.empty((eng.Ng, P), dtype=torch.float64, device=eng.device)
        scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=eng.device)
        call = lambda: _lib.check(lib.brie_fit_score_cross(eng.h, 0, X.data_ptr(), 32, pairs.ctypes.data, P,
                                                           res.data_ptr(), scratch.data_ptr(), eng._stream()))
        call()
        first = res.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        n_blk = -(-P // 36)
        out.append(dict(kind="cross_pass", shape=name, cells=eng.Nc, events=eng.Ng, Kc=int(d['Xc'].shape[1]),
                        group=k, pairs=P, fit_iters=iters, fit_s=fit_s, cross_ms=ms, cross_over_fit=ms / (1e3 * fit_s),
                        plane_reads=n_blk, read_GBps=n_blk * 4.0 * eng.Nc * eng.Ng / (ms * 1e-3) / 1e9,
                        scratch_MB=nbytes.value / 1e6, reps=reps,
                        repeat_bit_identical=bool(torch.equal(first, res)), **card()))
        del res, scratch
        torch.cuda.empty_cache()
    return out


def group_lrt_wall(iters, runs, Gs):
    import torch
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.utils.synth import simulate_counts_device
    Nc, Ng = 5000, 5000
    d = simulate_counts_device(Nc, Ng, design='none', seed=1)
    layers = [t[:, :Ng].cpu().numpy() for t in d['layers']]
    Xc = np.random.default_rng(0).binomial(1, 0.3, (Nc, 4)).astype(np.float32)
    kw = dict(Xc=Xc, effLen=d['effLen'], LRT_index=[], intercept_mode='gene', min_iter=iters, max_iter=iters,
              MC_size=1, n_eval=500, seed=3)
    variants = [0] + list(Gs)
    times = {G: [] for G in variants}
    for _ in range(runs):
        for G in variants:
            groups = [[(2 * i) % 4, (2 * i + 1) % 4] for i in range(G)] or None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fit_BRIE_matrix([x.copy() for x in layers], LRT_groups=groups, **kw)
            torch.cuda.synchronize()
            times[G].append(time.perf_counter() - t0)
    base = float(np.median(times[0]))
    return [dict(kind="group_lrt_wall", shape="C2", cells=Nc, events=Ng, Kc=4, groups=G, fit_iters=iters,
                 median_s=float(np.median(times[G])), runs_s=times[G], over_none=float(np.median(times[G])) / base,
                 byte_model_over_none=1.0 + G, **card()) for G in variants]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=1200)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--shapes", default="C2,C3-slab")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("group_cost: needs a CUDA device")
    recs = []
    for name in args.shapes.split(","):
        recs += cross_vs_fit(name, args.iters, args.reps, (2, 8, 32))
        torch.cuda.empty_cache()
    recs += group_lrt_wall(args.iters, args.runs, (1, 4))
    lines = [json.dumps(r) for r in recs]
    print("\n".join(lines), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
