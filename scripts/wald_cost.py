"""Cost of the Wald information pass (brie_fit_wald_info) against the fit it reads.

Shapes (one model each, per-event intercept, three count layers with effective lengths, counts drawn on the device):
  C2        5 000 cells x 5 000 events, one binary covariate (Kc 1 -> K~ 2, 3 pairs, one pair block);
  C3-slab   100 000 cells x 2 500 events, the C3 design (Kc 3 -> K~ 4, 10 pairs, one pair block);
  C3-slab16 the same slab with 16 covariates (K~ 17, 153 pairs, 5 pair blocks of 36): the pass reads Z_std_log
            once per pair block.
The fit runs a fixed schedule (min_iter = max_iter = --iters) and is timed by the host clock around
FitEngine.fit with a device synchronise; the information pass is timed with CUDA events around --reps calls of the
ABI entry point after a warm-up call (device output only: no copy to the host).  Prints one JSON line per shape and
writes them to --out, with the card's name and power limit (read-only nvidia-smi query).

    python scripts/wald_cost.py [--iters 1200] [--reps 20] [--out profiles/wald_cost.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


SHAPES = {
    "C2": dict(Nc=5000, Ng=5000, design='binary1', Kc=None),
    "C3-slab": dict(Nc=100000, Ng=2500, design='mixed3', Kc=None),
    "C3-slab16": dict(Nc=100000, Ng=2500, design='mixed3', Kc=16),
}


def run_shape(name, iters, reps):
    import torch
    from brie_b200 import _lib
    from brie_b200.engine import FitEngine
    from brie_b200.utils.synth import simulate_counts_device
    sh = SHAPES[name]
    Xc = None
    if sh['Kc'] is not None:
        Xc = np.random.default_rng(3).standard_normal((sh['Nc'], sh['Kc'])).astype(np.float32)
        Xc[:, 0] = Xc[:, 0] > 0
    d = simulate_counts_device(sh['Nc'], sh['Ng'], design=sh['design'], seed=1, Xc=Xc)
    eng = FitEngine(d['layers'], effLen=d['effLen'], Xc=d['Xc'], MC_size=1, seed=7, n_events=sh['Ng'])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.fit(min_iter=iters, max_iter=iters, n_eval=500)
    torch.cuda.synchronize()
    fit_s = time.perf_counter() - t0
    lib = eng.lib
    nbytes, kt = C.c_size_t(), C.c_int32()
    _lib.check(lib.brie_fit_wald_sizes(eng.h, 0, C.byref(nbytes), C.byref(kt)))
    n_pairs = kt.value * (kt.value + 1) // 2
    info = torch.empty((eng.Ng, n_pairs), dtype=torch.float64, device=eng.device)
    scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=eng.device)
    call = lambda: _lib.check(lib.brie_fit_wald_info(eng.h, 0, info.data_ptr(), scratch.data_ptr(), eng._stream()))
    call()
    first = info.clone()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    torch.cuda.synchronize()
    wald_ms = e0.elapsed_time(e1) / reps
    n_pblk = -(-n_pairs // (4 if n_pairs <= 4 else 12 if n_pairs <= 12 else 36))
    read_bytes = n_pblk * eng.Nc * eng.Ng * 4.0                   # Z_std_log once per pair block
    return dict(shape=name, cells=eng.Nc, events=eng.Ng, Kc=int(d['Xc'].shape[1]), k_tilde=kt.value,
                n_pairs=n_pairs, pair_blocks=n_pblk, fit_iters=iters, fit_s=fit_s,
                fit_ms_per_step=1e3 * fit_s / iters, wald_ms=wald_ms, wald_over_fit=wald_ms / (1e3 * fit_s),
                wald_read_GBps=read_bytes / (wald_ms * 1e-3) / 1e9, scratch_MB=nbytes.value / 1e6,
                repeat_bit_identical=bool(torch.equal(first, info)), **card())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=1200)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wald_cost: needs a CUDA device")
    lines = []
    for name in args.shapes.split(","):
        line = json.dumps(run_shape(name, args.iters, args.reps))
        print(line, flush=True)
        lines.append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
