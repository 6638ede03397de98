"""Cost of the score-test pass (brie_fit_score_parts) against the fit it reads.

Shapes (one model each, per-event intercept, three count layers with effective lengths, counts drawn on the device):
  C2        5 000 cells x 5 000 events, one binary covariate (Kc 1 -> K~ 2);
  C3-slab   100 000 cells x 2 500 events, the C3 design (Kc 3 -> K~ 4).
Each shape is scored against J = 64 and J = 512 standard-normal candidates in one call of the ABI entry point
(device outputs only: no copy to the host).  The fit runs a fixed schedule (min_iter = max_iter = --iters) and is
timed by the host clock around FitEngine.fit with a device synchronise; the pass is timed with CUDA events around
--reps calls after a warm-up call.  The FP64 operation count is the one the statistic needs per (cell, event):
J (K~ + 3) + K~ fused multiply-adds or multiplies (U, A with its w x product, B, Ut); the rate is that count over
the pass time.  Prints one JSON line per (shape, J) and writes them to --out, with the card's name and power limit
(read-only nvidia-smi query).

    python scripts/score_cost.py [--iters 1200] [--reps 10] [--out profiles/score_cost.jsonl]
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


def run_shape(name, iters, reps, Js):
    import torch
    from brie_b200 import _lib
    from brie_b200.engine import FitEngine
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
    out = []
    for J in Js:
        X = torch.randn((eng.Nc, J), generator=torch.Generator().manual_seed(J)).to(eng.device)
        nbytes, kt = C.c_size_t(), C.c_int32()
        _lib.check(lib.brie_fit_score_sizes(eng.h, 0, J, C.byref(nbytes), C.byref(kt)))
        kt = kt.value
        new = lambda *s: torch.empty(s, dtype=torch.float64, device=eng.device)
        U, A, B, Ut = new(eng.Ng, J), new(eng.Ng, J), new(eng.Ng, J, kt), new(eng.Ng, kt)
        scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=eng.device)
        call = lambda: _lib.check(lib.brie_fit_score_parts(eng.h, 0, X.data_ptr(), J, J, U.data_ptr(), A.data_ptr(),
                                                           B.data_ptr(), Ut.data_ptr(), scratch.data_ptr(),
                                                           eng._stream()))
        call()
        first = B.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        flops = float(eng.Nc) * eng.Ng * (J * (kt + 3) + kt)
        out.append(dict(shape=name, cells=eng.Nc, events=eng.Ng, Kc=int(d['Xc'].shape[1]), k_tilde=kt, J=J,
                        fit_iters=iters, fit_s=fit_s, score_ms=ms, score_over_fit=ms / (1e3 * fit_s),
                        fp64_ops=flops, fp64_Tops=flops / (ms * 1e-3) / 1e12, scratch_MB=nbytes.value / 1e6,
                        reps=reps, repeat_bit_identical=bool(torch.equal(first, B)), **card()))
        del U, A, B, Ut, scratch, X
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=1200)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--shapes", default="C2,C3-slab")
    ap.add_argument("--J", default="64,512")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("score_cost: needs a CUDA device")
    lines = []
    for name in args.shapes.split(","):
        for rec in run_shape(name, args.iters, args.reps, [int(j) for j in args.J.split(",")]):
            line = json.dumps(rec)
            print(line, flush=True)
            lines.append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
