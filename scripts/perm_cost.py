"""Wall-time cost of the permutation null (fit_BRIE_matrix n_perm) on config C2.

C2: 5 000 cells x 5 000 events, three count layers with effective lengths, one binary cell covariate, LRT on
it (LRT_index=[0], base_mode 'full', per-event intercept).  Times fit_BRIE_matrix at n_perm = 0 and n_perm = 8,
alternating the two in one process after a warm-up of both, with a fixed step count (min_iter = max_iter) so
that both arms run the same schedule.  Prints one JSON line with both walls (median over the repetitions),
their ratio, and the card's name and power limit (read-only nvidia-smi query).

    python scripts/perm_cost.py [--reps 3] [--iters 3000] [--out profiles/perm_cost_c2.json]
"""
import argparse
import contextlib
import io
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3000)
    ap.add_argument("--n-perm", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("perm_cost: needs a CUDA device")
    from brie_b200.models import fit_BRIE_matrix
    from brie_b200.utils.synth import simulate_counts
    Nc, Ng = 5000, 5000
    d = simulate_counts(Nc, Ng, design='binary1', seed=1)
    layers = [np.ascontiguousarray(x, np.float32) for x in d['layers']]
    kw = dict(Xc=d['Xc'], effLen=d['effLen'], LRT_index=[0], intercept_mode='gene', MC_size=1, seed=7,
              host_side_effect=False)

    def fit(n_perm, iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            r = fit_BRIE_matrix(layers, min_iter=iters, max_iter=iters, n_perm=n_perm, **kw)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    for B in (0, args.n_perm):                                  # warm-up: module load, allocator, both plans
        fit(B, 60)
    walls = {0: [], args.n_perm: []}
    for _ in range(args.reps):
        for B in (0, args.n_perm):
            dt, r = fit(B, args.iters)
            walls[B].append(dt)
    w0, wb = float(np.median(walls[0])), float(np.median(walls[args.n_perm]))
    out = dict(workload="C2 fit_BRIE_matrix, 5000 cells x 5000 events, Kc=1, LRT_index=[0], full base",
               iters=args.iters, n_perm=args.n_perm, reps=args.reps, wall_s_n_perm_0=w0,
               wall_s_n_perm=wb, ratio=wb / w0, walls_n_perm_0=walls[0], walls_n_perm=walls[args.n_perm],
               byte_model_ratio=1 + args.n_perm / 2, **card())
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
