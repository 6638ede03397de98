#!/usr/bin/env python
"""Per-pass accounting of the two-step passes of one `run_steps(K)` call on a bench.py shape (default: the C3 headline).

bench.py's roofline assumes one step per fused launch.  A per-event-only fit now takes its steps in pairs: a sums-only
pre-pass (kl_sums_kernel, plus gram_kernel), then K // 2 passes of elbo_step_kernel that each take two steps, each
followed by event_update_kernel.  This script times every kernel of the call with torch.profiler (CUDA activity) and
reports, per kind: launches, total and mean device time.  It then reports the bytes each kind moves and the rate it
reaches under the pair byte model (DESIGN.md section 3):
  pass      (count bytes + 48 M) per cell x event: counts as packed codes (4 B) or float32 tiles (4 B per layer),
            Z_loc, Z_std_log and their four Adam moments read and written, per model;
  pre-pass  8 M per cell x event (Z_loc, Z_std_log read);
and the call's wall time per step (CUDA events) and bytes per cell x event x step.

    python scripts/pair_pass_time.py [--shape C3] [--steps 20] [--warmup 5] [--json OUT]

Needs a GPU; writes nothing unless --json is given.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (shapes and the engine builder of the benchmark)

KINDS = ("elbo_step_kernel", "kl_sums_kernel", "gram_kernel", "event_update_kernel")


def kind_of(name):
    for k in KINDS:
        if k in name:
            return k
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default=bench.HEAD, choices=sorted(bench.SHAPES))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--json", help="also write the report to this file")
    args = ap.parse_args()
    ctx = bench.Ctx()
    torch = ctx.torch
    if ctx.world != 1:
        sys.exit("one GPU only")
    (lo, hi), group, Ng = bench.shard_of(ctx, args.shape)
    eng, _ = bench.build_engine(ctx, args.shape, lo, hi, Ng, group)
    K = args.steps
    eng.run_steps(args.warmup)
    torch.cuda.synchronize()

    # wall time of the call without the profiler
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.run_steps(K)
    e1.record()
    torch.cuda.synchronize()
    call_ms = e0.elapsed_time(e1)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.run_steps(K)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        k = kind_of(ev.name)
        n, us = per.get(k, (0, 0.0))
        per[k] = (n + 1, us + ev.time_range.elapsed_us())

    M, Nc = eng.M, eng.Nc
    count_b = 4 if eng.count_format == "code8" else 4 * eng.n_layers
    cells_events = float(Nc) * eng.Ng
    pass_bytes = (count_b + 48 * M) * cells_events
    pre_bytes = 8 * M * cells_events
    n_pass, n_single = K // 2, K % 2
    rep = {"shape": args.shape, "gpu": torch.cuda.get_device_name(), "steps": K, "models": M, "cells": Nc,
           "events": eng.Ng, "count_format": eng.count_format, "call_ms": call_ms, "ms_per_step": call_ms / K,
           "kernels": {k: {"launches": n, "total_ms": us / 1e3, "mean_ms": us / 1e3 / n} for k, (n, us) in per.items()}}
    step = rep["kernels"].get("elbo_step_kernel")
    pre = rep["kernels"].get("kl_sums_kernel")
    if step and n_single == 0 and step["launches"] == n_pass:   # an odd K's last launch is a single step
        rep["pass_ms"] = step["mean_ms"]
        rep["pass_TBps"] = pass_bytes / (step["mean_ms"] * 1e-3) / 1e12
    if pre:
        rep["prepass_ms"] = pre["mean_ms"]
        rep["prepass_TBps"] = pre_bytes / (pre["mean_ms"] * 1e-3) / 1e12
    rep["bytes_per_cell_event_step"] = ((n_pass + n_single) * (count_b + 48 * M) + (8 * M if pre else 0)) / K
    rep["call_TBps"] = rep["bytes_per_cell_event_step"] * cells_events * K / (call_ms * 1e-3) / 1e12
    print(json.dumps(rep, indent=1))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
