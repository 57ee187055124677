"""Per-kernel time of the anchored SPECTRAL leapfrog: drift + key, sort (scan + scatter), K1 (the expansion blocks of every
anchor cell, anchor_transform_kernel), K2 (anchored_step_kernel), from torch.profiler's CUDA activity records.

    python tools/anchored_breakdown.py [--out DIR]

Shapes: C4 (512^2 two-frame, 16,777,216 packets, 2 sub-steps per step) and 65,536 packets at 512^2 (two packets per
anchor cell: K1 costs the same whatever the packet count).  The whole step is also timed with CUDA events
(L2 not flushed; median of 5).  Prints one JSON object per shape and writes them to DIR/anchored_breakdown.json.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def classify(name):
    if "anchor_key_kernel" in name:
        return "drift_key"
    if "anchor_scan_kernel" in name or "anchor_scatter_kernel" in name:
        return "sort"
    if "anchor_transform_kernel" in name:
        return "K1"
    if "anchored_step_kernel" in name:
        return "K2"
    if "axpby" in name:
        return "stack_blend"
    return "other"


def one_shape(torch, S, W, n, steps=3):
    w = W.make_workload("C4", n_packets=n)
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL, device=0)
    eng.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
    eng.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
    eng.set_packets(w.x, w.y, w.k, w.l)
    sub = 2
    args = (S.SCHEME_LEAPFROG, w.dt / sub, sub, 0.5 / sub, 1.0 / sub)
    for _ in range(2):
        eng.step(*args)
    ms = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.step(*args)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            eng.step(*args)
        torch.cuda.synchronize()
    eng.close()
    per = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        key = classify(ev.name)
        per[key] = per.get(key, 0.0) + ev.device_time / 1e3 / steps
    return {"packets": n, "nx": w.nx, "substeps_per_step": sub, "step_ms_events_median": float(np.median(ms)),
            "kernel_ms_per_step": {k: round(v, 4) for k, v in sorted(per.items())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this tool measures on the GPU")
    import swraytracing_b200 as S
    from swraytracing_b200 import workloads as W
    props = torch.cuda.get_device_properties(0)
    res = {"device": props.name, "shapes": [one_shape(torch, S, W, n) for n in (16777216, 65536)]}
    print(json.dumps(res))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "anchored_breakdown.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
