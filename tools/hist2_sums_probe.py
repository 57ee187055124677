"""Cost of swrt_hist2_sums at the C4 size (16.8M packets, one GPU), next to swrt_hist2 on the same bins and one C4
leapfrog step.

    python tools/hist2_sums_probe.py [--packets N] [--reps R] [--out FILE.json]

hist2_sums(KMAG, THETA) is timed with 128 x 256 and 512 x 512 bins (and 32 x 36, the size at which a per-CTA copy of the
counters would still fit shared memory), on uniformly random wavevectors and on the C4 ring initial condition, with one
weight kind (energy) and all four.  The actions are spread over [0.5, 2].  Per case: the whole call as a caller sees it
(host clock: scale pass, memsets, sums kernel, accumulators copied back and rounded on the host), measured in alternating
repeats with swrt_hist2 on the same bins, median / min / max of each; the kernels alone (torch.profiler, CUDA activity, a
separate pass); and the host rounding (swrt_fixed_sums_to_double) alone.  The counts are checked against swrt_hist2's.  The
card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import swraytracing_b200 as S  # noqa: E402
from swraytracing_b200 import workloads as W  # noqa: E402
from hist2_probe import card, kernel_ms  # noqa: E402

KERNELS = ["hist2_sums_kernel", "weight_scale_kernel", "omega_kernel", "hist2_kernel"]


def alternating_ms(fns, reps):
    """wall times (ms) of each callable, run in turn rep by rep after one warm-up each"""
    for f in fns:
        f()
    ts = [[] for _ in fns]
    for _ in range(reps):
        for i, f in enumerate(fns):
            t0 = time.perf_counter()
            f()
            ts[i].append((time.perf_counter() - t0) * 1e3)
    return [{"median": float(np.median(t)), "min": float(np.min(t)), "max": float(np.max(t))} for t in ts]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--packets", type=int, default=0, help="0 = the C4 count (16,777,216)")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    a = ap.parse_args()
    if S.load_library().swrt_device_count() < 1:
        sys.exit("hist2_sums_probe: no CUDA device (the probe measures the GPU and has no CPU path)")
    import torch
    torch.cuda.init()
    w = W.make_workload("C4", n_packets=a.packets or None)
    n = w.n_packets
    k0 = float(np.hypot(w.k[0], w.l[0]))
    rs = np.random.default_rng(5)
    th = rs.uniform(-np.pi, np.pi, n)
    km = rs.uniform(0.0, 2.0 * k0, n)
    act = rs.uniform(0.5, 2.0, n)
    cases = {"random": (km * np.cos(th), km * np.sin(th)), "ring": (w.k, w.l)}
    del th, km
    grids = {f"{nb[0]}x{nb[1]}": (np.linspace(0.0, 2.0 * k0, nb[0] + 1), np.linspace(-np.pi, np.pi, nb[1] + 1))
             for nb in ((32, 36), (128, 256), (512, 512))}
    kinds = {"nw=1": [S.W_ENERGY], "nw=4": [S.W_ACTION, S.W_ENERGY, S.W_PSEUDO_K, S.W_PSEUDO_L]}
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL)
    eng.set_flow_spectral(w.psik, 0, w.u_mean)
    eng.set_flow_spectral(w.psik2, 1, w.u_mean)
    res = {"card": card(), "packets": n, "reps": a.reps, "cases": {}}
    print(f"card: {res['card']}; {n} packets; {a.reps} alternating repeats")
    for cname, (k, l) in cases.items():
        eng.set_packets(w.x, w.y, k, l, act)
        for gname, (xe, ye) in grids.items():
            h2 = lambda: eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)                               # noqa: E731
            for kname, wk in kinds.items():
                hs = lambda: eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, wk)                   # noqa: E731
                sums, counts, acc = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, wk, return_acc=True)
                ok = bool(np.array_equal(counts, h2()))
                exps = eng.weight_scale(wk)
                t0 = time.perf_counter()
                S.fixed_sums_to_double(acc, exps)
                host_ms = (time.perf_counter() - t0) * 1e3
                t_sums, t_h2 = alternating_ms([hs, h2], a.reps)
                kt = kernel_ms(hs, a.reps, KERNELS)
                row = {"hist2_sums_call_ms": t_sums, "hist2_call_ms": t_h2, "kernel_ms": kt, "host_rounding_ms": host_ms,
                       "counts_equal_hist2": ok, "occupied_bins": int(np.count_nonzero(counts))}
                res["cases"][f"{cname} {gname} {kname}"] = row
                print(f"  {cname:6s} {gname:7s} {kname}: hist2_sums call {t_sums['median']:.2f} ms [{t_sums['min']:.2f}, {t_sums['max']:.2f}]"
                      f" vs hist2 {t_h2['median']:.2f} ms [{t_h2['min']:.2f}, {t_h2['max']:.2f}];"
                      f" kernels {({kk: round(v * 1e3, 1) for kk, v in kt.items()})} us; host rounding {host_ms:.2f} ms;"
                      f" counts equal hist2: {ok}")
    eng.set_packets(w.x, w.y, w.k, w.l)
    step = lambda: eng.step(S.SCHEME_LEAPFROG, w.dt / 2, 2, 0.25, 0.5)      # noqa: E731  one C4 step: 2 fused sub-steps
    t_step, = alternating_ms([step], max(a.reps // 2, 3))
    res["c4_leapfrog_step_ms"] = t_step
    print(f"  one C4 leapfrog step (2 sub-steps): {t_step['median']:.2f} ms [{t_step['min']:.2f}, {t_step['max']:.2f}]")
    eng.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
