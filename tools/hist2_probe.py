"""Cost of swrt_hist2 at the C4 size (16.8M packets, one GPU), next to swrt_hist_omega and one C4 leapfrog step.

    python tools/hist2_probe.py [--packets N] [--reps R] [--out FILE.json]

hist2(KMAG, THETA) is timed with 128 x 256 bins (128 KB of u32 counters: the per-CTA shared-memory path) and 512 x 512 bins
(the global-counter path), on uniformly random wavevectors and on the C4 ring initial condition (every packet on |k| = k0,
so the |k| axis holds one bin).  Two numbers per case: the whole call as a caller sees it (host clock; memset, kernel,
counts copied back) and the histogram kernel alone (torch.profiler, CUDA activity, in a separate pass).  Each case's
counts are checked against a host histcounts2 of the device's own packet_quantity arrays.  The card's name, power limit
and maximum SM clock are read in the same run.  k and l of 16.8M packets are 269 MB, more than the 126 MB L2, so every
pass reads them from HBM."""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import swraytracing_b200 as S  # noqa: E402
from swraytracing_b200 import workloads as W  # noqa: E402
from test_hist2_contract import histcounts2  # noqa: E402

HBM_TBS = 7.7          # data-sheet HBM3e bandwidth of one B200 (not measured here)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def wall_ms(fn, reps):
    fn()                                                   # warm-up (module load, buffer growth, edge upload)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def kernel_ms(fn, reps, names):
    """mean device time per call of the kernels whose name contains one of ``names`` (torch.profiler)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.key_averages():
        key = next((n for n in names if n in e.key), None)
        if key:
            tot[key] = tot.get(key, 0.0) + e.self_device_time_total / 1e3
    return {k: v / reps for k, v in tot.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--packets", type=int, default=0, help="0 = the C4 count (16,777,216)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    a = ap.parse_args()
    if S.load_library().swrt_device_count() < 1:
        sys.exit("hist2_probe: no CUDA device (the probe measures the GPU and has no CPU path)")
    import torch
    torch.cuda.init()
    w = W.make_workload("C4", n_packets=a.packets or None)
    n = w.n_packets
    k0 = float(np.hypot(w.k[0], w.l[0]))
    rs = np.random.default_rng(5)
    th = rs.uniform(-np.pi, np.pi, n)
    km = rs.uniform(0.0, 2.0 * k0, n)
    cases = {"uniform": (km * np.cos(th), km * np.sin(th)), "ring": (w.k, w.l)}
    del th, km
    grids = {"128x256 (shared)": (np.linspace(0.0, 2.0 * k0, 129), np.linspace(-np.pi, np.pi, 257)),
             "512x512 (global)": (np.linspace(0.0, 2.0 * k0, 513), np.linspace(-np.pi, np.pi, 513))}
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL)
    eng.set_flow_spectral(w.psik, 0, w.u_mean)
    eng.set_flow_spectral(w.psik2, 1, w.u_mean)
    res = {"card": card(), "packets": n, "k0": k0, "reps": a.reps,
           "bytes_bound_us": n * 16 / (HBM_TBS * 1e12) * 1e6, "bytes_bound_note": "k and l, 16 B a packet, at the data-sheet "
           f"{HBM_TBS} TB/s; not measured", "cases": {}}
    print(f"card: {res['card']}; {n} packets; k0 = {k0:.4f}; k,l read bound {res['bytes_bound_us']:.1f} us (data sheet)")
    for cname, (k, l) in cases.items():
        eng.set_packets(w.x, w.y, k, l)
        row = {}
        vk, vt = eng.packet_quantity(S.Q_KMAG), eng.packet_quantity(S.Q_THETA)
        for gname, (xe, ye) in grids.items():
            N = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)
            ok = bool(np.array_equal(N, histcounts2(vk, vt, xe, ye)))
            f = lambda: eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)          # noqa: E731
            med, best = wall_ms(f, a.reps)
            kt = kernel_ms(f, a.reps, ["hist2_kernel"])
            row[gname] = {"call_ms_median": med, "call_ms_min": best, "kernel_ms": kt.get("hist2_kernel"), "equals_host": ok,
                          "occupied_bins": int(np.count_nonzero(N)), "counted": int(N.sum())}
            print(f"  {cname:8s} hist2 {gname:17s}: call {med:.3f} ms (min {best:.3f}), kernel {kt.get('hist2_kernel', float('nan')) * 1e3:.1f} us,"
                  f" {row[gname]['occupied_bins']} bins occupied, equals host histcounts2: {ok}")
        edges = np.linspace(0.0, float(np.sqrt(w.f ** 2 + w.gH * 4 * k0 * k0)), 300)
        f = lambda: eng.hist_omega(edges)                                # noqa: E731
        med, best = wall_ms(f, a.reps)
        kt = kernel_ms(f, a.reps, ["hist_kernel", "omega_kernel"])
        row["hist_omega 299 bins"] = {"call_ms_median": med, "call_ms_min": best, "kernel_ms": kt}
        print(f"  {cname:8s} hist_omega 299 bins : call {med:.3f} ms (min {best:.3f}), kernels {({k: round(v * 1e3, 1) for k, v in kt.items()})} us")
        res["cases"][cname] = row
    eng.set_packets(w.x, w.y, w.k, w.l)
    step = lambda: eng.step(S.SCHEME_LEAPFROG, w.dt / 2, 2, 0.25, 0.5)      # noqa: E731  one C4 step: 2 fused sub-steps
    med, best = wall_ms(step, max(a.reps // 4, 3))
    res["c4_leapfrog_step"] = {"call_ms_median": med, "call_ms_min": best, "kernel_ms": eng.last_kernel_ms()[0]}
    print(f"  one C4 leapfrog step (2 sub-steps): call {med:.2f} ms (min {best:.2f}), packet kernel {eng.last_kernel_ms()[0]:.2f} ms")
    eng.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
