"""swrt_ode23_packets without events against swrt_ode23_packets_events with four non-terminal events (X, Y, |k|, omega),
once returning four records per packet and once with ev_cap = 0 (counts only, which isolates the device work from the
copy of the records to the host), on the reference's unit of work: one per-packet ode23 solve over a QG step [0, dt]
between two flow frames (qgsw_raytrace.m:141-150), C3 flow (256^2).  The three solves alternate in one process; the
wall time of a solve ends in a device synchronise and is the median of the repeats.  The event levels sit at the median
of the initial state, so about half the packets start on each side.  The device name and power limit are read in the
same run.  With a second argument, the rows are also written to that JSON file.
    python tools/ode23_events_probe.py [reps [out.json]]"""
import json, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np
import swraytracing_b200 as S
from swraytracing_b200 import workloads as W

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
print("device:", gpu)
MODES = (("SPECTRAL", S.MODE_SPECTRAL), ("LAGRANGE6", S.MODE_LAGRANGE6), ("NUFFT", S.MODE_NUFFT))


def solve_ms(e, w, events, cap, reps):
    ts = []
    for _ in range(reps):
        e.set_packets(w.x, w.y, w.k, w.l)
        e.synchronize()
        t0 = time.perf_counter()
        st = e.ode23_packets([0.0, w.dt], w.dt, events=events, ev_cap=cap)
        e.synchronize()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts)), st


rows = []
for n, modes, r in ((50, MODES, reps), (1 << 20, MODES[1:], max(2, reps // 10))):
    w = W.make_workload("C3", n_packets=n)
    om = np.sqrt(w.f * w.f + w.gH * (w.k * w.k + w.l * w.l))
    events = [(S.EVENT_X, float(np.median(w.x))), (S.EVENT_Y, float(np.median(w.y))),
              (S.EVENT_KMAG, float(np.median(np.hypot(w.k, w.l)))), (S.EVENT_OMEGA, float(np.median(om)))]
    for name, mode in modes:
        e = S.Engine(w.nx, w.L, w.f, w.gH, mode)
        e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
        variants = ((None, 0), (events, 4), (events, 0))
        for ev, cap in variants:                         # warm-up: stacks, grids, module loads, per-packet state
            solve_ms(e, w, ev, cap, 1)
        res = [[] for _ in variants]
        for _ in range(3):                               # alternate the solves
            for j, (ev, cap) in enumerate(variants):
                ms, st = solve_ms(e, w, ev, cap, r)
                res[j].append(ms)
        row = {"n": n, "mode": name, "events_found": int(st["events"]), "packets_with_events": int((st["ne"] > 0).sum()),
               "plain_ms": float(np.median(res[0])), "events_ms": float(np.median(res[1])),
               "events_cap0_ms": float(np.median(res[2])), "plain_ms_all": res[0], "events_ms_all": res[1],
               "events_cap0_ms_all": res[2]}
        rows.append(row)
        print(f"C3 flow, {n:8d} packets, {name:9s}: swrt_ode23_packets {row['plain_ms']:8.3f} ms, with 4 events "
              f"{row['events_ms']:8.3f} ms (ratio {row['events_ms'] / row['plain_ms']:.3f}), counts only "
              f"{row['events_cap0_ms']:8.3f} ms (ratio {row['events_cap0_ms'] / row['plain_ms']:.3f}); "
              f"{row['events_found']} events in {row['packets_with_events']} packets")
        e.close()
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as fh:
        json.dump({"device": gpu, "rows": rows}, fh, indent=1)
