"""swrt_ode23_packets_tspans_events against swrt_ode23_packets_tspans (the same rows, no events) and
swrt_ode23_packets_events (one shared forward tspan) on the reference's unit of work: one per-packet ode23 solve over a QG
step between two flow frames, C3 flow (256^2), 1M packets, four non-terminal events (X, Y, |k|, omega at the median of
the initial state, as tools/ode23_events_probe.py sets them).
  forward:  every row [0, dt]; all three entry points take the same steps.
  backward: every row [dt, 0] (back-tracing over the step); swrt_ode23_packets_events refuses it.
The event solves run with four records per packet and with ev_cap = 0 (counts only, which leaves out the copy of the
records to the host).
The solves alternate in one process; the wall time of a solve ends in a device synchronise, and the median and the
min-max of the repeats are reported.  The device name and power limit are read in the same run.
    python tools/ode23_tspans_events_probe.py [reps [out.json]]"""
import json, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np
import swraytracing_b200 as S
from swraytracing_b200 import workloads as W

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
print("device:", gpu)
n = 1 << 20
w = W.make_workload("C3", n_packets=n)
om = np.sqrt(w.f * w.f + w.gH * (w.k * w.k + w.l * w.l))
EVENTS = [(S.EVENT_X, float(np.median(w.x))), (S.EVENT_Y, float(np.median(w.y))),
          (S.EVENT_KMAG, float(np.median(np.hypot(w.k, w.l)))), (S.EVENT_OMEGA, float(np.median(om)))]
fwd_rows = np.repeat(np.array([[0.0], [w.dt]]), n, axis=1)
bwd_rows = fwd_rows[::-1].copy()
CASES = {
    "fwd_packets_events": lambda e: e.ode23_packets([0.0, w.dt], w.dt, events=EVENTS, ev_cap=4),
    "fwd_tspans": lambda e: e.ode23_packets(fwd_rows, w.dt),
    "fwd_tspans_events": lambda e: e.ode23_packets_tspans_events(fwd_rows, w.dt, EVENTS, ev_cap=4),
    "bwd_tspans": lambda e: e.ode23_packets(bwd_rows, w.dt),
    "bwd_tspans_events": lambda e: e.ode23_packets_tspans_events(bwd_rows, w.dt, EVENTS, ev_cap=4),
    "fwd_packets_events_cap0": lambda e: e.ode23_packets([0.0, w.dt], w.dt, events=EVENTS, ev_cap=0),
    "fwd_tspans_events_cap0": lambda e: e.ode23_packets_tspans_events(fwd_rows, w.dt, EVENTS, ev_cap=0),
    "bwd_tspans_events_cap0": lambda e: e.ode23_packets_tspans_events(bwd_rows, w.dt, EVENTS, ev_cap=0),
}
KEYS = ("steps", "rejected", "status", "t_end")


def solve(e, call):
    e.set_packets(w.x, w.y, w.k, w.l)
    e.synchronize()
    t0 = time.perf_counter()
    st = call(e)
    e.synchronize()
    return 1e3 * (time.perf_counter() - t0), st


rows = []
for name, mode in (("LAGRANGE6", S.MODE_LAGRANGE6), ("NUFFT", S.MODE_NUFFT)):
    e = S.Engine(w.nx, w.L, w.f, w.gH, mode)
    e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
    for call in CASES.values():                          # warm-up: grids, module loads, per-packet and event state
        solve(e, call)
    ms = {k: [] for k in CASES}
    st = {}
    for _ in range(reps):                                # alternate the solves
        for k, call in CASES.items():
            t, st[k] = solve(e, call)
            ms[k].append(t)
    a, b = st["fwd_packets_events"], st["fwd_tspans_events"]
    fwd_equal = all(np.array_equal(a[k], b[k], equal_nan=True) for k in KEYS + ("te", "ye", "ie", "ne"))
    solve_equal = all(np.array_equal(st[d + "_tspans"][k], st[d + "_tspans_events"][k]) for d in ("fwd", "bwd") for k in KEYS)
    row = {"mode": name, "n": n, "forward_records_equal_packets_events": bool(fwd_equal),
           "solves_equal_tspans": bool(solve_equal), "ms": ms}
    for k in CASES:
        r = row[k] = {"median_ms": float(np.median(ms[k])), "min_ms": float(min(ms[k])), "max_ms": float(max(ms[k])),
                      "rounds": int((st[k]["steps"] + st[k]["rejected"]).max()), "accepted": int(st[k]["nsteps"]),
                      "events": int(st[k].get("events", 0))}
        print(f"C3 256^2, {n} packets, {name:9s} {k:23s}: median {r['median_ms']:8.2f} ms (min {r['min_ms']:.2f}, max "
              f"{r['max_ms']:.2f}), {r['rounds']} rounds, {r['accepted']} accepted packet-steps, {r['events']} events")
    print(f"  forward records equal swrt_ode23_packets_events': {fwd_equal}; solves equal swrt_ode23_packets_tspans': "
          f"{solve_equal}")
    rows.append(row)
    e.close()
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as fh:
        json.dump({"device": gpu, "rows": rows}, fh, indent=1)
