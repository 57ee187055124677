"""swrt_ode23_packets (one shared tspan) against swrt_ode23_packets_tspans (a tspan row per packet) on the reference's unit
of work: one ode23 solve per packet over a QG step [0, dt] between two flow frames, C3 flow (256^2), 1M packets.
  shared:    every row [0, dt], so both solves take the same steps; the two alternate in one process, and the spread of
             the repeats is reported beside the medians.
  staggered: staggered release, packet i over [tau_i, dt] with tau_i uniform in [0, dt/2].  Its step counts differ from
             the shared solve, so it is reported per round (the slowest packet's attempts) and per accepted packet-step.
The wall time of a solve ends in a device synchronise.  The device name and power limit are read in the same run.
    python tools/ode23_tspans_probe.py [reps [out.json]]"""
import json, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np
import swraytracing_b200 as S
from swraytracing_b200 import workloads as W

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
print("device:", gpu)
n = 1 << 20
w = W.make_workload("C3", n_packets=n)
shared_rows = np.repeat(np.array([[0.0], [w.dt]]), n, axis=1)
tau = np.random.RandomState(1).uniform(0.0, 0.5 * w.dt, n)
staggered_rows = np.stack([tau, np.full(n, w.dt)])
CASES = {"packets": [0.0, w.dt], "tspans_shared": shared_rows, "tspans_staggered": staggered_rows}


def solve(e, tspan):
    e.set_packets(w.x, w.y, w.k, w.l)
    e.synchronize()
    t0 = time.perf_counter()
    st = e.ode23_packets(tspan, w.dt)
    e.synchronize()
    return 1e3 * (time.perf_counter() - t0), st


rows = []
for name, mode in (("LAGRANGE6", S.MODE_LAGRANGE6), ("NUFFT", S.MODE_NUFFT)):
    e = S.Engine(w.nx, w.L, w.f, w.gH, mode)
    e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
    for ts in CASES.values():                            # warm-up: grids, module loads, per-packet state
        solve(e, ts)
    ms = {k: [] for k in CASES}
    st = {}
    for _ in range(reps):                                # alternate the solves
        for k, ts in CASES.items():
            t, st[k] = solve(e, ts)
            ms[k].append(t)
    a, b = st["packets"], st["tspans_shared"]
    same = all(np.array_equal(a[k], b[k]) for k in ("steps", "rejected", "status", "t_end"))
    row = {"mode": name, "n": n, "results_equal": bool(same), "ms": ms}
    for k in CASES:
        rounds = int((st[k]["steps"] + st[k]["rejected"]).max())
        row[k] = {"median_ms": float(np.median(ms[k])), "min_ms": float(min(ms[k])), "max_ms": float(max(ms[k])),
                  "rounds": rounds, "accepted": int(st[k]["nsteps"]), "host_waits": int(st[k]["host_waits"]),
                  "ms_per_round": float(np.median(ms[k])) / rounds,
                  "ns_per_accepted_packet_step": 1e6 * float(np.median(ms[k])) / int(st[k]["nsteps"])}
        r = row[k]
        print(f"C3 256^2, {n} packets, {name:9s} {k:17s}: median {r['median_ms']:8.2f} ms (min {r['min_ms']:.2f}, max "
              f"{r['max_ms']:.2f}), {r['rounds']} rounds, {r['ms_per_round']:.3f} ms/round, "
              f"{r['ns_per_accepted_packet_step']:.3f} ns/accepted packet-step, {r['host_waits']} host waits")
    print(f"  shared rows give the swrt_ode23_packets result: {same}")
    rows.append(row)
    e.close()
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as fh:
        json.dump({"device": gpu, "rows": rows}, fh, indent=1)
