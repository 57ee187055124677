"""swrt_ode23 (one controller for the ensemble) against swrt_ode23_packets (one controller per packet) on the reference's
unit of work: one ode23 solve over a QG step [0, dt] between two flow frames (qgsw_raytrace.m:141-150), C3 flow (256^2).
The two solves alternate in one process; the wall time of a solve ends in a device synchronise and is the median of the
repeats.  The device name and power limit are read in the same run.  With a second argument, the rows are also written
to that JSON file.
    python tools/ode23_packets_probe.py [reps [out.json]]"""
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


def solve_ms(e, w, per_packet, reps):
    ts = []
    for _ in range(reps):
        e.set_packets(w.x, w.y, w.k, w.l)
        e.synchronize()
        t0 = time.perf_counter()
        st = e.ode23_packets([0.0, w.dt], w.dt) if per_packet else e.ode23([0.0, w.dt], w.dt)
        e.synchronize()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts)), st


rows = []
for n, modes, r in ((50, MODES, reps), (1 << 20, MODES[1:], max(2, reps // 10))):
    w = W.make_workload("C3", n_packets=n)
    for name, mode in modes:
        e = S.Engine(w.nx, w.L, w.f, w.gH, mode)
        e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
        for pp in (False, True):                         # warm-up: stacks, grids, module loads, per-packet state
            solve_ms(e, w, pp, 1)
        res = {False: [], True: []}
        for _ in range(3):                               # alternate the two solves
            for pp in (False, True):
                ms, st = solve_ms(e, w, pp, r)
                res[pp].append(ms)
                if pp:
                    stp = st
                else:
                    stc = st
        steps = stp["steps"] + stp["rejected"]
        row = {"n": n, "mode": name, "coupled_steps": stc["nsteps"], "coupled_rejected": stc["nfailed"],
               "packet_attempts_max": int(steps.max()), "packet_attempts_mean": float(steps.mean()),
               "packets_host_waits": stp["host_waits"], "coupled_ms": float(np.median(res[False])),
               "packets_ms": float(np.median(res[True])), "coupled_ms_all": res[False], "packets_ms_all": res[True]}
        rows.append(row)
        print(f"C3 flow, {n:8d} packets, {name:9s}: swrt_ode23 {row['coupled_ms']:8.3f} ms ({row['coupled_steps']} steps, "
              f"{row['coupled_rejected']} rejected), swrt_ode23_packets {row['packets_ms']:8.3f} ms (attempts per packet: "
              f"max {row['packet_attempts_max']}, mean {row['packet_attempts_mean']:.2f}; {row['packets_host_waits']} host "
              f"waits)  ratio {row['packets_ms'] / row['coupled_ms']:.2f}")
        e.close()
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as fh:
        json.dump({"device": gpu, "rows": rows}, fh, indent=1)
