"""Host controller (reference_api.ode23, two host waits per attempt) against the device controller (swrt_ode23, a few host
waits per solve) on the reference's unit of work: one ode23 solve over a QG step [0, dt] between two flow frames
(qgsw_raytrace.m:141-150), C3 flow (256^2).  The two controllers alternate in one process; the device name and power
limit are read in the same run.  With a second argument, the rows are also written to that JSON file.
    python tools/ode23_device_probe.py [reps [out.json]]"""
import json, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np
import swraytracing_b200 as S
from swraytracing_b200 import workloads as W, reference_api as R

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
print("device:", gpu)
MODES = (("SPECTRAL", S.MODE_SPECTRAL), ("LAGRANGE6", S.MODE_LAGRANGE6), ("NUFFT", S.MODE_NUFFT))


def solve_ms(e, w, host, reps):
    """median wall time of one solve (ending in a device synchronise), packets reset before each"""
    ts = []
    for _ in range(reps):
        e.set_packets(w.x, w.y, w.k, w.l)
        e.synchronize()
        t0 = time.perf_counter()
        st = R.ode23(e, [0.0, w.dt], w.dt) if host else e.ode23([0.0, w.dt], w.dt)
        e.synchronize()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts)), st


rows = []
for n, modes, r in ((50, MODES, reps), (1 << 20, MODES[1:], max(2, reps // 10))):
    w = W.make_workload("C3", n_packets=n)
    for name, mode in modes:
        e = S.Engine(w.nx, w.L, w.f, w.gH, mode)
        e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
        for host in (True, False):                       # warm-up: stacks, grids, module loads
            solve_ms(e, w, host, 1)
        res = {True: [], False: []}
        for _ in range(3):                               # alternate the controllers
            for host in (True, False):
                ms, st = solve_ms(e, w, host, r)
                res[host].append(ms)
        row = {"n": n, "mode": name, "nsteps": st["nsteps"], "nfailed": st["nfailed"], "host_waits": st["host_waits"],
               "host_ms": float(np.median(res[True])), "device_ms": float(np.median(res[False])),
               "host_ms_all": res[True], "device_ms_all": res[False]}
        rows.append(row)
        print(f"C3 flow, {n:8d} packets, {name:9s}: host controller {row['host_ms']:8.3f} ms, device controller "
              f"{row['device_ms']:8.3f} ms per solve ({row['nsteps']} steps, {row['nfailed']} rejected, "
              f"{row['host_waits']} host waits)  ratio {row['host_ms'] / row['device_ms']:.2f}")
        e.close()
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as fh:
        json.dump({"device": gpu, "rows": rows}, fh, indent=1)
