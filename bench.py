#!/usr/bin/env python
"""bench.py -- packet-steps/sec of the SWRaytracing hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--single-process] [--dump-outputs DIR]

HEADLINE (value, e2e, roofline of the one JSON line) = BASELINE.json configs[3], the configuration its target sentence is
quoted on: **C4** -- two-layer-type flow on a 512^2 spectral grid (L = 20, mean shear), two stored frames blended on the
device, **16,777,216 packets in total, split N ways** (``"scaling": "strong"``), SPECTRAL mode (the dense fp64 DMMA
contraction north_star names).  One bench "step" = ``substeps`` leapfrog sub-steps of one flow step
(ode_symplectic.m:33-37 with the time-centred frame blend alpha_j = (j + 1/2)/m) in ONE packet-kernel launch, followed by
the omega histogram (the diagnostic the multi-GPU path all-reduces).  The other GPU configs -- C2 (steady 128^2, 65,536
packets), C3 (256^2 two-frame, 1,048,576 packets in total, strong) and C5 (step_packet_xka, 4,194,304 packets) -- are
timed in the same run with fewer steps and reported under ``"configs"``, each with value / e2e / roofline.

Keys (task contract): value = device-resident throughput (CUDA events on the handle's stream, L2 flushed between timed
steps, max over ranks); e2e = the same through ONE C-ABI call with HOST buffers (``swrt_step_host``: upload, steps and
download inside the timed region), measured with pinned AND with ordinary pageable buffers (``e2e.pageable``);
roofline = executed DMMA flops of the dominant kernel / its event-timed duration against the fp64 peak MEASURED IN THIS
RUN (torch.matmul fp64 8192^3, best of 5); gather modes are reported against a gather-rate probe measured in this run
(``bound: "l2"``); cpu_baseline = the oracle's C port of the reference's own path (two-frame 6x6 Lagrange leapfrog) on the
host cores.  ``--impl reference`` times that CPU port alone on the same config.

``--single-process``: the N GPUs are driven by ONE process through a multi-device handle (swrt_params.ngpu = N, in-library
sharding + NCCL) instead of one torchrun rank per GPU.

``--dump-outputs DIR``: after the timed steps, the headline's packet state and omega histogram as left by its last timed
step go to DIR/*.npy.  Inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "packet-steps/sec (spectral U,gradU eval + symplectic step)"
UNIT = "packet-steps/s"
# cross-checks only (round-1 measurements on this pool); the denominators used are measured in the run
FP64_DGEMM_TFLOPS_R01 = 35.5
FP64_DMMA_TFLOPS = 37.1      # DMMA m8n8k4 issue-rate ceiling (tools/fp64_peak.cu)
SUBSTEPS = {"C1": 16, "C2": 16, "C3": 16, "C4": 2, "C5": 2}
DESCR = {
    "C2": "C2: steady 128^2 spectral grid, 65,536 packets, leapfrog (symplectic_full_fourier.m)",
    "C3": "C3: time-dependent 256^2 spectral grid, two-frame blend, 1,048,576 packets in total, leapfrog (qgsw_raytrace.m)",
    "C4": "C4: two-layer-type flow on a 512^2 spectral grid (L = 20, mean shear), two-frame blend, 16,777,216 packets in total, leapfrog (qg2layersw_raytrace.m)",
    "C5": "C5: step_packet_xka (wave action, refraction by H) on a synthetic geostrophic 256^2 state, 4,194,304 packets (raytrace_sw.m)",
}
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch from the committed ncu --set full captures
# (tools/r02h_traffic.sh at the bench's own launch shapes: profiles/r02h_spec512_c4_fullsize_ncu_summary.json, r02h_traffic.csv);
# key = (workload, fused sub-steps, packets of this process); other shapes report null
NCU_TRAFFIC_BYTES = {("C4", 2, 16777216): 596984832 + 561957888,     # 1.16 GB = 1.08 x (64 B of packet state per packet + stacks)
                     ("C3", 16, 1048576): 60381696 + 13184256,
                     ("C5", 2, 4194304): 186920448 + 154308352,
                     ("C2", 16, 65536): 2526464}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="swrt", choices=["swrt", "reference"])
    ap.add_argument("--workload", default="C4", help="headline workload (default C4, the configuration BASELINE.json's target is quoted on)")
    ap.add_argument("--packets", type=int, default=0, help="TOTAL packets of the headline workload (0 = the workload's own count)")
    ap.add_argument("--substeps", type=int, default=0, help="fused leapfrog sub-steps per bench step (0 = per-workload default)")
    ap.add_argument("--mtiles", type=int, default=0)
    ap.add_argument("--side-steps", type=int, default=5, help="timed steps of the side configs and side modes")
    ap.add_argument("--configs", default="C2,C3,C5", help="side configs reported under \"configs\" ('' = none)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-modes", action="store_true", help="skip the LAGRANGE6 / NUFFT legs of the headline workload")
    ap.add_argument("--single-process", action="store_true", help="drive --gpus N devices from this one process (multi-device handle)")
    ap.add_argument("--mode", default="spectral", choices=["spectral", "nufft", "lagrange6"],
                    help="evaluation mode of the HEADLINE legs (value, e2e, roofline); default = the dense DMMA contraction")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline's last timed step computed to DIR/<name>.npy (float64): the packet state "
                         f"x, y, k, l (a fixed, seeded sample of {DUMP_MAX_PACKETS} packets when there are more) and omega_hist")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "swrt":
        ap.error("--dump-outputs writes the GPU arm's outputs")
    if args.dump_outputs and not args.single_process and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs needs the whole ensemble in one process (use --single-process for several GPUs)")
    return args


TOTALS = {"C2": 65536, "C3": 1048576, "C4": 16777216, "C5": 4194304}
DUMP_MAX_PACKETS = 1 << 20          # 4 float64 arrays of this length = 32 MiB of --dump-outputs
DUMP_SEED = 0
GRID = {"C1": 64, "C2": 128, "C3": 256, "C4": 512, "C5": 256}
SCHEME = {"C5": "rk4_xka"}


def config_for(name, n_gpus, sub, packets_total=0):
    """the `config` object BOTH arms print, key for key (the driver compares them); what is specific to an arm -- evaluation
    mode, sharding, L2 policy -- goes under "arm" """
    return {"workload": DESCR.get(name, name), "name": name, "nx": GRID.get(name), "packets_total": packets_total or TOTALS.get(name),
            "scheme": SCHEME.get(name, "leapfrog"), "substeps_per_step": sub, "n_gpus": n_gpus,
            "field": "full-spectrum random-phase QG streamfunction (every (kx,ky) non-zero)", "histogram_bins": 299}


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], None, set(), []
        note = None
        if not self.rows:
            # the timed regions were shorter than nvidia-smi's start-up + sampling period: one sample right after them
            try:
                one = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().splitlines()
                self.rows = [[c.strip() for c in one[0].split(",")]] if one else []
                note = "timed regions shorter than the sampling period: one sample taken right after them"
            except Exception:
                pass
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1]); power.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        # "under load" = the samples drawing more than half the maximum power seen (idle samples between legs excluded)
        load = [s for s, p in zip(sm, power) if power and p >= 0.5 * max(power)] or sm
        out = {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
               "sm_mhz_min": float(min(load)) if load else None, "power_w_max": max(power) if power else None}
        if note:
            out["note"] = note
        return out


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle port; the only places bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------
_CPU_CACHE = {}


def _cpu_setup(w):
    from oracle import c_oracle as CO
    from swraytracing_b200 import workloads as W
    key = (w.name, w.nx)
    if key not in _CPU_CACHE:
        frames = []
        for psik in (w.psik, w.psik2):
            if psik is None:
                continue
            planes = W.planes_from_psik(psik, w.L, w.u_mean)
            frames.append(CO.prepare_grids([W._fulspec_ifft(p) for p in planes]))   # gridded planes (what grid_U / SpectralScheme build)
        _CPU_CACHE[key] = frames
    return _CPU_CACHE[key]


def _use_all_host_threads(CO):
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0 alone and is meant to use every host
    core this process may run on, so the thread count is set explicitly (an OMP_NUM_THREADS the USER chose is kept)."""
    if os.environ.get("SWRT_CPU_THREADS"):
        CO.set_threads(int(os.environ["SWRT_CPU_THREADS"]))
    elif "TORCHELASTIC_RUN_ID" in os.environ or "OMP_NUM_THREADS" not in os.environ:
        try:
            CO.set_threads(len(os.sched_getaffinity(0)))
        except AttributeError:
            CO.set_threads(os.cpu_count() or 1)


def cpu_reference_rate(w, sub, target_s=12.0):
    """packet-steps/s of the reference's own path -- ode_symplectic leapfrog with 6x6 Lagrange interpolation of the six
    gridded planes (SpectralScheme.m:45-68, interpolate.m), both stored frames interpolated and blended as interpolate_U.m
    does when the flow is time-dependent -- restated in C (oracle/swrt_oracle.c), all host threads.  Bounded sample of
    ~target_s on the first 65,536 packets of the workload."""
    import ctypes as C
    from oracle import c_oracle as CO
    _use_all_host_threads(CO)
    frames = _cpu_setup(w)
    n = min(w.n_packets, 65536)
    x, y, k, l = (np.ascontiguousarray(a[:n]).copy() for a in (w.x, w.y, w.k, w.l))
    lib = CO.lib()
    two = len(frames) == 2

    def run(nsteps):
        # `nsteps` leapfrog steps in place, as whole flow steps of `sub` sub-steps each
        args = [CO._p(x), CO._p(y), CO._p(k), CO._p(l), C.c_int64(n)]
        t0 = time.perf_counter()
        if two:
            for _ in range(nsteps // sub):
                lib.orc_leapfrog_lagrange2(*args, CO._table(frames[0]), CO._table(frames[1]), C.c_int(w.nx), C.c_double(w.dx), C.c_double(1e-13),
                                           C.c_double(w.f), C.c_double(w.gH), C.c_double(w.dt / sub), C.c_int(sub), C.c_double(0.5 / sub), C.c_double(1.0 / sub))
        else:
            lib.orc_leapfrog_lagrange(*args, CO._table(frames[0]), C.c_int(w.nx), C.c_double(w.dx), C.c_double(1e-13), C.c_double(w.f),
                                      C.c_double(w.gH), C.c_double(w.dt / sub if two else w.dt), C.c_int(nsteps))
        return time.perf_counter() - t0

    t1 = run(sub)                                          # calibration (also warms caches)
    reps = min(4000, max(1, int(target_s / max(t1, 1e-4))))
    el = run(sub * reps)
    what = "two-frame blend (interpolate_U.m), " if two else ""
    return n * sub * reps / el, CO.num_threads(), (f"{n} packets x {sub * reps} leapfrog steps of {w.name} ({el:.1f} s), {what}"
                                                    "6x6 Lagrange (reference semantics), C port + OpenMP")


def cpu_spectral_rate(w, target_s=8.0):
    """the dense Fourier-sum evaluation (what the GPU arm computes) as a C port on the host cores"""
    from oracle import c_oracle as CO
    from swraytracing_b200 import workloads as W
    planes = W.planes_from_psik(w.psik, w.L)
    n = 2048 if w.nx <= 256 else 512
    x, y, k, l = (a[:n].copy() for a in (w.x, w.y, w.k, w.l))
    t0 = time.perf_counter()
    CO.leapfrog_spectral(x, y, k, l, planes, w.dx, w.nx, w.f, w.gH, w.dt, 1, precise=False)
    t1 = time.perf_counter() - t0
    reps = max(1, min(64, int(target_s / max(t1, 1e-3))))
    t0 = time.perf_counter()
    CO.leapfrog_spectral(x, y, k, l, planes, w.dx, w.nx, w.f, w.gH, w.dt, reps, precise=False)
    el = time.perf_counter() - t0
    return n * reps / el, CO.num_threads(), f"{n} packets x {reps} leapfrog steps, dense trig sum in double, C port + OpenMP ({el:.1f} s)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from swraytracing_b200 import workloads as W
    sub = args.substeps or SUBSTEPS.get(args.workload, 16)
    w = W.make_workload(args.workload, n_packets=min(65536, args.packets) if args.packets else 65536)   # the CPU sample: the first 65,536 packets
    vals = []
    t_each = max(1.0, min(10.0, 150.0 / max(1, args.steps + args.warmup)))
    if os.environ.get("SWRT_BENCH_TARGET_S"):            # test hook: a shorter CPU sample per step
        t_each = float(os.environ["SWRT_BENCH_TARGET_S"])
    threads, sample = 1, ""
    for _ in range(args.warmup):
        cpu_reference_rate(w, sub, target_s=t_each)
    for _ in range(args.steps):
        v, threads, sample = cpu_reference_rate(w, sub, target_s=t_each)
        vals.append(v)
    value = float(np.median(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": config_for(args.workload, args.gpus, sub, args.packets),
            "arm": {"impl": "C port of the reference's own path (oracle/swrt_oracle.c), OpenMP", "sample_packets": w.n_packets},
            "note": "the reference's own CPU path (gridded planes + 6x6 Lagrange interpolate, both frames blended) restated in C with OpenMP; "
                    "the MATLAB original cannot run here (it sustains ~1e3 packet-steps/s, SURVEY.md 6).  Host-side throughput is "
                    "independent of the GPU count.",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    _emit(line)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
_JSON_FD = None


def _claim_stdout():
    """Keep stdout for the ONE JSON line: everything else that writes to fd 1 (NCCL prints its version banner there, library
    chatter) is sent to stderr from here on."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


class Ctx:
    """process topology of this run"""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.args = args
        self.single = bool(args.single_process)
        self.world = 1 if self.single else int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = 0 if self.single else int(os.environ.get("RANK", "0"))
        self.local = 0 if self.single else int(os.environ.get("LOCAL_RANK", "0"))
        self.ngpu_handle = args.gpus if self.single else 1          # devices behind ONE handle
        self.n_gpus = args.gpus if self.single else self.world      # GPUs working on the job
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault("NCCL_DEBUG", "WARN")        # NCCL otherwise prints its version banner on stdout, next to the JSON line
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        # > 126 MB L2, on every device this process drives
        self.flush = [torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=torch.device("cuda", self.local + i))
                      for i in range(self.ngpu_handle)]

    def flush_l2(self, i):
        for f in self.flush:
            f.fill_(i & 0xFF)
        for d in range(self.ngpu_handle):
            self.torch.cuda.synchronize(self.local + d)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        for d in range(self.ngpu_handle):
            self.torch.cuda.synchronize(self.local + d)

    def max_over_ranks(self, v):
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, ok):
        if self.dist is None:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())


def measure_fp64_peak(ctx):
    """fp64 matmul 8192^3 on this device, best of 5, timed with CUDA events -> TFLOP/s (the tensor roofline denominator)"""
    torch = ctx.torch
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    c = torch.empty(n, n, dtype=torch.float64, device="cuda")
    sampler = ClockSampler(ctx.local).start()
    torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b, out=c); e1.record(); e1.synchronize()
        best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) * 1e-12)
    clk = sampler.stop()
    del a, b, c
    torch.cuda.empty_cache()
    return best, clk


def make_engine(S, W, w, mode, ctx, mtiles=0):
    eng = S.Engine(w.nx, w.L, w.f, w.gH, mode, device=ctx.local, ngpu=ctx.ngpu_handle)
    eng.set_tuning(mtiles)
    if w.scheme == "rk4_xka":
        eng.set_flow_planes_spectral(W.planes_from_psik(w.psik, w.L, w.u_mean, etak=w.extra["etak"]), slot=0)
    else:
        eng.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
        if w.psik2 is not None:
            eng.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
    return eng


def measure(ctx, name, total_packets, sub, steps, warmup, mode_name, peaks, headline=False, dump=False):
    """time one workload on this process's shard: device-resident `value`, end-to-end `e2e` (pinned + pageable host buffers
    through swrt_step_host), the dominant kernel's roofline.  Returns the dict that goes into the JSON line; with `dump`,
    also (under "_outputs") what the last timed device-resident step left: packet state and omega histogram."""
    import swraytracing_b200 as S
    from swraytracing_b200 import workloads as W
    from swraytracing_b200.distributed import ShardedEnsemble, shard_range
    torch, args = ctx.torch, ctx.args
    weak = (name == "C2" and not total_packets)                 # C2 is BASELINE's one-GPU case: 65,536 packets PER GPU when N > 1
    w = W.make_workload(name, n_packets=(65536 * ctx.n_gpus if weak else total_packets) or None)
    n_total = w.n_packets
    lo, hi = shard_range(n_total, ctx.rank, ctx.world)          # this rank's contiguous shard of the job's packets
    n = hi - lo
    xs, ys, ks, ls = (np.ascontiguousarray(a[lo:hi]) for a in (w.x, w.y, w.k, w.l))
    mode = {"spectral": S.MODE_SPECTRAL, "nufft": S.MODE_NUFFT, "lagrange6": S.MODE_LAGRANGE6}[mode_name]
    eng = make_engine(S, W, w, mode, ctx, args.mtiles)
    time_dependent = w.psik2 is not None
    scheme = {"leapfrog": S.SCHEME_LEAPFROG, "rk4_packet": S.SCHEME_RK4_PACKET, "rk4_xka": S.SCHEME_RK4_XKA}[w.scheme]
    a0, da = (0.5 / sub, 1.0 / sub) if time_dependent else (0.0, 0.0)     # time-centred alpha_j = (j + 1/2)/m (SURVEY 7.0)
    dt_sub = w.dt / sub if time_dependent else w.dt                       # m sub-steps span ONE flow step of the two-frame configs
    om_max = float(np.sqrt(w.f ** 2 + w.gH * 4 * (w.k ** 2 + w.l ** 2).max()))
    edges = np.linspace(0.0, om_max, 300)            # 299 bins (analysis/load_data.m:38-39)
    ens = ShardedEnsemble(eng, n_total, ctx.rank, ctx.world, ctx.dist, device=torch.device("cuda", ctx.local))
    pipe = ens.hist_pipeline(edges) if not ctx.single else None
    last_counts = [None]

    def one_step_resident():
        """one bench step = the fused packet kernel + the omega histogram of the new state.  Under torchrun the histogram's
        all-reduce (the path's only collective) is pipelined one step behind (distributed.HistPipeline); a multi-device
        handle reduces inside libswrt (NCCL, stream-ordered) and hands back the global counts."""
        eng.step_async(scheme, dt_sub, sub, a0, da)  # queue the packet kernel(s), do not wait
        if pipe is not None:
            done = pipe.rotate()                     # host work under the running kernel
            pipe.launch()
            if done is not None:
                last_counts[0] = done
        else:
            last_counts[0] = eng.hist_omega(edges)

    # ---- device-resident leg: `value` ----
    eng.set_packets(xs, ys, ks, ls)
    for _ in range(max(3, warmup)):
        one_step_resident()
    if pipe is not None:
        pipe.drain()
    ctx.barrier()
    sampler = ClockSampler(ctx.local).start() if (ctx.rank == 0 and headline) else None
    eng.launch_count(reset=True)
    step_ms = []
    t_wall0 = time.perf_counter()
    for i in range(steps):
        ctx.flush_l2(i)                                              # flush L2 between timed iterations
        eng.timer_start()
        one_step_resident()
        step_ms.append(eng.timer_stop())
    t0 = time.perf_counter()
    if pipe is not None:
        last_counts[0] = pipe.drain()[-1]                            # the pipeline's tail is not hidden: add its exposed wait
    eng.synchronize()
    step_ms[-1] += (time.perf_counter() - t0) * 1e3
    ctx.barrier()
    wall = time.perf_counter() - t_wall0
    launches = eng.launch_count()
    total_ms = ctx.max_over_ranks(float(np.sum(step_ms)))
    value = n_total * sub * steps / (total_ms * 1e-3)
    hist_total = int(np.asarray(last_counts[0]).sum())
    outputs = None
    if dump:
        # read before the legs below step the same packets further
        state = eng.get_packets()
        if n > DUMP_MAX_PACKETS:
            pick = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MAX_PACKETS, replace=False))
            state = [a[pick] for a in state]
        outputs = dict(zip("xykl", state), omega_hist=np.asarray(last_counts[0], dtype=np.float64))

    # dominant-kernel time: re-time the packet kernel(s) alone with the handle's own event pair
    k_ms, nl = [], 1
    for i in range(min(steps, 5)):
        ctx.flush_l2(i)
        eng.step(scheme, dt_sub, sub, a0, da)
        ms, nl = eng.last_kernel_ms()
        k_ms.append(ms)
    kernel_ms = float(np.mean(k_ms))

    # ---- e2e leg: host buffers through ONE C-ABI call (swrt_step_host), pinned and pageable ----
    def e2e_leg(src, dst, nsteps_e2e):
        for _ in range(2):
            eng.step_host(scheme, dt_sub, sub, *src, alpha0=a0, dalpha=da, out=dst)
        ctx.barrier()
        ms = []
        for i in range(nsteps_e2e):
            ctx.flush_l2(i)
            t0 = time.perf_counter()
            eng.step_host(scheme, dt_sub, sub, *src, alpha0=a0, dalpha=da, out=dst)
            ms.append((time.perf_counter() - t0) * 1e3)             # host clock: the call returns when the download is complete
        tot = ctx.max_over_ranks(float(np.sum(ms)))
        return n_total * sub * nsteps_e2e / (tot * 1e-3), tot / nsteps_e2e

    pin_t = [torch.from_numpy(a.copy()).pin_memory() for a in (xs, ys, ks, ls)]
    out_t = [torch.empty(n, dtype=torch.float64).pin_memory() for _ in range(4)]
    e2e_value, e2e_ms = e2e_leg([p.numpy() for p in pin_t], [p.numpy() for p in out_t], steps)
    del pin_t, out_t
    page_src = [a.copy() for a in (xs, ys, ks, ls)]                  # ordinary malloc'ed numpy arrays: what a MEX / ctypes caller hands over
    page_dst = [np.empty(n) for _ in range(4)]
    e2e_page_value, e2e_page_ms = e2e_leg(page_src, page_dst, min(steps, max(3, args.side_steps)))
    clocks = sampler.stop() if sampler else None       # sampled across the resident, kernel-only and e2e timed regions

    # ---- sharding check: this rank's first packets recomputed at a DIFFERENT position of a fresh one-device ensemble ----
    shard_ok = None
    if ctx.n_gpus > 1 and headline:
        m = min(n, 65536)
        eng.set_packets(xs, ys, ks, ls)
        eng.step(scheme, dt_sub, sub, a0, da)
        mine = np.stack(eng.get_packets())[:, :m]
        saved = ctx.ngpu_handle
        ctx.ngpu_handle = 1
        fresh = make_engine(S, W, w, mode, ctx, args.mtiles)
        ctx.ngpu_handle = saved
        pad = 37                                                     # shifts every packet to another tile / lane
        z = np.zeros(pad)
        fresh.set_packets(np.concatenate([z, xs[:m]]), np.concatenate([z, ys[:m]]), np.concatenate([z + 1.0, ks[:m]]), np.concatenate([z, ls[:m]]))
        fresh.step(scheme, dt_sub, sub, a0, da)
        ref = np.stack(fresh.get_packets())[:, pad:]
        fresh.close()
        shard_ok = ctx.all_true(np.array_equal(mine, ref))

    # ---- roofline of the dominant kernel ----
    if mode_name == "spectral":
        ncontract = eng.contracted_planes()                         # 3: psi-hat moments (6 nx^2 flops); 6: six planes (12 nx^2)
        # plane-evaluations contracted per packet-step: leapfrog = one six-plane evaluation (3 moment planes when
        # the flow is psi-hat); step_packet = six planes + 3 x (u,v); step_packet_xka = 4 x (u,v,H) + seven planes
        plane_evals = {"leapfrog": ncontract, "rk4_packet": ncontract + 6, "rk4_xka": 19}[w.scheme]
        flops_per_packet_step = eng.work_per_eval(plane_evals)      # EXECUTED DMMA flops per packet-step (+-kx folded)
        n_dev = -(-n // ctx.ngpu_handle)                            # packets behind the slowest device of this handle
        flops_per_launch = flops_per_packet_step * n_dev * sub
        achieved = flops_per_launch / (kernel_ms * 1e-3) * 1e-12
        peak = peaks["fp64_tflops"]
        tw = {0: "twiddle-rotation", 1: "twiddle-table(smem)", 2: "twiddle-table(L2)"}[S.engine.spectral_geometry(w.nx, ncontract, 1)["twiddle_table"]]
        inst = (f"swrt::spectral_kernel<{ncontract},{24 // ncontract},1,LEAPFROG,{'psi' if ncontract == 3 else 'planes'},{tw}>" if w.scheme == "leapfrog" else
                f"swrt::spectral_rk4_kernel<{'xka' if w.scheme == 'rk4_xka' else 'packet'},{'psi' if (ncontract == 3 and w.scheme != 'rk4_xka') else 'planes'},"
                f"{'twiddle-table(smem)' if w.nx <= 128 else 'twiddle-table(L2)'}> (fused: 5 contractions + RK4 update per step)")
        roofline = {"bound": "tensor", "achieved": round(achieved, 3), "peak": round(peak, 3), "unit": "TFLOP/s",
                    "frac": round(achieved / peak, 4), "traffic": NCU_TRAFFIC_BYTES.get((name, sub, n)),
                    "kernel": inst + " (fp64 DMMA m8n8k4)", "kernel_ms": round(kernel_ms, 4), "kernel_launches_per_step": nl,
                    "contracted_planes": ncontract, "flops_per_packet_step": flops_per_packet_step,
                    "algorithmic_flops_per_launch": flops_per_launch,
                    "peak_source": "measured in this run: torch.matmul fp64 8192^3 (cuBLAS DGEMM), best of 5, CUDA events; "
                                   f"round-1 measurement on this pool {FP64_DGEMM_TFLOPS_R01}; MEASURED_PEAKS.json has no fp64 entry",
                    "frac_of_dmma_issue_peak": round(achieved / FP64_DMMA_TFLOPS, 4),
                    "hbm_bytes_per_packet_step": 64.0 / sub}
    else:
        # gather modes: algorithmic bytes = stencil-node bytes gathered per evaluation x evaluations per launch, served from an
        # L2-resident table through L1TEX; the denominator is the scattered-gather rate measured in this run (swrt_gather_probe)
        evals = {"leapfrog": 1, "rk4_packet": 4 if mode_name == "nufft" else 5, "rk4_xka": 5 if mode_name == "nufft" else 19 / 6}[w.scheme]
        frames = 2 if (time_dependent and mode_name == "lagrange6") else 1      # the exact two-frame leapfrog gathers both frames
        npl_node = 7 if (w.scheme == "rk4_xka" and mode_name == "nufft") else 6     # NUFFT flows that carry H gather 32-byte (u,v,H,0) nodes
        per_ps = eng.work_per_eval(npl_node) * evals * frames
        n_dev = -(-n // ctx.ngpu_handle)
        ach = per_ps * n_dev * sub / (kernel_ms * 1e-3) * 1e-9
        kname = {("nufft", "leapfrog"): "swrt::nufft_leapfrog_kernel", ("nufft", "rk4_packet"): "swrt::nufft_rk4_kernel<false>",
                 ("nufft", "rk4_xka"): "swrt::nufft_rk4_kernel<true>", ("lagrange6", "leapfrog"): f"swrt::lagrange_leapfrog_kernel<6,{'true' if frames == 2 else 'false'}>",
                 ("lagrange6", "rk4_packet"): "swrt::lagrange_rk4_kernel<6,false>", ("lagrange6", "rk4_xka"): "swrt::lagrange_rk4_kernel<7,true>"}[(mode_name, w.scheme)]
        roofline = {"bound": "l2", "achieved": round(ach, 1), "peak": round(peaks["gather_gbs"], 1), "unit": "GB/s",
                    "frac": round(ach / peaks["gather_gbs"], 4), "traffic": None, "kernel": kname, "kernel_ms": round(kernel_ms, 4),
                    "kernel_launches_per_step": nl, "gathered_bytes_per_packet_step": per_ps,
                    "peak_source": "measured in this run: swrt_gather_probe (scattered 64-byte segments of a 16 MiB L2-resident table, "
                                   "quad of lanes per segment, 8 loads in flight per lane)",
                    "hbm_bytes_per_packet_step": 64.0 / sub}

    res = {"value": value, "unit": UNIT, "ms_per_step": total_ms / steps, "steps": steps, "scaling": "weak" if weak else "strong",
           "config": config_for(name, ctx.n_gpus, sub, 0 if weak else n_total),
           "arm": {"mode": mode_name.upper(), "packets_this_run": n_total, "packets_per_gpu": -(-n_total // ctx.n_gpus),
                   "l2": "flushed between timed steps (256 MiB write per device)"},
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * 8 * n, "d2h_bytes_per_step": 4 * 8 * n, "ms_per_step": e2e_ms,
                   "host_buffers": "pinned", "call": "swrt_step_host (one C-ABI call: upload, steps, download)",
                   "pageable": {"value": e2e_page_value, "unit": UNIT, "ms_per_step": e2e_page_ms,
                                "host_buffers": "pageable (ordinary numpy / mxArray memory), staged through libswrt's pinned ring"},
                   "frac_of_resident": round(e2e_value / value, 4), "pageable_frac_of_resident": round(e2e_page_value / value, 4)},
           "gpu_launches": int(launches), "roofline": roofline, "histogram_total": hist_total,
           "wall_s_timed_region": round(wall, 3)}
    if clocks:
        res["clocks"] = clocks
    if shard_ok is not None:
        res["shard_bit_identical"] = shard_ok
    res["_w"] = w
    res["_sub"] = sub
    res["_outputs"] = outputs
    eng.close()
    return res


def side_mode(ctx, name, total_packets, sub, steps, mode_name, peaks):
    r = measure(ctx, name, total_packets, sub, steps, 3, mode_name, peaks)
    return {"value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "e2e": r["e2e"], "roofline": r["roofline"],
            "gpu_launches": r["gpu_launches"]}


def main():
    args = parse()
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the swrt arm has no CPU fallback (use --impl reference for the CPU port)")
    import swraytracing_b200 as S
    ctx = Ctx(args)
    rank = ctx.rank

    # ---- roofline denominators, measured in this run (rank 0's device; the other ranks idle at the barrier) ----
    peaks = {"fp64_tflops": FP64_DGEMM_TFLOPS_R01, "gather_gbs": 0.0}
    peak_clk = None
    if rank == 0:
        peaks["fp64_tflops"], peak_clk = measure_fp64_peak(ctx)
        peaks["gather_gbs"] = S.engine.gather_probe(1 << 24, 5, ctx.local)
    if ctx.dist is not None:
        t = torch.tensor([peaks["fp64_tflops"], peaks["gather_gbs"]], dtype=torch.float64, device="cuda")
        ctx.dist.broadcast(t, 0)
        peaks["fp64_tflops"], peaks["gather_gbs"] = float(t[0]), float(t[1])
    ctx.barrier()

    name = args.workload
    sub = args.substeps or SUBSTEPS.get(name, 16)
    head = measure(ctx, name, args.packets, sub, args.steps, args.warmup, args.mode, peaks, headline=True, dump=bool(args.dump_outputs))
    w = head.pop("_w"); head.pop("_sub")
    outputs = head.pop("_outputs")
    if outputs is not None:
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for key, arr in outputs.items():
            np.save(out_dir / f"{key}.npy", arr)

    configs = {}
    for cname in [c for c in args.configs.split(",") if c and c != name]:
        r = measure(ctx, cname, 0, SUBSTEPS.get(cname, 16), args.side_steps, 3, args.mode, peaks)
        r.pop("_w"); r.pop("_sub"); r.pop("_outputs")
        configs[cname] = r

    side = {}
    if not args.no_side_modes:
        for mname in ("lagrange6", "nufft"):
            if mname != args.mode:
                side[mname] = side_mode(ctx, name, args.packets, sub, args.side_steps, mname, peaks)

    cpu = cpu_spec = None
    if rank == 0 and ctx.n_gpus == 1 and not args.no_cpu_baseline and w.scheme == "leapfrog":
        hook = os.environ.get("SWRT_BENCH_TARGET_S")             # test hook: a shorter CPU sample
        v, cores, sample = cpu_reference_rate(w, sub, **({"target_s": float(hook)} if hook else {}))
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
        v2, cores2, sample2 = cpu_spectral_rate(w, **({"target_s": float(hook)} if hook else {}))
        cpu_spec = {"value": v2, "unit": UNIT, "cores": cores2, "kind": "port", "sample": sample2}

    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": ctx.n_gpus, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": head["config"],
                "arm": dict(head["arm"], parallelism=(f"one process, multi-device handle (ngpu = {ctx.n_gpus}), in-library NCCL" if ctx.single
                                                      else f"one process per GPU (torchrun), packets sharded x{ctx.n_gpus}, flow replicated")),
                "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "clocks": head.get("clocks"),
                "wall_s_timed_region": head["wall_s_timed_region"], "histogram_total": head["histogram_total"],
                "peaks_measured": {"fp64_matmul_tflops": round(peaks["fp64_tflops"], 3), "gather_probe_gbs": round(peaks["gather_gbs"], 1),
                                   "clocks_during_matmul": peak_clk}}
        if "shard_bit_identical" in head:
            line["shard_bit_identical"] = head["shard_bit_identical"]
        if cpu:
            line["cpu_baseline"] = cpu
            line["cpu_baseline_spectral"] = cpu_spec
        if configs:
            line["configs"] = configs
        line.update(side)
        _emit(line)
    if ctx.dist is not None:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
