"""The reference's production driver with everything on the device: ``qgsw_raytrace``.

``qgsw_raytrace(nx, Npackets, near_inertial_factor, T_Fr_days, packet_delay_days, U_g, f, Cg)`` keeps the
signature and control flow of qg_flow_ray_trace/qgsw_raytrace.m:1-180 -- initial PV, packet ring, dt from
the initial flow, the AB3 QG loop, per-step packet advection between the previous and the new flow frame,
packet frames every ``packet_steps_per_save`` steps, PV frames every ``steps_per_save`` steps -- but the QG
solver (engine.QGFlow), the flow-frame construction, and the packet integrator run on the GPU and the
packet state only comes back to the host when a frame is written.  Host work that remains is set-up
(random phases, file I/O); the reference's log header is reproduced so ``parse_data``
(symplectic_full_fourier.m:66-82) still reads it.
"""
from __future__ import annotations

import math
import time

import numpy as np

from . import fieldio
from .engine import (Engine, QGFlow, QG2Flow, MODE_SPECTRAL, SCHEME_LEAPFROG, SCHEME_RK4_PACKET, SCHEME_RK4_XKA, k2g_dev,
                     g2k_dev)
from .reference_api import ode23, matlab_linspace


class _Integrator:
    """A driver's ``integrator=`` name: 'ode23' (reference_api.ode23, the host controller), 'ode23_device' (the controller
    on the device, swrt_ode23), 'ode23_packets' (one controller per packet, swrt_ode23_packets) or, where the driver has
    it, 'leapfrog'.  Any other name raises ValueError."""

    def __init__(self, name, driver, leapfrog=True):
        names = ("ode23", "ode23_device", "ode23_packets") + (("leapfrog",) if leapfrog else ())
        if name not in names:
            raise ValueError(f"{driver}: unknown integrator {name!r} (expected one of {', '.join(names)})")
        self.ode23 = name != "leapfrog"
        self.per_packet = name == "ode23_packets"
        self.opts = {"on_device": name == "ode23_device", "per_packet": self.per_packet}

    def counters(self):
        """the stats entries only the per-packet solve reports"""
        return {"ode23_stopped_packets": 0} if self.per_packet else {}

    def step(self, eng, dt, stats):
        """ode23 over [0, dt] between flow slots 0 and 1, counted into ``stats``"""
        st = ode23(eng, [0.0, dt], dt, **self.opts)
        stats["ode23_steps"] += st["nsteps"]; stats["ode23_failed"] += st["nfailed"]
        if self.per_packet:
            stats["ode23_stopped_packets"] += st["stopped"]


def wavenumber_grids(nx):
    """[kx_,ky_] = ndgrid(-kmax:kmax, 0:kmax) (qgsw_raytrace.m:18-20)"""
    kmax = nx // 2 - 1
    kx = np.arange(-kmax, kmax + 1, dtype=np.float64)[:, None] * np.ones((1, kmax + 1))
    ky = np.ones((2 * kmax + 1, 1)) * np.arange(0, kmax + 1, dtype=np.float64)[None, :]
    return kx, ky


def initial_q(X, Y, a_g, K_d2, rs, k_min=5, k_max=8, ring=False):
    """qgsw_raytrace.m:191-214.  The chained comparison on :202 is always true in MATLAB, so every
    |k|,|l| <= k_max mode is summed (``ring=True`` gives the evidently intended annulus).
    ``rs``: numpy RandomState seeded like ``rng(146)`` (same mt19937 stream, column-major fill)."""
    q = np.zeros_like(X); U = np.zeros_like(X); V = np.zeros_like(X)
    n = 2 * k_max + 1
    phase = 2 * np.pi * rs.rand(n, n).T
    for k in range(-k_max, k_max + 1):
        for l in range(-k_max, k_max + 1):
            K2 = k * k + l * l
            if (not ring) or (k_min ** 2 < K2 <= k_max ** 2):
                wp = k * X + l * Y + phase[k + k_max, l + k_max]
                U -= l * np.sin(wp); V += k * np.sin(wp)
                q -= (K_d2 + K2) * np.cos(wp)
    return a_g / np.sqrt((U * U + V * V).max()) * q


def qgsw_raytrace(nx, Npackets, near_inertial_factor, T_Fr_days, packet_delay_days, U_g, f, Cg, *, outdir="data",
                  integrator="ode23", mode=MODE_SPECTRAL, r_drag=0.1, beta=0.0, force_strength=0.1, max_steps=None,
                  seed=146, device=0, log=print, leapfrog_substeps=4):
    """qgsw_raytrace.m:1-180 on the device.  ``integrator``: 'ode23' (the reference), 'ode23_device' (the same solve
    with the controller on the device, swrt_ode23), 'ode23_packets' (ode23 once per packet, each under its own controller,
    swrt_ode23_packets: a packet that blows up stops alone, counted in ``ode23_stopped_packets``) or 'leapfrog' (the fused
    symplectic stepper with time-centred frame blending).  ``max_steps`` truncates the run (tests)."""
    integ = _Integrator(integrator, "qgsw_raytrace")
    L = 2 * np.pi
    dx = L / nx
    xg = matlab_linspace(-L / 2, L / 2, nx)
    X, Y = np.meshgrid(xg, xg)
    kx_, ky_ = wavenumber_grids(nx)
    K2 = kx_ ** 2 + ky_ ** 2
    rs = np.random.RandomState(seed)                                   # rng(146)
    K_d2 = f / Cg
    T_days = T_Fr_days / f
    CFL_fraction = 0.05
    steps_per_save, packet_steps_per_save = 50, 5
    packet_delay = packet_delay_days / f

    q = initial_q(X, Y, U_g, K_d2, rs)
    qk = g2k_dev(q, device)
    wavenumber_factor = math.sqrt((near_inertial_factor ** 2 - 1) * f ** 2 / Cg ** 2)
    i = np.arange(1, Npackets + 1)
    pk = wavenumber_factor * np.cos(2 * np.pi * i / Npackets)
    pl = wavenumber_factor * np.sin(2 * np.pi * i / Npackets)
    r = rs.rand(Npackets, 2)                                           # rand(1,2) per packet, x then y
    px, py = L * r[:, 0] - L / 2, L * r[:, 1] - L / 2

    # time step and Froude number from the initial flow (qgsw_raytrace.m:62-73)
    psik = -qk / (K_d2 + K2)
    u0 = k2g_dev(-1j * ky_ * psik, device); v0 = k2g_dev(1j * kx_ * psik, device)
    U0 = math.sqrt((u0 * u0 + v0 * v0).max())
    Fr = U0 / Cg
    T = T_days / Fr ** 2
    dt = CFL_fraction * dx / U0
    Nsteps = int(math.ceil(T / dt))
    if max_steps is not None:
        Nsteps = min(Nsteps, int(max_steps))
    packet_step_start = int(math.ceil(packet_delay / dt))

    log("Resolution: %dx%d" % (nx, nx)); log("Number of packets: %d" % Npackets)
    log("Initial wavenumber radius: %f" % (near_inertial_factor * f)); log("Time step: %f" % dt)
    log("Simulation time: %f" % T); log("Spin-up time: %f" % packet_delay)
    log("Steps per save: %d" % steps_per_save); log("Steps per packet save: %d" % packet_steps_per_save)
    log("Coriolis parameter: %f" % f); log("Group velocity: %f" % Cg)
    log("Background velocity (parameter,computed): (%f,%f)" % (U_g, U0)); log("Froude Number: %f" % Fr)
    log("Deformation wavenumber: %f" % K_d2)

    writer = fieldio.PacketFrameWriter(outdir, L)
    writer.write(px, py, pk, pl, dt * (packet_step_start - 1), wrap=False)   # initial positions as drawn, :103-106
    fieldio.write_field(q, f"{outdir}/pv", 1); fieldio.write_field(0.0, f"{outdir}/pv_time", 1)

    qg = QGFlow(nx, L, qk, K_d2, dt, f, Cg, beta=beta, r_drag=r_drag, force_strength=force_strength, device=device)
    eng = Engine(nx, L, f, Cg ** 2, mode, device, bump=1e-10)     # qg_flow_ray_trace/interpolate.m:13, the copy this driver runs beside
    eng.set_packets(px, py, pk, pl)
    t = 0.0
    tic = time.time()
    stats = {"packet_steps": 0, "ode23_steps": 0, "ode23_failed": 0, **integ.counters()}
    for step in range(1, Nsteps + 1):
        if Npackets > 0 and t + dt > packet_delay:
            qg.to_flow(eng, 0)                                         # background_flow1 = grid_U(prev_qk), :141
        qg.step(1)
        t += dt
        if Npackets > 0 and t > packet_delay:
            qg.to_flow(eng, 1)                                         # background_flow2 = grid_U(qk), :142
            if integ.ode23:
                integ.step(eng, dt, stats)                                     # :143-150
            else:
                m = leapfrog_substeps
                eng.step(SCHEME_LEAPFROG, dt / m, m, 0.5 / m, 1.0 / m)
            stats["packet_steps"] += 1
            if (step - packet_step_start + 1) % packet_steps_per_save == 0:
                writer.write(*eng.get_packets(), t)                    # wrapped on save only, :160
        if step % steps_per_save == 0:
            fieldio.write_field(qg.get_grid(), f"{outdir}/pv", 0)
            fieldio.write_field(t, f"{outdir}/pv_time", 0)
    log("Real time elapsed: %.3f seconds" % (time.time() - tic))
    out = {"dt": dt, "Nsteps": Nsteps, "U0": U0, "Fr": Fr, "t": t, "packets": eng.get_packets(), "qk": qg.get(), **stats,
           "packet_frames": writer.frames}
    qg.close(); eng.close()
    return out


# =====================================================================================================
# The other four scripts BASELINE.json's configs name, each with its own control flow and defaults kept.
# They are scripts (no arguments) in the reference; here the constants edited in-file become keyword
# arguments whose defaults are the reference's values, and inputs the reference loads from files that are
# not in the tree (analysis/pv.bin, wavevort_231058_restart_frame100.mat) are arguments.
# =====================================================================================================

def parse_data(filename):
    """symplectic_full_fourier.m:66-82 / SW_zero_background_raytracing.m:146-162: read nx, Npackets, f, Cg,
    U_g back from a run log header (qgsw_raytrace.m:76-88) -> (resolution, Npackets, f, Cg, Ug)."""
    import re
    with open(filename, "r", errors="replace") as fh:
        text = fh.read(8192)
    def grab(pat, cast=float):
        m = re.search(pat, text)
        if not m:
            raise ValueError(f"parse_data: {pat!r} not found in {filename}")
        return cast(m.group(1))
    return (grab(r"Resolution: (\d+)x\d+", int), grab(r"Number of packets: (\d+)", int), grab(r"Coriolis parameter: ([-\d.eE+]+)"),
            grab(r"Group velocity: ([-\d.eE+]+)"), grab(r"Background velocity \(parameter,computed\): \(([-\d.eE+]+),"))


def _ring_packets(Nparticles, L, radius, rs):
    """symplectic_full_fourier.m:22-28: k on a ring, x = L*rand(1,2) - L/2 drawn per packet -> (1,2,Np) arrays"""
    i = np.arange(1, Nparticles + 1)
    r = rs.rand(Nparticles, 2)
    x = np.zeros((1, 2, Nparticles)); k = np.zeros((1, 2, Nparticles))
    k[0, 0] = radius * np.cos(2 * np.pi * i / Nparticles); k[0, 1] = radius * np.sin(2 * np.pi * i / Nparticles)
    x[0, 0] = L * r[:, 0] - L / 2; x[0, 1] = L * r[:, 1] - L / 2
    return x, k


def _frozen_flow_setup(q, nx, f, Cg, Nparticles, grid_lo, mode, device, seed, ring_radius=3.0):
    """the common head of symplectic_full_fourier.m:5-38 and SW_zero_background_raytracing.m:6-50"""
    from .reference_api import SpectralScheme, g2k, k2g
    L = 2 * np.pi
    K_d2 = f / Cg
    kx_, ky_ = wavenumber_grids(nx)
    K2 = kx_ ** 2 + ky_ ** 2
    rs = np.random.RandomState(seed)                                   # rng(123)
    X = matlab_linspace(grid_lo, grid_lo + L, nx)                       # linspace(0,L,nx) / linspace(-L/2,L/2,nx)
    XX, YY = np.meshgrid(X, X)
    gH = Cg ** 2
    scheme = SpectralScheme(L, nx, k2g(-g2k(q, device) / (K_d2 + K2), device), mode=mode, f=f, gH=gH, device=device)
    x, k = _ring_packets(Nparticles, L, ring_radius, rs)
    U = scheme.U(np.stack([XX.ravel(order="F"), YY.ravel(order="F")], axis=1))     # scheme.U([XX(:), YY(:)])
    U0 = float(np.sqrt((U ** 2).sum(axis=1)).max())
    Fr = U0 / Cg
    dt = 0.1 * (L / nx) / max(Cg, U0)
    return L, gH, scheme, x, k, U0, Fr, dt


def _omega_abs(scheme, x, k, f, gH):
    """omega(k) + dot(scheme.U(x), k, 2) over a (T,2,Np) history (symplectic_full_fourier.m:41,55)"""
    U = scheme.U(x)
    return np.sqrt(f * f + gH * (k ** 2).sum(axis=1)) + (U * k).sum(axis=1)


def symplectic_full_fourier(q=None, *, nx=None, f=None, Cg=None, run_log_file=None, pv=None, frame=2000, Nparticles=10,
                            Tend=None, save_stride=1, mode=MODE_SPECTRAL, seed=123, device=0):
    """symplectic_full_fourier.m:1-60 (BASELINE config 2): frozen QG frame -> SpectralScheme -> ring of packets
    -> ``ode_symplectic`` -> relative drift of the absolute frequency Omega = omega + U.k.

    The PV frame comes from ``q`` (nx x nx), or from frame ``frame`` of the write_field stream ``pv`` (the
    reference reads frame 2000 of analysis/pv, which is git-ignored); nx, f, Cg from ``run_log_file`` via
    ``parse_data`` when not given.  Returns dict(solver_x, solver_k, solver_t, solver_error, Omega_0, U0, Fr, dt,
    Tend).  ``save_stride`` > 1 keeps every stride-th row of the history (extension for large Nparticles)."""
    from .reference_api import ode_symplectic
    if run_log_file is not None:
        lnx, _, lf, lCg, _ = parse_data(run_log_file)
        nx, f, Cg = nx or lnx, f if f is not None else lf, Cg if Cg is not None else lCg
    if q is None:
        q = fieldio.read_field(pv, nx, nx, 1, [frame])[:, :, 0, 0] if pv is not None else None
    if q is None:
        raise ValueError("symplectic_full_fourier: pass the PV frame q, or pv=<write_field stream> (analysis/pv is not in the tree)")
    q = np.asarray(q, dtype=np.float64).reshape(nx, nx)
    L, gH, scheme, x, k, U0, Fr, dt = _frozen_flow_setup(q, nx, f, Cg, Nparticles, 0.0, mode, device, seed)
    Tend = 10 / (f * Fr ** 2) if Tend is None else Tend
    Omega_0 = _omega_abs(scheme, x, k, f, gH)
    sx, sk, st = ode_symplectic(x, k, dt, Tend, f, gH, scheme, save_stride=save_stride)
    Omega_abs = _omega_abs(scheme, sx, sk, f, gH)
    return {"solver_x": sx, "solver_k": sk, "solver_t": st, "solver_error": (Omega_abs - Omega_0) / Omega_0, "Omega_0": Omega_0,
            "U0": U0, "Fr": Fr, "dt": dt, "Tend": Tend, "scheme": scheme}


def SW_zero_background_raytracing(q=None, *, nx=None, f=None, Cg=None, run_log_file=None, pv=None, frame=2000, Nparticles=10,
                                  Tend=None, rtol=1e-6, atol=1e-7, mode=MODE_SPECTRAL, seed=123, device=0, integrator="ode23"):
    """SW_zero_background_raytracing.m:1-132 (BASELINE config 1): the same frozen frame and packet ring, integrated
    by ``ode23`` with RelTol 1e-6 / AbsTol 1e-7 and output requested at ``t_hist = dt*(0:Nsteps)`` (:70-78), RHS
    ``dx/dt = U + gH k/omega`` (:134-145,182-184).  ``q = zeros`` is the "zero background" of the file name
    (the hint on :28-29).  ``integrator='ode23_device'`` runs the solve with the controller on the device (swrt_ode23),
    ``integrator='ode23_packets'`` solves every packet under its own controller (swrt_ode23_packets).
    Returns dict(t_hist, solver_x, solver_k, solver_error, w, Omega_0, U0, Fr, dt, stats)."""
    from .engine import FLAG_RHS_GH
    integ = _Integrator(integrator, "SW_zero_background_raytracing", leapfrog=False)
    if run_log_file is not None:
        lnx, _, lf, lCg, _ = parse_data(run_log_file)
        nx, f, Cg = nx or lnx, f if f is not None else lf, Cg if Cg is not None else lCg
    if q is None and pv is not None:
        q = fieldio.read_field(pv, nx, nx, 1, [frame])[:, :, 0, 0]
    if q is None:
        raise ValueError("SW_zero_background_raytracing: pass the PV frame q (zeros for the zero-background case) or pv=<stream>")
    q = np.asarray(q, dtype=np.float64).reshape(nx, nx)
    L, gH, scheme, x, k, U0, Fr, dt = _frozen_flow_setup(q, nx, f, Cg, Nparticles, -np.pi, mode, device, seed)
    if Tend is None:
        if Fr == 0:
            raise ValueError("zero background flow: Fr = 0, pass Tend explicitly (the reference's 1/(f*Fr^2) is infinite)")
        Tend = 1 / (f * Fr ** 2)
    Nsteps = int(math.floor(Tend / dt))
    Omega_0 = _omega_abs(scheme, x, k, f, gH)[0]
    t_hist = dt * np.arange(0, Nsteps + 1)
    eng = Engine(nx, L, f, gH, mode, device, flags=FLAG_RHS_GH)
    eng.set_flow_spectral(scheme.psik)
    eng.set_packets(x[0, 0], x[0, 1], k[0, 0], k[0, 1])
    stats = ode23(eng, t_hist, None, rtol=rtol, atol=atol, **integ.opts)                          # steady flow: slot 0
    Y = stats.pop("Y")
    eng.close()
    solver_x, solver_k = Y[:, 0:2, :], Y[:, 2:4, :]
    w = np.sqrt(f * f + gH * (solver_k ** 2).sum(axis=1))
    Omega_abs = _omega_abs(scheme, solver_x, solver_k, f, gH)
    return {"t_hist": t_hist, "solver_x": solver_x, "solver_k": solver_k, "w": w, "solver_error": (Omega_abs - Omega_0) / Omega_0,
            "Omega_0": Omega_0, "U0": U0, "Fr": Fr, "dt": dt, "Nsteps": Nsteps, "stats": stats, "scheme": scheme}


def childress_soward_fields(nx, L, U0, km, a, faithful=True):
    """ray_trace_sw/raytrace.m:26-37 on ``[x_,y_] = ndgrid(0:dx:dx*(nx-1))``.  ``faithful=True`` keeps line 36 as
    written -- ``a*cos(km*x_)*cos(km*y_)`` is a MATRIX product there -- so v_x is what the reference computes;
    ``faithful=False`` uses the element-wise product the formula intends."""
    dx = L / nx
    x = dx * np.arange(nx)
    x_, y_ = np.meshgrid(x, x, indexing="ij")
    sx, cx, sy, cy = np.sin(km * x_), np.cos(km * x_), np.sin(km * y_), np.cos(km * y_)
    cc = (cx @ cy) if faithful else cx * cy
    U = {"u": -U0 * (sx * cy - a * cx * sy), "v": U0 * (cx * sy - a * sx * cy)}
    GradU = {"u_x": -km * U0 * (cx * cy + a * sx * sy), "u_y": km * U0 * (sx * sy + a * cx * cy),
             "v_x": -km * U0 * (sx * sy + a * cc), "v_y": km * U0 * (cx * cy + a * sx * sy)}
    psi = U0 / km * (sx * sy + a * cx * cy)
    return psi, U, GradU


def _packet_history_run(stepper, P0, dt, nsteps, save_stride, with_a):
    """the packet-major double loop of raytrace.m:50-54 / raytrace_sw.m:125-130 with all packets advanced together:
    column j of the history = state after j-1 steps (P(i,j)); every save_stride-th column is kept."""
    cols = list(range(0, nsteps, save_stride))
    names = ("x", "y", "k", "l") + (("a",) if with_a else ())
    hist = {n: np.zeros((P0["x"].size, len(cols))) for n in names}
    for n in names:
        hist[n][:, 0] = P0[n]
    eng = stepper.eng
    eng.set_packets(P0["x"], P0["y"], P0["k"], P0["l"], P0["a"] if with_a else None)
    done = 0
    for c in range(1, len(cols)):
        eng.step(SCHEME_RK4_XKA if with_a else SCHEME_RK4_PACKET, dt, cols[c] - done)
        done = cols[c]
        for n, v in zip(names, eng.get_packets(with_a=with_a)):
            hist[n][:, c] = v
    return hist, np.asarray(cols)


def raytrace(*, C0=1.0, Fr=0.1, f=4.0, a=0.25, np_=5, nx=256, nsteps=None, save_stride=1, faithful=True, mode=None, seed=5489,
             device=0):
    """ray_trace_sw/raytrace.m:1-64: packets in an analytic Childress-Soward flow advanced by ``step_packet``.
    Returns dict(P={x,y,k,l: (np, nsaved)}, t, omega, Cmag, K, psi, U, GradU, dt, nsteps).  ``seed`` 5489 is
    MATLAB's start-up generator state (the script never calls rng)."""
    from .engine import MODE_LAGRANGE6
    from .reference_api import PacketStepper
    mode = MODE_LAGRANGE6 if mode is None else mode
    U0 = Fr; L = 2 * np.pi
    kd = f / C0 ** 2; km = kd; ki = km * 10
    dx = L / nx
    dt = 0.3 * dx / max(C0, U0)
    Tend = 1 / (f * Fr ** 2)
    nsteps = int(round(Tend / dt)) if nsteps is None else int(nsteps)
    psi, U, GradU = childress_soward_fields(nx, L, U0, km, a, faithful)
    rs = np.random.RandomState(seed)
    r = rs.rand(np_, 2); i = np.arange(1, np_ + 1)
    P0 = {"x": r[:, 0] * L, "y": r[:, 1] * L, "k": ki * np.cos(2 * np.pi * i / np_), "l": ki * np.sin(2 * np.pi * i / np_)}
    stepper = PacketStepper(U, GradU, None, C0, f, dx, mode, device)
    P, cols = _packet_history_run(stepper, P0, dt, nsteps, save_stride, False)
    stepper.eng.close()
    K2 = P["k"] ** 2 + P["l"] ** 2
    omega = np.sqrt(f ** 2 + C0 ** 2 * K2)                              # cg_sw.m:22 without H
    return {"P": P, "t": dt * cols, "omega": omega, "Cmag": C0 ** 2 * np.sqrt(K2) / omega, "K": np.sqrt(K2), "psi": psi, "U": U,
            "GradU": GradU, "dt": dt, "nsteps": nsteps}


def geostrophic_fields(S, f, Cg, device=0):
    """ray_trace_sw/raytrace_sw.m:14-52: geostrophic mode of an [u,v,eta] state (the recipe of
    rsw/wavevortdecomp.m:41-45) and its gradients on the grid -> (U, GradU, H); transforms on the device."""
    S = np.asarray(S, dtype=np.float64)
    nx = S.shape[0]
    kx_, ky_ = wavenumber_grids(nx)
    K2_ = kx_ ** 2 + ky_ ** 2
    gH0 = Cg ** 2
    sig2_ = f ** 2 + gH0 * K2_
    uk, vk, etak = (g2k_dev(S[:, :, j], device) for j in range(3))
    zetak = 1j * (kx_ * vk - ky_ * uk)
    etagk = (f * etak - zetak) * f / sig2_
    ugk = -1j * ky_ * (gH0 / f * etagk)
    vgk = 1j * kx_ * (gH0 / f * etagk)
    H = 1 + k2g_dev(etagk, device)
    U = {"u": k2g_dev(ugk, device), "v": k2g_dev(vgk, device)}
    GradU = {"u_x": k2g_dev(1j * kx_ * ugk, device), "u_y": k2g_dev(1j * ky_ * ugk, device),
             "v_x": k2g_dev(1j * kx_ * vgk, device), "v_y": k2g_dev(1j * ky_ * vgk, device)}
    return U, GradU, H


def raytrace_sw(S, f, Cg, *, np_=10, nsteps=None, save_stride=1, mode=None, seed=5489, device=0):
    """ray_trace_sw/raytrace_sw.m:11-140 (BASELINE config 5): geostrophic part of a shallow-water state
    ``S(:,:,1:3) = [u,v,eta]`` (what ``load wavevort_231058_restart_frame100`` provides, with f and Cg), packets on
    the ring ki = 10 kd advanced by ``step_packet_xka`` with wave action.  Returns dict(P={x,y,k,l,a}, t, omega,
    Cmag, K, U, GradU, H, U0, Fr, dt, nsteps); omega/Cmag are cg_sw (:135) evaluated with H at each packet."""
    from .engine import MODE_LAGRANGE6
    from .reference_api import PacketStepper
    mode = MODE_LAGRANGE6 if mode is None else mode
    S = np.asarray(S, dtype=np.float64)
    nx = S.shape[0]
    gH0 = Cg ** 2; C0 = Cg
    U, GradU, H = geostrophic_fields(S, f, Cg, device)
    L = 2 * np.pi
    kd = f / C0; ki = kd * 10
    U0 = float(np.sqrt(U["u"] ** 2 + U["v"] ** 2).max())
    Fr = U0 / C0
    dx = L / nx
    dt = 0.3 * dx / max(C0, U0)
    if nsteps is None:
        nsteps = int(round(20 / (f * Fr ** 2) / dt))
    rs = np.random.RandomState(seed)
    r = rs.rand(np_, 2); i = np.arange(1, np_ + 1)
    P0 = {"x": r[:, 0] * L, "y": r[:, 1] * L, "k": ki * np.cos(2 * np.pi * i / np_), "l": ki * np.sin(2 * np.pi * i / np_),
          "a": np.ones(np_)}
    stepper = PacketStepper(U, GradU, H, C0, f, dx, mode, device)
    P, cols = _packet_history_run(stepper, P0, dt, int(nsteps), save_stride, True)
    # [C, omega] = cg_sw(k,l,C0,f,H) is a whole-grid field per packet in the reference (:135); the per-packet number
    # that is meaningful (and that the plots average) is the one at the packet: H interpolated to (x,y)
    Hp = stepper.eng.eval_at(P["x"].ravel(order="F"), P["y"].ravel(order="F"), with_H=True)[6].reshape(P["x"].shape, order="F")
    stepper.eng.close()
    K2 = P["k"] ** 2 + P["l"] ** 2
    omega = np.sqrt(f ** 2 + gH0 * Hp * K2)
    return {"P": P, "t": dt * cols, "omega": omega, "Cmag": gH0 * Hp * np.sqrt(K2) / omega, "K": np.sqrt(K2), "U": U, "GradU": GradU,
            "H": H, "U0": U0, "Fr": Fr, "dt": dt, "nsteps": int(nsteps)}



def initial_q_2layer(X, Y, a_g, K_d2, rs, k_min=10, k_max=30, ring=False):
    """qg2layersw_raytrace.m:250-273: the same random-phase sum as the one-layer driver with k_max = 30 (and the
    same always-true chained comparison on :262)."""
    return initial_q(X, Y, a_g, K_d2, rs, k_min=k_min, k_max=k_max, ring=ring)


def qg2layersw_raytrace(nx, Npackets, near_inertial_factor, T_Fr_days, packet_delay_Fr_days, U_g, f, Cg, *, outdir="data",
                        mode=MODE_SPECTRAL, max_steps=None, seed=5, device=0, log=print, k_max=30, integrator="ode23",
                        leapfrog_substeps=4):
    """qg_flow_ray_trace/qg2layersw_raytrace.m:1-247 (BASELINE config 4) on the device: two-layer QG with mean shear on
    L = 20, adaptive dt (:156-165), AB3 + integrating factor, packets advected through the TOP layer's
    ``grid_U`` frames (:187-196) by ode23 over [0, dt] ('ode23_device': controller on the device; 'ode23_packets': one
    controller per packet, stopped packets counted in ``ode23_stopped_packets``), packet frames every
    25 steps.  ``k_max`` (30 in the reference)
    and ``max_steps`` exist for tests."""
    integ = _Integrator(integrator, "qg2layersw_raytrace")
    L = 20.0
    dx = L / nx
    xg = matlab_linspace(-L / 2, L / 2, nx)
    X, Y = np.meshgrid(xg, xg, indexing="ij")                          # ndgrid (:16)
    rs = np.random.RandomState(seed)                                   # rng(5)
    beta = 0.0
    K_d2 = f / Cg
    shear_strength = 0.5
    T_Fr = T_Fr_days / f
    packet_delay_Fr = packet_delay_Fr_days / f
    CFL_fraction = 0.25
    alpha = 4; r = 0.4; nutune = 0.1
    steps_per_save = 10
    packet_delay_steps = packet_delay_Fr / f
    packet_steps_per_save = 25

    q1 = initial_q_2layer(X, Y, U_g, K_d2, rs, k_max=k_max)
    q1k = g2k_dev(q1, device)
    wavenumber_factor = math.sqrt((near_inertial_factor ** 2 - 1) * f ** 2 / Cg ** 2)
    i = np.arange(1, Npackets + 1)
    pk = wavenumber_factor * np.cos(2 * np.pi * i / Npackets)
    pl = wavenumber_factor * np.sin(2 * np.pi * i / Npackets)
    rr = rs.rand(Npackets, 2)
    px, py = L * rr[:, 0] - L / 2, L * rr[:, 1] - L / 2

    nu = nutune * dx ** (2 * alpha)
    qg = QG2Flow(nx, L, q1k, -q1k, K_d2, beta, shear_strength, r, nu, alpha, device)      # q2 = -q1 (:57)
    U0 = qg.max_speed()
    Fr = U0 / Cg
    T = T_Fr / Fr ** 2
    dt = CFL_fraction * dx / U0
    Nsteps = int(math.ceil(T / dt))
    packet_step_start = int(math.ceil(packet_delay_steps / dt))

    log("Resolution: %dx%d" % (nx, nx)); log("Number of packets: %d" % Npackets)
    log("Initial wavenumber radius: %f" % (near_inertial_factor * f)); log("Initial time step: %f" % dt)
    log("Simulation time: %f" % T); log("Spin-up time: %f" % packet_delay_steps)
    log("Steps per save: %d" % steps_per_save); log("Steps per packet save: %d" % packet_steps_per_save)
    log("Coriolis parameter: %f" % f); log("Group velocity: %f" % Cg)
    log("Background velocity (parameter,computed): (%f,%f)" % (U_g, U0)); log("Froude Number: %f" % Fr)
    log("Deformation wavenumber: %f" % K_d2)

    writer = fieldio.PacketFrameWriter(outdir, L)
    writer.write(px, py, pk, pl, dt * (packet_step_start - 1), wrap=False)            # :114-116 (unwrapped initial frame)
    fieldio.write_field(np.stack([q1, -q1], axis=2), f"{outdir}/pv", 1); fieldio.write_field(0.0, f"{outdir}/pv_time", 1)

    eng = Engine(nx, L, f, Cg ** 2, mode, device, bump=1e-10)     # qg_flow_ray_trace/interpolate.m:13, the copy this driver runs beside
    eng.set_packets(px, py, pk, pl)
    t = 0.0
    step = 0
    tic = time.time()
    stats = {"packet_steps": 0, "ode23_steps": 0, "ode23_failed": 0, "dt_changes": 0, **integ.counters()}
    while t <= T and (max_steps is None or step < max_steps):
        step += 1
        U0 = qg.max_speed()
        CFL_condition = CFL_fraction * dx / U0
        if CFL_condition < dt or dt < CFL_condition / 4:
            dt = CFL_fraction / 2 * dx / U0
            stats["dt_changes"] += 1
            log("CFL condition not met, max|u|=%f, new dt=%f" % (U0, dt))
        advect = Npackets > 0 and t + dt > packet_delay_steps
        if advect:
            qg.to_flow(eng, 0)                                         # background_flow1 = grid_U(prev_qk(:,:,:,1)), :187
        qg.step(dt)
        t = t + dt
        if advect:
            qg.to_flow(eng, 1)                                         # background_flow2 = grid_U(qk(:,:,:,1)), :188
            if integ.ode23:
                integ.step(eng, dt, stats)
            else:
                m = leapfrog_substeps
                eng.step(SCHEME_LEAPFROG, dt / m, m, 0.5 / m, 1.0 / m)
            stats["packet_steps"] += 1
            if (step - packet_step_start + 1) % packet_steps_per_save == 0:
                writer.write(*eng.get_packets(), t)
    log("Real time elapsed: %.3f seconds" % (time.time() - tic))
    out = {"dt": dt, "Nsteps": Nsteps, "steps": step, "U0": U0, "Fr": Fr, "t": t, "T": T, "packets": eng.get_packets(),
           "qk": (qg.get(0), qg.get(1)), **stats, "packet_frames": writer.frames}
    qg.close(); eng.close()
    return out


def load_data(directory, *, times=None, offset=500, bins=300, device=0):
    """analysis/load_data.m:11-64, the computational half (the plots are out of scope): read ``run.log`` and the
    ``packet_time / packet_x / packet_k`` frame streams a driver wrote, form omega = sqrt(f^2 + Cg^2 k.k) per packet and
    frame (:33), ``edges = linspace(0, max omega, 300)`` (:38-39), and for every window ``times(i) +- offset`` frames
    (:36-37,44-49) the histcounts distribution and ``energy = center .* distribution``; plus mean omega(t)/f (:63).
    The histograms run on the device (u64 counts, the reference's bin rule).  ``times`` are 1-based frame numbers as in
    the script; its default ``[1000, 30000, nframes - offset]`` is clipped to the frames that exist."""
    from pathlib import Path
    from .engine import HIST_INTRINSIC
    d = Path(directory)
    nx, Npackets, f, Cg, Ug = parse_data(d / "run.log")
    t, x_save, k_save = fieldio.load_packet_frames(d, Npackets)
    nfr = t.size
    omega = np.sqrt(f ** 2 + Cg ** 2 * (k_save ** 2).sum(axis=1))                   # (Np, frames)
    edges = matlab_linspace(0.0, omega.max(), bins)
    center = (edges[1:] + edges[:-1]) / 2
    if times is None:
        times = [tt for tt in (1000, 30000, nfr - offset) if offset < tt <= nfr - offset] or [max(1, nfr // 2)]
    eng = Engine(8, 2 * np.pi, f, Cg ** 2, MODE_SPECTRAL, device)                   # only its packet/histogram kernels are used
    windows = []
    for tc in times:
        lo, hi = max(1, tc - offset), min(nfr, tc + offset)                         # frames tc-offset : tc+offset, 1-based inclusive
        kk = k_save[:, 0, lo - 1:hi].ravel(order="F"); ll = k_save[:, 1, lo - 1:hi].ravel(order="F")
        eng.set_packets(np.zeros_like(kk), np.zeros_like(kk), kk, ll)
        counts = eng.hist_omega(edges, kind=HIST_INTRINSIC)
        windows.append({"time_index": int(tc), "frames": (lo, hi), "distribution": counts, "energy": center * counts.astype(np.float64)})
    eng.close()
    return {"nx": nx, "Npackets": Npackets, "f": f, "Cg": Cg, "Ug": Ug, "t_packet_save": t, "omega": omega, "edges": edges,
            "center": center, "windows": windows, "mean_omega": omega.mean(axis=0) / f}
