"""Host-side mirror of the reference's MATLAB calling surface for the packet hot path.

Same function names, argument order/meaning and array shapes as the reference (file:line cited per
function, relative to the reference tree), implemented on top of the C ABI (engine.py ->
libswrt.so).  Everything numeric runs on the GPU; there is no CPU fallback -- constructing any of
these without the CUDA library raises.

Array conventions follow the reference: gridded fields are ``F[ix, iy]`` (x first, MATLAB
``ndgrid``), spectral fields are ``fk[kx + kmax, ky]`` (g2k layout), packet positions for the
scheme classes are ``(T, 2, Np)`` and for the ``qgsw`` drivers ``(Np, 2)``.
"""
from __future__ import annotations

import math

import numpy as np

from . import engine as _e
from .engine import Engine, MODE_LAGRANGE6, MODE_SPECTRAL, SCHEME_LEAPFROG, SCHEME_RK4_PACKET, SCHEME_RK4_XKA

# ------------------------------------------------------------------------------------------------
# spectral <-> grid kit (setup path; device cuFFT through the C ABI)
# ------------------------------------------------------------------------------------------------

def g2k(fg, device=0):
    """qg_flow_ray_trace/g2k.m:1-9"""
    return _e.g2k_dev(fg, device)


def k2g(fk, device=0):
    """qg_flow_ray_trace/k2g.m:1-6 (+ fulspec.m:10-19)"""
    return _e.k2g_dev(fk, device)


def grid_U(qk, K_d2, K2, kx_, ky_, shear_strength=0.0, device=0):
    """qg_flow_ray_trace/grid_U.m:1-18 -> dict(u,v,ux,uy,vx,vy) of nx x nx grids.
    The six k2g transforms run on the device; the ik-multiplications are O(nx^2) setup."""
    psik = -np.asarray(qk) / (K_d2 + K2)
    vk = 1j * kx_ * psik
    uk = -1j * ky_ * psik
    planes = {"u": uk, "v": vk, "ux": 1j * kx_ * uk, "uy": 1j * ky_ * uk, "vx": 1j * kx_ * vk, "vy": 1j * ky_ * vk}
    out = {name: k2g(p, device) for name, p in planes.items()}
    out["u"] = out["u"] + shear_strength
    return out


def matlab_linspace(d1, d2, n=100):
    """MATLAB's ``linspace``: ``d1 + (0:n-1).*(d2 - d1)./(n-1)`` -- multiply, THEN divide -- with both ends forced.
    ``numpy.linspace`` multiplies by a pre-divided step instead, which differs in the last bit for most points; the grids and
    wavevector fans of the reference's scripts (symplectic_full_fourier.m:14, qgsw_raytrace.m:14, ideal_omega_distribution.m:3,
    analysis/load_data.m:39) are reproduced with MATLAB's formula.  (Found by executing ideal_omega_distribution.m.)"""
    d1 = float(d1); d2 = float(d2); n = int(n)
    if n <= 0:
        return np.zeros(0)
    if n == 1:
        return np.array([d2])
    y = d1 + np.arange(n, dtype=np.float64) * (d2 - d1) / (n - 1)
    y[0], y[-1] = d1, d2
    return y


# ------------------------------------------------------------------------------------------------
# interpolate / interpolate_par / interpolate2 / interpolate_U
# ------------------------------------------------------------------------------------------------
# The reference keeps two copies of interpolate.m that differ in one line: ray_trace_sw/interpolate.m:13 has bump 1e-13 (what
# SpectralScheme, step_packet* and the raytrace* drivers bind to, SpectralScheme.m:8), qg_flow_ray_trace/interpolate.m:13 has
# 1e-10 (what interpolate_U.m and the QG drivers' odefun bind to: runqgsw_raytrace.sbatch:25-27 copies that one next to them).
BUMP_LIVE = 1e-13
BUMP_QG = 1e-10


def interpolate(x, y, F, dx, dy, device=0):
    """ray_trace_sw/interpolate.m:1-50 -- FI = interpolate(x,y,F,dx,dy), bump 1e-13."""
    return _e.interpolate_dev(x, y, F, dx, dy, 1e-13, device)


def interpolate_par(x, y, F, dx, dy, device=0):
    """interpolate_par.m:1-53 -- the same stencil with bump 1e-10."""
    return _e.interpolate_dev(x, y, F, dx, dy, 1e-10, device)


def interpolate2(x, y, F, dx, dy, device=0):
    """interpolate2.m:1-19 is an abandoned ``interp2(...,'cubic')`` experiment whose call sites are all
    commented out (SpectralScheme.m:41,52-53,64-67); the name is kept as an alias of ``interpolate``."""
    return interpolate(x, y, F, dx, dy, device)


class FlowFrames:
    """Two background-flow frames resident on the device (what interpolate_U.m:5-17 re-interpolates
    on every call).  ``bf`` dicts use the reference's field names u,v,ux,uy,vx,vy (grid_U.m:11-17).
    ``bump`` defaults to 1e-10: interpolate_U.m binds to the interpolate.m beside it (BUMP_QG above)."""

    def __init__(self, bf1, bf2, h, f=1.0, gH=1.0, mode=MODE_LAGRANGE6, device=0, bump=BUMP_QG):
        nx = np.asarray(bf1["u"]).shape[0]
        self.eng = Engine(nx, h * nx, f, gH, mode, device, bump=bump)
        self.eng.set_flow_grid(*[bf1[n] for n in ("u", "v", "ux", "uy", "vx", "vy")], slot=0)
        if bf2 is not None:
            self.eng.set_flow_grid(*[bf2[n] for n in ("u", "v", "ux", "uy", "vx", "vy")], slot=1)

    def interpolate_U(self, alpha, x):
        x = np.asarray(x, dtype=np.float64)
        e = self.eng.eval_at(x[:, 0], x[:, 1], alpha)
        U = np.stack([e[0], e[1]], axis=1)
        return U, {"u_x": e[2], "u_y": e[3], "v_x": e[4], "v_y": e[5]}


def interpolate_U(background_flow1, background_flow2, alpha, x, h, device=0, bump=BUMP_QG):
    """qg_flow_ray_trace/interpolate_U.m:1-24 -- [U, nablaU] = interpolate_U(bf1, bf2, alpha, x, h)."""
    return FlowFrames(background_flow1, background_flow2, h, device=device, bump=bump).interpolate_U(alpha, x)


def generate_raytracing_ode(background_flow1, background_flow2, Npackets, f, Cg, tmax, h, device=0, mode=MODE_LAGRANGE6, bump=BUMP_QG):
    """qgsw_raytrace.m:258-268 -- returns odefun(t, y) with y = [x; y; k; l] (4*Np,)."""
    frames = FlowFrames(background_flow1, background_flow2, h, f=f, gH=Cg * Cg, mode=mode, device=device, bump=bump)

    def odefun(t, y):
        y = np.asarray(y, dtype=np.float64).ravel()
        n = Npackets
        frames.eng.set_packets(y[0:n], y[n:2 * n], y[2 * n:3 * n], y[3 * n:4 * n])
        return np.concatenate(frames.eng.rhs(t / tmax))

    return odefun


# ------------------------------------------------------------------------------------------------
# SpectralScheme / ode_symplectic
# ------------------------------------------------------------------------------------------------

class SpectralScheme:
    """SpectralScheme.m:1-69 (+ RaytracingScheme.m:9-16).  ``SpectralScheme(L, nx, psi_field)``.

    ``mode=MODE_SPECTRAL`` evaluates the planes by exact Fourier sum (the B200 contraction kernel);
    ``mode=MODE_LAGRANGE6`` reproduces the reference's gridded 6x6 Lagrange evaluation."""

    def __init__(self, L, nx, psi_field, mode=MODE_SPECTRAL, f=1.0, gH=1.0, device=0):
        self.L, self.nx, self.mode = float(L), int(nx), mode
        self.psik = g2k(np.asarray(psi_field, dtype=np.float64), device)
        self.eng = Engine(nx, L, f, gH, mode, device)
        self.eng.set_flow_spectral(self.psik)
        self._psi_eng = None
        self.device = device

    @staticmethod
    def _split(x):
        x = np.asarray(x, dtype=np.float64)
        if x.ndim == 2:          # (Np, 2)
            return x[:, 0], x[:, 1], None
        return x[:, 0, :].ravel(), x[:, 1, :].ravel(), x[:, 0, :].shape

    def streamfunction(self, x, y, t=0):
        """SpectralScheme.m:38-43"""
        dx = self.L / self.nx
        return interpolate(x, y, k2g(self.psik, self.device), dx, dx, self.device)

    def U(self, x, t=0):
        """SpectralScheme.m:45-54"""
        xx, yy, shp = self._split(x)
        e = self.eng.eval_at(xx, yy)
        if shp is None:
            return np.stack([e[0], e[1]], axis=1)
        u = np.zeros_like(np.asarray(x, dtype=np.float64))
        u[:, 0, :] = e[0].reshape(shp)
        u[:, 1, :] = e[1].reshape(shp)
        return u

    def grad_U(self, x, t=0):
        """SpectralScheme.m:56-68"""
        xx, yy, _ = self._split(x)
        e = self.eng.eval_at(xx, yy)
        return {"u_x": e[2], "u_y": e[3], "v_x": e[4], "v_y": e[5]}

    def grad_U_times_k(self, x, k, t=0):
        """RaytracingScheme.m:9-16"""
        g = self.grad_U(x, t)
        k = np.asarray(k, dtype=np.float64)
        out = np.zeros_like(k)
        if k.ndim == 2:
            out[:, 0] = g["u_x"] * k[:, 0] + g["v_x"] * k[:, 1]
            out[:, 1] = g["u_y"] * k[:, 0] + g["v_y"] * k[:, 1]
            return out
        kk, ll = k[:, 0, :], k[:, 1, :]
        out[:, 0, :] = (g["u_x"] * kk.ravel() + g["v_x"] * ll.ravel()).reshape(kk.shape)
        out[:, 1, :] = (g["u_y"] * kk.ravel() + g["v_y"] * ll.ravel()).reshape(ll.shape)
        return out


    # RaytracingScheme.m:18-31: diagnostics every scheme inherits (host arithmetic on the device-evaluated gradients)
    def vorticity(self, x, t=0):
        g = self.grad_U(x, t)
        return g["v_x"] - g["u_y"]

    def strain(self, x, t=0):
        g = self.grad_U(x, t)
        return np.sqrt((g["u_x"] - g["v_y"]) ** 2 + (g["v_x"] + g["u_y"]) ** 2)

    def okuboWeiss(self, x, t=0):
        """D = v_y^2 + v_x*u_y (RaytracingScheme.m:30; the reference's own call on :29 passes an undefined ``k``)"""
        g = self.grad_U(x, t)
        return g["v_y"] ** 2 + g["v_x"] * g["u_y"]


def ode_symplectic(x0, k0, dt, T, f, gH, scheme, save_stride=1):
    """ode_symplectic.m:1-37 -- [x, k, t] = ode_symplectic(x0, k0, dt, T, f, gH, scheme).

    x0, k0: (1, 2, Np).  Nsteps = floor(T/dt); row i holds the state after i leapfrog steps,
    t(i) = i*dt (zero-based).  ``save_stride`` (extension; the reference stores every step) keeps
    every stride-th row so the history fits at 64k-16M packets; all steps between two saved rows
    run as ONE fused kernel launch with the packet state in registers."""
    x0 = np.asarray(x0, dtype=np.float64); k0 = np.asarray(k0, dtype=np.float64)
    Nsteps = int(math.floor(T / dt))
    rows = list(range(0, Nsteps, save_stride))
    x = np.zeros((len(rows),) + x0.shape[1:]); k = np.zeros_like(x); t = np.zeros(len(rows))
    x[0] = x0[0]; k[0] = k0[0]
    eng = _engine_with(scheme, f, gH)   # the handle's f, gH are creation parameters
    eng.set_packets(x0[0, 0, :], x0[0, 1, :], k0[0, 0, :], k0[0, 1, :])
    done = 0
    for r in range(1, len(rows)):
        eng.step(SCHEME_LEAPFROG, dt, rows[r] - done)
        done = rows[r]
        xs, ys, ks, ls = eng.get_packets()
        x[r, 0], x[r, 1], k[r, 0], k[r, 1] = xs, ys, ks, ls
        t[r] = rows[r] * dt
    return x, k, t


def _engine_with(scheme, f, gH):
    """engine for ``scheme``'s flow with the integrator's f and gH (cached on the scheme)."""
    cache = scheme.__dict__.setdefault("_eng_cache", {})
    key = (float(f), float(gH))
    if key not in cache:
        e = Engine(scheme.nx, scheme.L, f, gH, scheme.mode, scheme.device)
        e.set_flow_spectral(scheme.psik)
        cache[key] = e
    return cache[key]


# ------------------------------------------------------------------------------------------------
# step_packet / step_packet_xka
# ------------------------------------------------------------------------------------------------

class PacketStepper:
    """Device-resident flow for the RK4 packet steppers (ray_trace_sw/step_packet.m,
    step_packet_xka.m).  U = dict(u,v), GradU = dict(u_x,u_y,v_x,v_y), H optional grid."""

    def __init__(self, U, GradU, H, C0, f, dx, mode=MODE_LAGRANGE6, device=0):
        nx = np.asarray(U["u"]).shape[0]
        self.eng = Engine(nx, dx * nx, f, C0 * C0, mode, device)
        self.eng.set_flow_grid(U["u"], U["v"], GradU["u_x"], GradU["u_y"], GradU["v_x"], GradU["v_y"], H)
        self.xka = H is not None

    def step(self, P, dt, nsteps=1):
        x, y, k, l = (np.atleast_1d(np.asarray(P[n], dtype=np.float64)) for n in ("x", "y", "k", "l"))
        a = np.atleast_1d(np.asarray(P["a"], dtype=np.float64)) if "a" in P else None
        self.eng.set_packets(x, y, k, l, a)
        self.eng.step(SCHEME_RK4_XKA if self.xka else SCHEME_RK4_PACKET, dt, nsteps)
        out = self.eng.get_packets(with_a=self.xka)
        names = ("x", "y", "k", "l", "a")[:len(out)]
        scalar = np.ndim(P["x"]) == 0
        return {n: (float(v[0]) if scalar else v) for n, v in zip(names, out)}


def step_packet(P, U, GradU, C0, f, dx, dy, dt, mode=MODE_LAGRANGE6, device=0):
    """ray_trace_sw/step_packet.m:1-78 -- Pout = step_packet(P,U,GradU,C0,f,dx,dy,dt).
    P may hold scalars (one packet, as the reference) or arrays (a struct array of packets)."""
    return PacketStepper(U, GradU, None, C0, f, dx, mode, device).step(P, dt)


def step_packet_xka(P, U, GradU, H, C0, f, dx, dy, dt, mode=MODE_LAGRANGE6, device=0):
    """ray_trace_sw/step_packet_xka.m:1-91 -- adds refraction by H and wave action a."""
    return PacketStepper(U, GradU, H, C0, f, dx, mode, device).step(P, dt)


def cg_sw(k, l, C0, f, U=None, H=None):
    """ray_trace_sw/cg_sw.m:1-32 -- [C, omega, omega_abs, divC, gradomega] = cg_sw(k,l,C0,f,U,H) as the post-processing
    loops of raytrace.m:57-63 / raytrace_sw.m:133-139 call it: host arithmetic on whatever shape ``H`` / ``U`` have
    (inside the steppers the same formulas run on the device, composed node-wise or point-wise).
    Returns (C dict x,y; omega; omega_abs; divC or None; gradomega dict or None)."""
    gH = C0 ** 2 * np.asarray(H, dtype=np.float64) if H is not None else C0 ** 2
    K2 = k ** 2 + l ** 2
    om = np.sqrt(f ** 2 + gH * K2)
    C = {"x": gH * k / om, "y": gH * l / om}
    divC = grad = None
    if U is not None:
        u, v = np.asarray(U["u"], dtype=np.float64), np.asarray(U["v"], dtype=np.float64)
        divC = (k * f * v - l * f * u - C["x"] ** 2 - C["y"] ** 2) / om
        grad = {"x": f * K2 * v / (2 * om), "y": -f * K2 * u / (2 * om)}
    return C, om, np.abs(om), divC, grad


def omega(k, f, gH):
    """symplectic_full_fourier.m:62-64 -- host helper, O(Np)."""
    k = np.asarray(k, dtype=np.float64)
    return np.sqrt(f * f + gH * np.sum(k * k, axis=1))


# ------------------------------------------------------------------------------------------------
# ode23 -- the production drivers' integrator (qgsw_raytrace.m:149, qg2layersw_raytrace.m:195)
# ------------------------------------------------------------------------------------------------

def ode23(target, tspan, tmax, rtol=1e-3, atol=1e-6, reduce_max=None, on_device=False, per_packet=False, events=None, ev_cap=4):
    """``[~, Y] = ode23(ray_ode, [0 dt], y0)`` for the packets resident in ``target`` (an Engine):
    MATLAB's ode23 = Bogacki-Shampine 3(2) pair with first-same-as-last, restated from its published
    description (Shampine & Reichelt, "The MATLAB ODE Suite", SIAM J. Sci. Comput. 18, 1997; MATLAB
    R2020b defaults RelTol 1e-3, AbsTol 1e-6, MaxStep 0.1*|tf-t0|).  MATLAB itself is not available,
    so parity is against the oracle's restatement of the same algorithm (parity unpinned).

    The stages run on the device (swrt_bs23_*); this controller is host logic.  The error norm is the
    inf-norm over ALL packets (the reference bundles them in one 4*Np system), so a multi-GPU caller
    passes ``reduce_max`` (an all-reduce MAX over ranks) and every rank takes identical decisions.
    RHS time dependence: alpha = t/tmax (qgsw_raytrace.m:261); ``tmax=None`` for a steady flow (one slot).  Returns dict(nsteps, nfailed, nfevals, t).

    A ``tspan`` with more than two entries (SW_zero_background_raytracing.m:73-78) additionally returns
    ``Y`` (len(tspan), 4, Np): the state at every requested time from the device-side cubic dense output
    (MATLAB ``ntrp23``, swrt_bs23_interp).  The step sequence follows MATLAB's controller, including the initial step
    ``min(hmax, |tspan(2)-tspan(1)|, 1/rh)``, which for a dense ``tspan`` is bounded by the first output interval.

    A decreasing ``tspan`` (``[T 0]``) integrates backward in time, as MATLAB's ode23 does: ``tdir = -1`` and every step
    is ``h = tdir*absh``, the step-size rules unchanged (they act on ``absh``); a dense row is written once the step has
    passed its time in the direction of integration.  A ``tspan`` entry that steps against that direction raises
    ``ValueError`` (equal neighbours are allowed).  Events stay forward-only.

    One deliberate deviation: a non-finite error estimate (a packet that blew up) REJECTS the step here and, at ``hmin``,
    raises; MATLAB's ``if err > rtol`` is false for NaN, so it would accept the step and carry NaNs on silently.

    ``on_device=True`` (single-process callers, no ``reduce_max``) runs the same solve as one ``Engine.ode23`` call, the
    controller in device memory (swrt_ode23); the returned dict then also holds ``host_waits``.

    ``per_packet=True`` solves every packet under its own controller instead (``Engine.ode23_packets``,
    swrt_ode23_packets): what MATLAB gives when ``ode23`` is called once per packet.  Nothing couples the packets, so
    ``reduce_max`` is refused with it; a packet whose step size falls below hmin stops alone (``stopped``, ``status``).
    ``events`` / ``ev_cap`` (per-packet solve only: the coupled solve has no events) locate level crossings of each
    packet's state as MATLAB's ``odeset('Events', ...)`` would, see ``Engine.ode23_packets``.  A 2-D ``tspan`` of shape
    ``(ntspan, Np)`` (per-packet solve only: the coupled solve has one t) gives packet ``i`` the tspan ``tspan[:, i]``."""
    if events is not None and not per_packet:
        raise ValueError("ode23: events need per_packet=True (the coupled solve has no events)")
    if not per_packet and np.ndim(tspan) != 1:
        raise ValueError("ode23: a per-packet (2-D) tspan needs per_packet=True (the coupled solve has one t)")
    if per_packet:
        if reduce_max is not None:
            raise ValueError("ode23: per_packet=True needs no reduce_max (the packets are not coupled)")
        if events is None:
            return target.ode23_packets(tspan, tmax, rtol, atol)
        return target.ode23_packets(tspan, tmax, rtol, atol, events=events, ev_cap=ev_cap)
    if on_device and reduce_max is None:
        return target.ode23(tspan, tmax, rtol, atol)
    red = reduce_max if reduce_max is not None else (lambda v: v)
    al = (lambda tt: tt / tmax) if tmax else (lambda tt: 0.0)       # tmax=None: steady flow, slot 0 only
    tspan = np.asarray(tspan, dtype=np.float64)
    t0, tfinal = float(tspan[0]), float(tspan[-1])
    tdir = 1.0 if tfinal >= t0 else -1.0      # MATLAB's tdir = sign(tfinal - t0): a decreasing tspan integrates backward
    if np.any(tdir * np.diff(tspan) < 0):
        raise ValueError("ode23: tspan must be monotonic (an entry goes against the direction from tspan[0] to tspan[-1])")
    dense = tspan.size > 2
    if dense:
        Y = np.zeros((tspan.size, 4, target.n)); Y[0] = np.stack(target.get_packets()); nxt = 1
    pw = 1.0 / 3.0
    threshold = atol / rtol
    hmax = min(abs(tfinal - t0), abs(0.1 * (tfinal - t0)))
    t = t0
    rh = red(target.bs23_begin(al(t), threshold)) / (0.8 * rtol ** pw)
    nfevals = 1
    hmin = 16 * np.spacing(abs(t))            # 16*eps(t)
    # MATLAB (odearguments / ode23): htspan = |tspan(2) - tspan(1)|, absh = min(hmax, htspan) -- for a dense tspan the FIRST
    # output interval, not the whole span, bounds the initial step
    absh = min(hmax, abs(float(tspan[1]) - float(tspan[0])))
    if absh * rh > 1:
        absh = 1 / rh
    absh = max(absh, hmin)
    nsteps = nfailed = 0
    done = False
    while not done:
        hmin = 16 * np.spacing(abs(t))
        absh = min(hmax, max(hmin, absh))
        h = tdir * absh
        if 1.1 * absh >= abs(tfinal - t):
            h = tfinal - t
            absh = abs(h)
            done = True
        nofailed = True
        while True:
            tnew = tfinal if done else t + h
            err = absh * red(target.bs23_attempt(h, [al(t + 0.5 * h), al(t + 0.75 * h), al(tnew)], threshold))
            nfevals += 3
            if not (err <= rtol):            # also catches NaN
                nfailed += 1
                if absh <= hmin:
                    raise RuntimeError(f"ode23: step size below hmin at t = {t!r} (a packet blew up?)")
                if nofailed:
                    nofailed = False
                    absh = max(hmin, absh * max(0.5, 0.8 * (rtol / err) ** pw)) if np.isfinite(err) else max(hmin, 0.5 * absh)
                else:
                    absh = max(hmin, 0.5 * absh)
                h = tdir * absh
                done = False
            else:
                break
        nsteps += 1
        if dense:
            while nxt < tspan.size and tdir * (tnew - tspan[nxt]) >= 0:
                Y[nxt] = np.stack(target.bs23_interp(h, 1.0 if tspan[nxt] == tnew else (tspan[nxt] - t) / h))
                nxt += 1
        target.bs23_accept()
        if nofailed:
            temp = 1.25 * (err / rtol) ** pw
            absh = absh / temp if temp > 0.2 else 5.0 * absh
        t = tnew
    stats = {"nsteps": nsteps, "nfailed": nfailed, "nfevals": nfevals, "t": t}
    if dense:
        stats["Y"] = Y
    return stats


def ideal_omega_distribution(scheme, f, Cg, k_0, edges, nangles=100):
    """ideal_omega_distribution.m:3-11: theoretical pdf of the absolute frequency omega_0 + U.k over the
    grid ``X = linspace(0, L, nx); [XX,YY] = meshgrid(X)`` (symplectic_full_fourier.m:14-15) and
    ``t = linspace(0, 2*pi)`` wavevector directions.  MATLAB's ``histogram`` picks its own bins; here the
    caller passes ``edges`` (histcounts rule).  Returns (counts, pdf) with pdf = counts/(N*binwidth)."""
    X = matlab_linspace(0.0, scheme.L, scheme.nx)
    XX, YY = np.meshgrid(X, X)
    t = matlab_linspace(0.0, 2 * np.pi, nangles)
    kvx, kvy = k_0 * np.cos(t), k_0 * np.sin(t)
    omega_0 = math.sqrt(f ** 2 + Cg ** 2 * k_0 ** 2)
    edges = np.asarray(edges, dtype=np.float64)
    counts = scheme.eng.ideal_omega_hist(XX.ravel(order="F"), YY.ravel(order="F"), kvx, kvy, omega_0, edges)
    width = np.diff(edges)
    total = XX.size * nangles
    return counts, counts / (total * np.where(width > 0, width, 1.0))
