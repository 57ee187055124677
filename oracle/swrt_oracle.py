"""CPU oracle for the SWRaytracing packet hot path -- TEST INFRASTRUCTURE ONLY.

This module is a numpy restatement of the reference's MATLAB algorithm for the one hot path
this repository accelerates (evaluate U, V, grad U at every wave packet + integrator step).
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it; the product (``swraytracing_b200``) never does.

Parity status -- what is pinned and what is not:

* **Pinned against the reference's own stored outputs** (``tests/test_reference_goldens.py``,
  fixture ``tests/golden/reference_runlogs.json`` extracted from /root/reference by the committed
  script ``tests/golden/make_reference_goldens.py``): the chain ``rng(146)``/``rand`` ->
  ``initial_q`` (with the always-true chained comparison of qgsw_raytrace.m:202) -> ``g2k`` ->
  ``grid_U`` -> ``k2g``/``fulspec`` -> ``U0`` -> ``dt``.  The 19 MATLAB R2020b run logs the
  reference ships (run.log, analysis/job-*/run-*/run.log) print U0, Fr and dt to six decimals for
  ten U_g -- reproduced digit for digit -- and the stored ``pv_time`` frame stream (2,682 frames of
  ``t = t + dt``) is reproduced bit for bit but for three frames at 1-2 ulps, which fixes U0 to a
  few ulps of what MATLAB computed.
* **Pinned against the reference itself, executed here** for the packet arithmetic (``interpolate``,
  ``interpolate_U``, the ``odefun`` right-hand side, ``SpectralScheme`` constructor / ``U`` / ``grad_U`` /
  ``grad_U_times_k``, ``ode_symplectic`` x 100 steps, ``cg_sw``, ``step_packet`` and ``step_packet_xka`` x 3
  steps): ``tests/golden/octave_out/*.bin`` are the outputs of the UNMODIFIED reference ``.m`` files, run from
  where they lie under /root/reference by ``oracle/minimat`` (the MATLAB-subset interpreter of this repository --
  neither MATLAB nor GNU Octave exists in the image) through the recipe ``tests/golden/make_octave_goldens.m`` on
  203 seeded packets; generator ``tests/golden/run_reference_recipe.py``, provenance (sha256 of every executed
  reference file) in ``octave_out/PROVENANCE.json``.  ``tests/test_octave_goldens.py`` holds this module, the C port
  and -- under ``-m gpu`` -- the CUDA path to them at 1e-12 (fields, RHS) / 1e-9 (trajectories); measured: this
  module equals them BIT FOR BIT on all twelve outputs.  The interpreter is generic MATLAB semantics, not a
  restatement of the path, and is itself pinned to numbers real MATLAB produced (``tests/test_minimat.py``: the
  unmodified ``qgsw_raytrace.m`` run under it prints MATLAB R2020b's log header character for character and lands
  within 2 ulps of the stored ``pv_time`` stream; the unmodified ``rsw/k2g.m`` reproduces ``rsw/matlab.mat``).
  The same recipe runs unchanged under real MATLAB / Octave (``tests/golden/make_octave_goldens.m``'s header) for
  anyone who wants the cross-check; its output would replace the committed files one for one.
* **parity unpinned** only at the MATLAB-builtin boundary ``ode23``: it is MathWorks code, not the reference's,
  so there is nothing of the reference's to execute; the restated controller is checked against scipy's RK23
  tableau, closed forms and MATLAB's documented step-size rules (``tests/test_oracle_kat.py``).  The known-answer
  tests derived from the reference's own scripts (SURVEY.md section 4, items 1-6) stay as a second net:
  grid-node identity of ``interpolate``, the closed-form Childress-Soward flow of
  ``ray_trace_sw/raytrace.m:31-37``, the zero-flow analytic trajectory, the direct trig-sum pattern
  of ``scratch/fourier_interpolate_test.m:92-136``, the ``g2k(k2g(.))`` round trip, and the
  Omega-drift bound of ``symplectic_full_fourier.m:54-57``.

Every function cites the reference file:line it follows (paths relative to /root/reference).
Array layout follows MATLAB: ``F[ix, iy]`` with x the first index; in memory the oracle keeps
numpy C-order arrays and converts explicitly where the C ABI wants column-major.
"""
from __future__ import annotations

import math
import numpy as np

# --------------------------------------------------------------------------------------------
# MATLAB numeric primitives (SURVEY.md Appendix A)
# --------------------------------------------------------------------------------------------

def matlab_mod(a, m):
    """MATLAB ``mod(a,m)`` for m>0: ``a - floor(a/m)*m`` in [0,m]; ``mod(-tiny,m)`` rounds to m.
    numpy's ``np.mod`` on floats (fmod + sign fix-up) produces the same doubles."""
    return np.mod(a, m)


def matlab_linspace(a, b, n):
    """MATLAB ``linspace(a,b,n)``: ``a + (0:n-1)*(b-a)/(n-1)`` with the end point forced to b
    (used by analysis/load_data.m:39)."""
    a = float(a); b = float(b)
    out = a + np.arange(n, dtype=np.float64) * (b - a) / (n - 1)
    out[-1] = b
    return out


def matlab_rand_stream(seed):
    """``rng(seed)`` = mt19937ar; ``rand`` yields the same 53-bit doubles as numpy's legacy
    RandomState (qgsw_raytrace.m:23, symplectic_full_fourier.m:11)."""
    return np.random.RandomState(seed)


def histcounts(w, edges):
    """``histcounts(w, edges)`` (analysis/load_data.m:47): bin i counts edges[i] <= w < edges[i+1],
    the last bin also includes w == edges[-1]; out-of-range and NaN values are dropped."""
    w = np.asarray(w, dtype=np.float64).ravel()
    edges = np.asarray(edges, dtype=np.float64)
    nb = len(edges) - 1
    counts = np.zeros(nb, dtype=np.uint64)
    ok = ~np.isnan(w) & (w >= edges[0]) & (w <= edges[-1])
    w = w[ok]
    idx = np.searchsorted(edges, w, side="right") - 1   # edges[idx] <= w < edges[idx+1]
    idx[w == edges[-1]] = nb - 1
    idx = idx[(idx >= 0) & (idx < nb)]
    np.add.at(counts, idx, 1)
    return counts


# --------------------------------------------------------------------------------------------
# Spectral <-> grid kit
# --------------------------------------------------------------------------------------------

def wavenumbers(nx):
    """``[kx_,ky_] = ndgrid(-kmax:kmax, 0:kmax)`` (SpectralScheme.m:12-13, qgsw_raytrace.m:18-20)."""
    kmax = nx // 2 - 1
    kx = np.arange(-kmax, kmax + 1, dtype=np.float64)[:, None]
    ky = np.arange(0, kmax + 1, dtype=np.float64)[None, :]
    kx_, ky_ = np.broadcast_arrays(kx, ky)
    return kx_.copy(), ky_.copy()


def g2k(fg):
    """qg_flow_ray_trace/g2k.m:5-9: ``fftshift(fft2(fg))/nx^2`` restricted to rows 2:end
    (kx=-kmax..kmax) and columns kmax+2:end (ky=0..kmax)."""
    nx = fg.shape[0]
    kmax = nx // 2 - 1
    fkt = np.fft.fftshift(np.fft.fft2(fg)) / nx**2
    return fkt[1:, kmax + 1:].copy()


def fulspec(fk):
    """qg_flow_ray_trace/fulspec.m:10-19: fill the lower half plane by conjugate symmetry,
    zero the Nyquist row/column, and conjugate-symmetrise the ky=0 column from its kx>0 half."""
    nkx, nky = fk.shape
    nx = nkx + 1
    kmax = nky - 1
    fkf = np.zeros((nx, nx), dtype=np.complex128)
    fup = fk.astype(np.complex128).copy()
    # fup(kmax:-1:1,1) = conj(fup(kmax+2:nkx,1))
    fup[kmax - 1::-1, 0] = np.conj(fup[kmax + 1:nkx, 0])
    # fdn = conj(fup(nkx:-1:1, nky:-1:2))
    fdn = np.conj(fup[::-1, nky - 1:0:-1])
    fkf[1:nx, nky:nx] = fup
    fkf[1:nx, 1:nky] = fdn
    return fkf


def k2g(fk):
    """qg_flow_ray_trace/k2g.m:5-6: ``nx^2*ifft2(ifftshift(fulspec(fk)))``.  MATLAB's ifft2 returns
    a real matrix for exactly conjugate-symmetric input except for Im F(0,0); numpy leaves ~1e-17
    imaginary residue, so the real part is taken (SURVEY.md Appendix A)."""
    nx = fk.shape[0] + 1
    return (nx**2 * np.fft.ifft2(np.fft.ifftshift(fulspec(fk)))).real


def symmetrise_ky0(fk):
    """The ky=0 treatment of fulspec.m:16 applied to a half-plane array: F(-kx,0) := conj F(kx,0),
    and Im F(0,0) dropped (it cannot contribute to the real field k2g returns)."""
    fk = np.array(fk, dtype=np.complex128)
    nkx = fk.shape[0]
    kmax = (nkx - 1) // 2
    fk[kmax - 1::-1, 0] = np.conj(fk[kmax + 1:nkx, 0])
    fk[kmax, 0] = fk[kmax, 0].real
    return fk


def velocity_planes_k(psik, kx_, ky_):
    """Spectral velocity and gradient planes from psi-hat:
    SpectralScheme.m:18-25 (= grid_U.m:3-9): u=-i ky psi, v=i kx psi, ux=i kx u, uy=i ky u, ..."""
    uk = -1j * ky_ * psik
    vk = 1j * kx_ * psik
    return [uk, vk, 1j * kx_ * uk, 1j * ky_ * uk, 1j * kx_ * vk, 1j * ky_ * vk]


def grid_U(qk, K_d2, K2, kx_, ky_, shear_strength=0.0):
    """qg_flow_ray_trace/grid_U.m:2-17: psi=-q/(K_d2+K2); six k2g's; mean shear added to u.
    Returns dict with keys u,v,ux,uy,vx,vy (the reference's struct field names)."""
    psik = -qk / (K_d2 + K2)
    uk, vk, ukx, uky, vkx, vky = velocity_planes_k(psik, kx_, ky_)
    return {"u": k2g(uk) + shear_strength, "v": k2g(vk), "ux": k2g(ukx), "uy": k2g(uky),
            "vx": k2g(vkx), "vy": k2g(vky)}


def grid_U_planes_k(qk, K_d2, K2, kx_, ky_, shear_strength=0.0):
    """Spectral-coefficient form of grid_U: the same six planes before k2g; the mean shear is the
    (kx,ky)=(0,0) coefficient of u (grid_U.m:11)."""
    psik = -qk / (K_d2 + K2)
    planes = velocity_planes_k(psik, kx_, ky_)
    kmax = (qk.shape[0] - 1) // 2
    planes[0] = planes[0].copy()
    planes[0][kmax, 0] += shear_strength
    return planes


# --------------------------------------------------------------------------------------------
# interpolate.m -- 6x6 Lagrange stencil (reference semantics of "field at packet")
# --------------------------------------------------------------------------------------------

IORD = 2
BUMP_LIVE = 1e-13     # ray_trace_sw/interpolate.m:13
BUMP_PAR = 1e-10      # interpolate_par.m:13
BUMP_QG = 1e-10       # qg_flow_ray_trace/interpolate.m:13 -- the reference keeps TWO copies of interpolate.m that differ in this one
#                       line; interpolate_U.m / odefun run next to the qg_flow_ray_trace copy (runqgsw_raytrace.sbatch:25-27 copies
#                       it into the run directory, qgsw_raytrace is started from there), SpectralScheme.m:8 puts ./ray_trace_sw/ in
#                       front.  Found by executing the drivers' nested odefun unmodified (tests/test_reference_locals.py): the two
#                       bumps differ by ~1e-10 of the field, 100 x the 1e-12 the RHS is held to.


def _lagrange_weights(a, bump):
    """interpolate.m:33-41: w_i = prod_{j != i, j=-2..3} (a - j + bump)/(j - i), multiply then
    divide, j ascending.  ``a`` is an array of fractional positions; returns (6, n)."""
    w = np.ones((2 * (IORD + 1),) + a.shape, dtype=np.float64)
    for i in range(-IORD, IORD + 2):
        for j in range(-IORD, IORD + 2):
            if i != j:
                w[i + IORD] = w[i + IORD] * (a - j + bump) / (j - i)
    return w


def interpolate(x, y, F, dx, dy, bump=BUMP_LIVE):
    """ray_trace_sw/interpolate.m:12-49 (vectorised over packets, same per-packet operation
    order): xl=mod(x/dx,nx); i0=1+floor(xl); ax=1+xl-i0; 36-term sum, i outer / j inner,
    term (wx_i*wy_j)*F(ig,jg); BOTH indices wrap with nx (interpolate.m:45-46)."""
    x = np.asarray(x, dtype=np.float64); y = np.asarray(y, dtype=np.float64)
    shp = x.shape
    x = x.ravel(); y = y.ravel()
    nx, ny = F.shape
    xl = matlab_mod(x / dx, nx)
    yl = matlab_mod(y / dy, ny)
    i0 = 1 + np.floor(xl)
    j0 = 1 + np.floor(yl)
    ax = 1 + xl - i0
    ay = 1 + yl - j0
    wx = _lagrange_weights(ax, bump)
    wy = _lagrange_weights(ay, bump)
    i0 = i0.astype(np.int64); j0 = j0.astype(np.int64)
    FI = np.zeros_like(x)
    for i in range(-IORD, IORD + 2):
        ig = np.mod(i0 + i - 1, nx)            # zero-based (reference: 1 + mod(...))
        for j in range(-IORD, IORD + 2):
            jg = np.mod(j0 + j - 1, nx)        # wraps with nx, as the reference does
            FI = FI + wx[i + IORD] * wy[j + IORD] * F[ig, jg]
    return FI.reshape(shp)


def interpolate_par(x, y, F, dx, dy):
    """interpolate_par.m:12-51: the same stencil with bump=1e-10."""
    return interpolate(x, y, F, dx, dy, bump=BUMP_PAR)


def interpolate_U(bf1, bf2, alpha, x, h, bump=BUMP_QG):
    """qg_flow_ray_trace/interpolate_U.m:1-24.  x: (Np,2).  Returns U (Np,2) and dict nablaU with
    u_x,u_y,v_x,v_y; linear blend (1-alpha)*F1 + alpha*F2 of twelve interpolations -- by the ``interpolate.m`` that sits
    next to it (``bump`` = 1e-10, see BUMP_QG); ``bump=BUMP_LIVE`` gives the same function bound to ray_trace_sw's copy."""
    xx = x[:, 0]; yy = x[:, 1]
    U1 = np.stack([interpolate(xx, yy, bf1["u"], h, h, bump), interpolate(xx, yy, bf1["v"], h, h, bump)], axis=1)
    U2 = np.stack([interpolate(xx, yy, bf2["u"], h, h, bump), interpolate(xx, yy, bf2["v"], h, h, bump)], axis=1)
    U = (1 - alpha) * U1 + alpha * U2
    nablaU = {}
    for name, key in (("u_x", "ux"), ("u_y", "uy"), ("v_x", "vx"), ("v_y", "vy")):
        g1 = interpolate(xx, yy, bf1[key], h, h, bump)
        g2 = interpolate(xx, yy, bf2[key], h, h, bump)
        nablaU[name] = (1 - alpha) * g1 + alpha * g2
    return U, nablaU


# --------------------------------------------------------------------------------------------
# Exact trig-sum evaluation (the SPECTRAL mode's oracle; SURVEY.md 7.0)
# --------------------------------------------------------------------------------------------

def spectral_eval(x, y, fk, dx, nx, dtype=np.longdouble):
    """Direct Fourier-series sum of a half-plane coefficient array at packet positions (pattern:
    scratch/fourier_interpolate_test.m:125-136, generalised to complex coefficients):

      F = sum_kx Fs(kx,0) e^{i kx tx} + 2 Re sum_{ky>=1} sum_kx F(kx,ky) e^{i(kx tx + ky ty)},
      tx = 2 pi xl/nx, xl = mod(x/dx, nx)   (the reduced coordinate of interpolate.m:21-22).

    Accumulates in ``dtype`` (long double by default) so the result is good to ~1e-17 relative."""
    x = np.asarray(x, dtype=np.float64).ravel(); y = np.asarray(y, dtype=np.float64).ravel()
    fk = symmetrise_ky0(fk)
    nkx, nky = fk.shape
    kmax = nky - 1
    xl = matlab_mod(x / dx, nx).astype(dtype)
    yl = matlab_mod(y / dx, nx).astype(dtype)
    two_pi = 2 * np.arccos(dtype(-1))
    tx = two_pi * xl / nx
    ty = two_pi * yl / nx
    kx = np.arange(-kmax, kmax + 1).astype(dtype)
    ky = np.arange(0, kmax + 1).astype(dtype)
    fr = fk.real.astype(dtype); fi = fk.imag.astype(dtype)
    wy = np.full(nky, 2, dtype=dtype); wy[0] = 1
    out = np.zeros(x.shape, dtype=dtype)
    # chunk over packets to bound memory
    step = max(1, 2_000_000 // (nkx * max(nky, 1)))
    for s in range(0, x.size, max(step, 16)):
        e = slice(s, s + max(step, 16))
        ax = np.outer(tx[e], kx)                      # (p, nkx)
        cx, sx = np.cos(ax), np.sin(ax)
        gr = cx @ fr - sx @ fi                        # Re sum_kx F e^{i kx tx}, (p, nky)
        gi = cx @ fi + sx @ fr
        ay = np.outer(ty[e], ky)
        cy, sy = np.cos(ay), np.sin(ay)
        out[e] = ((gr * cy - gi * sy) * wy).sum(axis=1)
    return out


def spectral_eval_planes(x, y, planes_k, dx, nx, dtype=np.longdouble):
    """Evaluate a list of coefficient planes; returns float64 array (nplanes, Np)."""
    return np.stack([spectral_eval(x, y, p, dx, nx, dtype).astype(np.float64) for p in planes_k])


# --------------------------------------------------------------------------------------------
# Schemes (SpectralScheme.m / RaytracingScheme.m)
# --------------------------------------------------------------------------------------------

class SpectralScheme:
    """SpectralScheme.m:6-68.  ``mode='lagrange'`` is the reference behaviour (gridded fields +
    interpolate); ``mode='spectral'`` evaluates the same coefficient planes by exact trig sum."""

    def __init__(self, L, nx, psi_field, mode="lagrange"):
        self.L = float(L); self.nx = int(nx); self.mode = mode
        kx_, ky_ = wavenumbers(nx)
        kappa = 1.0  # SpectralScheme multiplies by integer kx,ky (domain 2*pi), SpectralScheme.m:18-25
        psik = g2k(psi_field)
        self.psik = psik
        self.planes_k = velocity_planes_k(psik, kappa * kx_, kappa * ky_)
        self.psi_field = k2g(psik)
        names = ("u", "v", "u_x", "u_y", "v_x", "v_y")
        self.fields = {n: k2g(p) for n, p in zip(names, self.planes_k)}

    def _dx(self):
        return self.L / self.psi_field.shape[0]          # SpectralScheme.m:39,46,57

    def _eval(self, name, xx, yy):
        dx = self._dx()
        if self.mode == "lagrange":
            return interpolate(xx, yy, self.fields[name], dx, dx)
        idx = ("u", "v", "u_x", "u_y", "v_x", "v_y").index(name)
        return spectral_eval(xx, yy, self.planes_k[idx], dx, self.nx).astype(np.float64)

    def streamfunction(self, x, y, t=0):
        dx = self._dx()
        if self.mode == "lagrange":
            return interpolate(x, y, self.psi_field, dx, dx)
        return spectral_eval(x, y, self.psik, dx, self.nx).astype(np.float64).reshape(np.shape(x))

    def U(self, x, t=0):
        """x: (T,2,Np) as in the reference, or (Np,2).  SpectralScheme.m:45-54."""
        x = np.asarray(x, dtype=np.float64)
        if x.ndim == 2:
            xx, yy = x[:, 0], x[:, 1]
            return np.stack([self._eval("u", xx, yy), self._eval("v", xx, yy)], axis=1)
        xx = x[:, 0, :]; yy = x[:, 1, :]
        u = np.zeros_like(x)
        u[:, 0, :] = self._eval("u", xx.ravel(), yy.ravel()).reshape(xx.shape)
        u[:, 1, :] = self._eval("v", xx.ravel(), yy.ravel()).reshape(xx.shape)
        return u

    def grad_U(self, x, t=0):
        """SpectralScheme.m:56-68: dict of flat arrays u_x,u_y,v_x,v_y."""
        x = np.asarray(x, dtype=np.float64)
        if x.ndim == 2:
            xx, yy = x[:, 0], x[:, 1]
        else:
            xx = x[:, 0, :].ravel(); yy = x[:, 1, :].ravel()
        return {n: self._eval(n, xx, yy) for n in ("u_x", "u_y", "v_x", "v_y")}

    def grad_U_times_k(self, x, k, t=0):
        """RaytracingScheme.m:9-16: [(u_x k + v_x l), (u_y k + v_y l)], same shape as k."""
        g = self.grad_U(x, t)
        k = np.asarray(k, dtype=np.float64)
        out = np.zeros_like(k)
        if k.ndim == 2:
            kk, ll = k[:, 0], k[:, 1]
            out[:, 0] = g["u_x"] * kk + g["v_x"] * ll
            out[:, 1] = g["u_y"] * kk + g["v_y"] * ll
            return out
        kk = k[:, 0, :]; ll = k[:, 1, :]
        out[:, 0, :] = (g["u_x"] * kk.ravel() + g["v_x"] * ll.ravel()).reshape(kk.shape)
        out[:, 1, :] = (g["u_y"] * kk.ravel() + g["v_y"] * ll.ravel()).reshape(ll.shape)
        return out


    # RaytracingScheme.m:18-31 (inherited diagnostics)
    def vorticity(self, x, t=0):
        g = self.grad_U(x, t)
        return g["v_x"] - g["u_y"]

    def strain(self, x, t=0):
        g = self.grad_U(x, t)
        return np.sqrt((g["u_x"] - g["v_y"]) ** 2 + (g["v_x"] + g["u_y"]) ** 2)

    def okuboWeiss(self, x, t=0):
        """RaytracingScheme.m:28-31 calls ``obj.grad_U(x, k, t)`` with an undefined ``k`` (it errors in MATLAB);
        the formula on :30 is what is restated: D = v_y^2 + v_x*u_y."""
        g = self.grad_U(x, t)
        return g["v_y"] ** 2 + g["v_x"] * g["u_y"]


class DifferenceScheme:
    """DifferenceScheme.m:1-46: U and grad U by centred finite differences of an analytic streamfunction
    handle ``psi(x, y, t)`` with h = eps^(1/3).  Not on the packet path of any driver (the only call site is the
    commented hint in SW_zero_background_raytracing.m:22-23); restated because it is the reference's own
    independent check of SpectralScheme: both schemes must agree to the finite-difference error."""

    def __init__(self, stream):
        self.h = np.finfo(np.float64).eps ** (1.0 / 3.0)        # nthroot(eps, 3)
        self.psi = stream

    def streamfunction(self, x, y, t=0):
        return self.psi(x, y, t)

    def U(self, x, t=0):
        x = np.asarray(x, dtype=np.float64)
        xx, yy = (x[:, 0], x[:, 1]) if x.ndim == 2 else (x[:, 0, :], x[:, 1, :])
        h = self.h
        u = np.zeros_like(x)
        v_ = (self.psi(xx + h / 2, yy, t) - self.psi(xx - h / 2, yy, t)) / h
        u_ = -(self.psi(xx, yy + h / 2, t) - self.psi(xx, yy - h / 2, t)) / h
        if x.ndim == 2:
            u[:, 0], u[:, 1] = u_, v_
        else:
            u[:, 0, :], u[:, 1, :] = u_, v_
        return u

    def grad_U(self, x, t=0):
        x = np.asarray(x, dtype=np.float64)
        xx, yy = (x[:, 0], x[:, 1]) if x.ndim == 2 else (x[:, 0, :].ravel(), x[:, 1, :].ravel())
        h, p = self.h, self.psi
        v_x = (p(xx + h, yy, t) - 2 * p(xx, yy, t) + p(xx - h, yy, t)) / h / h
        u_y = -(p(xx, yy + h, t) - 2 * p(xx, yy, t) + p(xx, yy - h, t)) / h / h
        v_y = (p(xx + h / 2, yy + h / 2, t) + p(xx - h / 2, yy - h / 2, t) - p(xx - h / 2, yy + h / 2, t)
               - p(xx + h / 2, yy - h / 2, t)) / h / h
        return {"u_x": -v_y, "u_y": u_y, "v_x": v_x, "v_y": v_y}


class PlanesScheme:
    """A scheme defined directly by six coefficient planes (u,v,ux,uy,vx,vy) on a domain of side L
    (what grid_U builds for the qgsw drivers), evaluated either by k2g+interpolate or trig sum."""

    def __init__(self, L, nx, planes_k, mode="lagrange", planes_k2=None):
        self.L = float(L); self.nx = int(nx); self.mode = mode
        self.planes_k = [np.asarray(p, dtype=np.complex128) for p in planes_k]
        self.fields = [k2g(p) for p in self.planes_k] if mode == "lagrange" else None

    def eval6(self, x, y):
        dx = self.L / self.nx
        if self.mode == "lagrange":
            return np.stack([interpolate(x, y, F, dx, dx) for F in self.fields])
        return spectral_eval_planes(x, y, self.planes_k, dx, self.nx)

    def U(self, x, t=0):
        e = self.eval6(x[:, 0], x[:, 1])
        return np.stack([e[0], e[1]], axis=1)

    def grad_U_times_k(self, x, k, t=0):
        e = self.eval6(x[:, 0], x[:, 1])
        return np.stack([e[2] * k[:, 0] + e[4] * k[:, 1], e[3] * k[:, 0] + e[5] * k[:, 1]], axis=1)


# --------------------------------------------------------------------------------------------
# Integrators
# --------------------------------------------------------------------------------------------

def omega_of_k(k, l, f, gH):
    """ode_symplectic.m:10 / load_data.m:33: sqrt(f^2 + gH*(k^2+l^2))."""
    return np.sqrt(f * f + gH * (k * k + l * l))


def leapfrog_step(x, y, k, l, dt, f, gH, eval6):
    """One step of ode_symplectic.m:13-21,33-37 on flat arrays.  ``eval6(x,y)`` returns the six
    planes (u,v,ux,uy,vx,vy) at the packets.  phi1(dt/2): x += dt/2*gH*k/omega(k);
    phi2(dt): x += dt*U(x1), k -= dt*(gradU(x1))^T k (old k on the right); phi1(dt/2)."""
    h = dt / 2
    w = np.sqrt(f ** 2 + gH * (k * k + l * l))
    x1 = x + h * (gH * k / w)
    y1 = y + h * (gH * l / w)
    u, v, ux, uy, vx, vy = eval6(x1, y1)
    x2 = x1 + dt * u
    y2 = y1 + dt * v
    k2 = k - dt * (ux * k + vx * l)
    l2 = l - dt * (uy * k + vy * l)
    w = np.sqrt(f ** 2 + gH * (k2 * k2 + l2 * l2))
    x3 = x2 + h * (gH * k2 / w)
    y3 = y2 + h * (gH * l2 / w)
    return x3, y3, k2, l2


def ode_symplectic(x0, k0, dt, T, f, gH, scheme, save_stride=1):
    """ode_symplectic.m:1-37.  x0,k0: (1,2,Np).  Nsteps=floor(T/dt); rows 2..Nsteps hold the state
    after 1..Nsteps-1 leapfrog steps; t(i)=(i-1)dt.  ``save_stride`` thins the stored history
    (an extension: the reference stores every step, ode_symplectic.m:25-27)."""
    Nsteps = int(math.floor(T / dt))
    x0 = np.asarray(x0, dtype=np.float64); k0 = np.asarray(k0, dtype=np.float64)
    rows = list(range(0, Nsteps, save_stride))
    xs = np.zeros((len(rows),) + x0.shape[1:]); ks = np.zeros_like(xs); ts = np.zeros(len(rows))
    xs[0] = x0[0]; ks[0] = k0[0]
    x, y = x0[0, 0, :].copy(), x0[0, 1, :].copy()
    k, l = k0[0, 0, :].copy(), k0[0, 1, :].copy()

    def eval6(xx, yy):
        xa = np.stack([xx, yy], axis=1)
        U = scheme.U(xa)
        g = scheme.grad_U(xa)
        return U[:, 0], U[:, 1], g["u_x"], g["u_y"], g["v_x"], g["v_y"]

    r = 1
    for i in range(1, Nsteps):
        x, y, k, l = leapfrog_step(x, y, k, l, dt, f, gH, eval6)
        if i % save_stride == 0:
            xs[r, 0], xs[r, 1], ks[r, 0], ks[r, 1] = x, y, k, l
            ts[r] = i * dt
            r += 1
    return xs, ks, ts


def odefun_rhs(x, y, k, l, alpha, bf1, bf2, f, Cg, h, bump=BUMP_QG):
    """qgsw_raytrace.m:259-265 (same in qg2layersw_raytrace.m:298-304): RHS of the ode23 system.
    dxdt = U + Cg*k/sqrt(f^2+Cg^2|k|^2)  (note Cg, not Cg^2); dkdt = -(gradU)^T k."""
    U, nab = interpolate_U(bf1, bf2, alpha, np.stack([x, y], axis=1), h, bump)
    w = np.sqrt(f ** 2 + Cg ** 2 * (k * k + l * l))
    dxdt = U[:, 0] + Cg * k / w
    dydt = U[:, 1] + Cg * l / w
    dkdt = -(nab["u_x"] * k + nab["v_x"] * l)
    dldt = -(nab["u_y"] * k + nab["v_y"] * l)
    return dxdt, dydt, dkdt, dldt


def rhs_from_eval(e6, k, l, f, Cg):
    """The same RHS given the six evaluated planes (mode-independent part of odefun)."""
    u, v, ux, uy, vx, vy = e6
    w = np.sqrt(f ** 2 + Cg ** 2 * (k * k + l * l))
    return u + Cg * k / w, v + Cg * l / w, -(ux * k + vx * l), -(uy * k + vy * l)


def cg_sw(k, l, C0, f, U=None, H=None):
    """ray_trace_sw/cg_sw.m:15-31.  With H (grid, or per-packet point values) gH=C0^2*H and every
    output has H's shape.  Returns (Cx, Cy, omega, divC, gox, goy)."""
    gH = C0 ** 2 * H if H is not None else C0 ** 2
    K2 = k ** 2 + l ** 2
    omega = np.sqrt(f ** 2 + gH * K2)
    Cx = gH * k / omega
    Cy = gH * l / omega
    divC = gox = goy = None
    if U is not None and H is not None:
        divC = (k * f * U["v"] - l * f * U["u"] - Cx ** 2 - Cy ** 2) / omega
        gox = f * K2 * U["v"] / (2 * omega)
        goy = -f * K2 * U["u"] / (2 * omega)
    return Cx, Cy, omega, divC, gox, goy


def _rk4_linear_k(k, l, dt, uxi, uyi, vxi, vyi, oxi=0.0, oyi=0.0):
    """step_packet.m:65-78 / step_packet_xka.m:69-82: RK4 on (k,l) with a frozen matrix."""
    k1 = dt * (-uxi * k - vxi * l - oxi)
    l1 = dt * (-uyi * k - vyi * l - oyi)
    k2 = dt * (-uxi * (k + k1 / 2) - vxi * (l + l1 / 2) - oxi)
    l2 = dt * (-uyi * (k + k1 / 2) - vyi * (l + l1 / 2) - oyi)
    k3 = dt * (-uxi * (k + k2 / 2) - vxi * (l + l2 / 2) - oxi)
    l3 = dt * (-uyi * (k + k2 / 2) - vyi * (l + l2 / 2) - oyi)
    k4 = dt * (-uxi * (k + k3) - vxi * (l + l3) - oxi)
    l4 = dt * (-uyi * (k + k3) - vyi * (l + l3) - oyi)
    return k + (k1 + 2 * k2 + 2 * k3 + k4) / 6, l + (l1 + 2 * l2 + 2 * l3 + l4) / 6


def step_packet(P, U, GradU, C0, f, dx, dy, dt):
    """ray_trace_sw/step_packet.m:37-78 for ONE packet (scalars in dict P with x,y,k,l).
    The reference interpolates the grid ``U.u + C.x`` (scalar added to every node)."""
    Cx, Cy, *_ = cg_sw(P["k"], P["l"], C0, f)
    Fu = U["u"] + Cx; Fv = U["v"] + Cy
    ip = lambda xx, yy, F: float(interpolate(np.array([xx]), np.array([yy]), F, dx, dy)[0])
    x1 = dt * ip(P["x"], P["y"], Fu); y1 = dt * ip(P["x"], P["y"], Fv)
    x2 = dt * ip(P["x"] + x1 / 2, P["y"] + y1 / 2, Fu); y2 = dt * ip(P["x"] + x1 / 2, P["y"] + y1 / 2, Fv)
    x3 = dt * ip(P["x"] + x2 / 2, P["y"] + y2 / 2, Fu); y3 = dt * ip(P["x"] + x2 / 2, P["y"] + y2 / 2, Fv)
    x4 = dt * ip(P["x"] + x3, P["y"] + y3, Fu); y4 = dt * ip(P["x"] + x3, P["y"] + y3, Fv)
    out = {"x": P["x"] + (x1 + 2 * x2 + 2 * x3 + x4) / 6, "y": P["y"] + (y1 + 2 * y2 + 2 * y3 + y4) / 6}
    # gradients at the OLD position (step_packet.m:58-61)
    g = [ip(P["x"], P["y"], GradU[n]) for n in ("u_x", "u_y", "v_x", "v_y")]
    out["k"], out["l"] = _rk4_linear_k(P["k"], P["l"], dt, g[0], g[1], g[2], g[3])
    return out


def step_packet_xka(P, U, GradU, H, C0, f, dx, dy, dt):
    """ray_trace_sw/step_packet_xka.m:38-91 for ONE packet; cg_sw fields are whole grids."""
    Cx, Cy, om, divC, gox, goy = cg_sw(P["k"], P["l"], C0, f, U, H)
    Fu = U["u"] + Cx; Fv = U["v"] + Cy
    ip = lambda xx, yy, F: float(interpolate(np.array([xx]), np.array([yy]), F, dx, dy)[0])
    x1 = dt * ip(P["x"], P["y"], Fu); y1 = dt * ip(P["x"], P["y"], Fv)
    x2 = dt * ip(P["x"] + x1 / 2, P["y"] + y1 / 2, Fu); y2 = dt * ip(P["x"] + x1 / 2, P["y"] + y1 / 2, Fv)
    x3 = dt * ip(P["x"] + x2 / 2, P["y"] + y2 / 2, Fu); y3 = dt * ip(P["x"] + x2 / 2, P["y"] + y2 / 2, Fv)
    x4 = dt * ip(P["x"] + x3, P["y"] + y3, Fu); y4 = dt * ip(P["x"] + x3, P["y"] + y3, Fv)
    out = {"x": P["x"] + (x1 + 2 * x2 + 2 * x3 + x4) / 6, "y": P["y"] + (y1 + 2 * y2 + 2 * y3 + y4) / 6}
    # gradients, grad(omega), div C at the NEW position (step_packet_xka.m:59-65)
    g = [ip(out["x"], out["y"], GradU[n]) for n in ("u_x", "u_y", "v_x", "v_y")]
    oxi = ip(out["x"], out["y"], gox); oyi = ip(out["x"], out["y"], goy)
    dci = ip(out["x"], out["y"], divC)
    out["k"], out["l"] = _rk4_linear_k(P["k"], P["l"], dt, g[0], g[1], g[2], g[3], oxi, oyi)
    a = P["a"]
    a1 = dt * (-a * dci); a2 = dt * (-(a + a1 / 2) * dci); a3 = dt * (-(a + a2 / 2) * dci); a4 = dt * (-(a + a3) * dci)
    out["a"] = a + (a1 + 2 * a2 + 2 * a3 + a4) / 6
    return out


def rk4_step_batch(x, y, k, l, a, dt, C0, f, fields, dx, xka, mode="lagrange", planes_k=None, nx=None, eval_planes=None):
    """Vectorised-over-packets restatement of step_packet / step_packet_xka.

    mode='lagrange': identical arithmetic to the reference, but the per-packet scalar that the
    reference adds to every grid node (``U.u + C.x``) is added at the 36 stencil nodes only, i.e.
    sum_ij w_ij (F_ij + c) -- the same value the reference computes, without forming nx^2 temps.
    For xka the node-wise fields (C, divC, grad omega) are composed at the stencil nodes.
    mode='spectral': the continuous ray equations -- U,V,H and gradients evaluated by exact trig sum
    at the point and composed pointwise (SURVEY.md 7.2 'step_packet_xka composes fields ...').
    fields: dict u,v,u_x,u_y,v_x,v_y[,H] of grids (lagrange) ; planes_k: list of 6 or 7 coefficient
    planes (spectral; H plane is eta_g, H = 1 + eta_g is applied by putting 1 in its (0,0) mode).
    eval_planes: optional ``(x, y, planes) -> (len(planes), n)`` evaluator of the spectral mode, e.g. the C oracle's
    long-double sums (c_oracle.spectral_eval), which are fast enough for grids above 128^2; default spectral_eval here."""
    n = x.size
    K2 = k * k + l * l
    if mode == "lagrange":
        def ev(xx, yy, fn):
            return _stencil_apply(xx, yy, fields["u"].shape[0], dx, fn)
        if not xka:
            w0 = np.sqrt(f ** 2 + C0 ** 2 * K2)
            Cx = C0 ** 2 * k / w0; Cy = C0 ** 2 * l / w0
            fu = lambda ig, jg: fields["u"][ig, jg] + Cx
            fv = lambda ig, jg: fields["v"][ig, jg] + Cy
        else:
            def node(ig, jg):
                gH = C0 ** 2 * fields["H"][ig, jg]
                om = np.sqrt(f ** 2 + gH * K2)
                return gH, om
            def fu(ig, jg):
                gH, om = node(ig, jg); return fields["u"][ig, jg] + gH * k / om
            def fv(ig, jg):
                gH, om = node(ig, jg); return fields["v"][ig, jg] + gH * l / om
        x1 = dt * ev(x, y, fu); y1 = dt * ev(x, y, fv)
        x2 = dt * ev(x + x1 / 2, y + y1 / 2, fu); y2 = dt * ev(x + x1 / 2, y + y1 / 2, fv)
        x3 = dt * ev(x + x2 / 2, y + y2 / 2, fu); y3 = dt * ev(x + x2 / 2, y + y2 / 2, fv)
        x4 = dt * ev(x + x3, y + y3, fu); y4 = dt * ev(x + x3, y + y3, fv)
        xn = x + (x1 + 2 * x2 + 2 * x3 + x4) / 6
        yn = y + (y1 + 2 * y2 + 2 * y3 + y4) / 6
        gx, gy = (xn, yn) if xka else (x, y)
        g = [ev(gx, gy, (lambda ig, jg, nm=nm: fields[nm][ig, jg])) for nm in ("u_x", "u_y", "v_x", "v_y")]
        if xka:
            def f_ox(ig, jg):
                gH, om = node(ig, jg); return f * K2 * fields["v"][ig, jg] / (2 * om)
            def f_oy(ig, jg):
                gH, om = node(ig, jg); return -f * K2 * fields["u"][ig, jg] / (2 * om)
            def f_dc(ig, jg):
                gH, om = node(ig, jg)
                cx = gH * k / om; cy = gH * l / om
                return (k * f * fields["v"][ig, jg] - l * f * fields["u"][ig, jg] - cx ** 2 - cy ** 2) / om
            oxi = ev(xn, yn, f_ox); oyi = ev(xn, yn, f_oy); dci = ev(xn, yn, f_dc)
        else:
            oxi = oyi = 0.0; dci = None
    else:
        npl = len(planes_k)
        def e_all(xx, yy, idx):
            if eval_planes is not None:
                return list(eval_planes(xx, yy, [planes_k[i] for i in idx]))
            return [spectral_eval(xx, yy, planes_k[i], dx, nx).astype(np.float64) for i in idx]
        def vel(xx, yy):
            if not xka:
                u, v = e_all(xx, yy, (0, 1))
                w0 = np.sqrt(f ** 2 + C0 ** 2 * K2)
                return u + C0 ** 2 * k / w0, v + C0 ** 2 * l / w0
            u, v, Hh = e_all(xx, yy, (0, 1, 6))
            gH = C0 ** 2 * Hh; om = np.sqrt(f ** 2 + gH * K2)
            return u + gH * k / om, v + gH * l / om
        ux_, uy_ = vel(x, y); x1 = dt * ux_; y1 = dt * uy_
        ux_, uy_ = vel(x + x1 / 2, y + y1 / 2); x2 = dt * ux_; y2 = dt * uy_
        ux_, uy_ = vel(x + x2 / 2, y + y2 / 2); x3 = dt * ux_; y3 = dt * uy_
        ux_, uy_ = vel(x + x3, y + y3); x4 = dt * ux_; y4 = dt * uy_
        xn = x + (x1 + 2 * x2 + 2 * x3 + x4) / 6
        yn = y + (y1 + 2 * y2 + 2 * y3 + y4) / 6
        gx, gy = (xn, yn) if xka else (x, y)
        if xka:
            u, v, g0, g1, g2, g3, Hh = e_all(gx, gy, range(7))
            g = [g0, g1, g2, g3]
            gH = C0 ** 2 * Hh; om = np.sqrt(f ** 2 + gH * K2)
            cx = gH * k / om; cy = gH * l / om
            oxi = f * K2 * v / (2 * om); oyi = -f * K2 * u / (2 * om)
            dci = (k * f * v - l * f * u - cx ** 2 - cy ** 2) / om
        else:
            g = e_all(gx, gy, (2, 3, 4, 5)); oxi = oyi = 0.0; dci = None
    kn, ln = _rk4_linear_k(k, l, dt, g[0], g[1], g[2], g[3], oxi, oyi)
    an = a
    if xka:
        a1 = dt * (-a * dci); a2 = dt * (-(a + a1 / 2) * dci); a3 = dt * (-(a + a2 / 2) * dci); a4 = dt * (-(a + a3) * dci)
        an = a + (a1 + 2 * a2 + 2 * a3 + a4) / 6
    return xn, yn, kn, ln, an


def _stencil_apply(x, y, nx, dx, node_fn, bump=BUMP_LIVE):
    """interpolate.m:18-49 with the gridded field replaced by ``node_fn(ig,jg)`` (zero-based index
    arrays) evaluated at the 36 stencil nodes: sum_i sum_j (wx_i*wy_j)*node, i outer, j inner."""
    xl = matlab_mod(x / dx, nx); yl = matlab_mod(y / dx, nx)
    i0 = 1 + np.floor(xl); j0 = 1 + np.floor(yl)
    ax = 1 + xl - i0; ay = 1 + yl - j0
    wx = _lagrange_weights(ax, bump); wy = _lagrange_weights(ay, bump)
    i0 = i0.astype(np.int64); j0 = j0.astype(np.int64)
    FI = np.zeros_like(x)
    for i in range(-IORD, IORD + 2):
        ig = np.mod(i0 + i - 1, nx)
        for j in range(-IORD, IORD + 2):
            jg = np.mod(j0 + j - 1, nx)
            FI = FI + wx[i + IORD] * wy[j + IORD] * node_fn(ig, jg)
    return FI


# --------------------------------------------------------------------------------------------
# Driver-side restatements used to build test/bench inputs
# --------------------------------------------------------------------------------------------

def initial_q(X, Y, a_g, K_d2, rs, k_min=5, k_max=8, ring=False):
    """qgsw_raytrace.m:191-214.  The chained comparison on :202 ``k_min^2 < k^2+l^2 <= k_max^2``
    parses as ``(k_min^2 < K2) <= k_max^2`` = always true, so every |k|,|l|<=k_max mode is summed;
    ``ring=True`` gives the evidently intended annulus.  ``rs`` = RandomState (rng(146))."""
    q = np.zeros_like(X); U = np.zeros_like(X); V = np.zeros_like(X)
    n = 2 * k_max + 1
    phase = 2 * np.pi * rs.rand(n, n).T        # MATLAB fills column-major
    for k in range(-k_max, k_max + 1):
        for l in range(-k_max, k_max + 1):
            K2 = k * k + l * l
            if (not ring) or (k_min ** 2 < K2 <= k_max ** 2):
                wp = k * X + l * Y + phase[k + k_max, l + k_max]
                U = U - l * np.sin(wp)
                V = V + k * np.sin(wp)
                q = q - (K_d2 + K2) * np.cos(wp)
    speed2 = U ** 2 + V ** 2
    return a_g / np.sqrt(speed2.max()) * q


def init_packets(Npackets, L, radius, rs):
    """qgsw_raytrace.m:54-60 / symplectic_full_fourier.m:22-28: k on a ring, x ~ L*rand(1,2)-L/2
    drawn per packet (x then y interleaved)."""
    i = np.arange(1, Npackets + 1)
    k = radius * np.cos(2 * np.pi * i / Npackets)
    l = radius * np.sin(2 * np.pi * i / Npackets)
    r = rs.rand(Npackets, 2)
    return L * r[:, 0] - L / 2, L * r[:, 1] - L / 2, k, l


def wrap_position(x, L):
    """qgsw_raytrace.m:160: mod(x + L/2, L) - L/2 (applied only when saving)."""
    return matlab_mod(x + L / 2, L) - L / 2


def omega_histogram(k, l, f, Cg, edges):
    """analysis/load_data.m:33,38-49: omega=sqrt(f^2+Cg^2 K^2) -> histcounts; energy=centre*count."""
    w = np.sqrt(f ** 2 + Cg ** 2 * (k * k + l * l))
    counts = histcounts(w, edges)
    centre = (edges[1:] + edges[:-1]) / 2
    return counts, centre * counts.astype(np.float64)


def childress_soward(nx, L, U0, km, a):
    """ray_trace_sw/raytrace.m:25-37 closed-form flow on the grid x=0:dx:dx*(nx-1) (ndgrid).  The
    reference's line 36 uses ``*`` (matrix product) instead of ``.*`` in v_x; the elementwise form
    (the evident intent, and equal to it when a=0) is used here."""
    dx = L / nx
    x = np.arange(nx) * dx
    x_, y_ = np.meshgrid(x, x, indexing="ij")
    s, c = np.sin, np.cos
    psi = U0 / km * (s(km * x_) * s(km * y_) + a * c(km * x_) * c(km * y_))
    U = {"u": -U0 * (s(km * x_) * c(km * y_) - a * c(km * x_) * s(km * y_)),
         "v": U0 * (c(km * x_) * s(km * y_) - a * s(km * x_) * c(km * y_))}
    G = {"u_x": -km * U0 * (c(km * x_) * c(km * y_) + a * s(km * x_) * s(km * y_)),
         "u_y": km * U0 * (s(km * x_) * s(km * y_) + a * c(km * x_) * c(km * y_)),
         "v_x": -km * U0 * (s(km * x_) * s(km * y_) + a * c(km * x_) * c(km * y_)),
         "v_y": km * U0 * (c(km * x_) * c(km * y_) + a * s(km * x_) * s(km * y_))}
    return psi, U, G


def childress_soward_point(x, y, U0, km, a):
    """The same closed form at arbitrary points (u,v,u_x,u_y,v_x,v_y)."""
    s, c = np.sin, np.cos
    return np.stack([-U0 * (s(km * x) * c(km * y) - a * c(km * x) * s(km * y)),
                     U0 * (c(km * x) * s(km * y) - a * s(km * x) * c(km * y)),
                     -km * U0 * (c(km * x) * c(km * y) + a * s(km * x) * s(km * y)),
                     km * U0 * (s(km * x) * s(km * y) + a * c(km * x) * c(km * y)),
                     -km * U0 * (s(km * x) * s(km * y) + a * c(km * x) * c(km * y)),
                     km * U0 * (c(km * x) * c(km * y) + a * s(km * x) * s(km * y))])


# --------------------------------------------------------------------------------------------
# ode23 (MATLAB builtin; un-vendored third-party arithmetic, MATLAB R2020b per run.log:4)
# --------------------------------------------------------------------------------------------

def ode23(odefun, tspan, y0, rtol=1e-3, atol=1e-6):
    """Restatement of the published algorithm behind MATLAB's ``ode23`` as the reference calls it
    (``[~,Y] = ode23(ray_ode, [0 dt], y0)``, qgsw_raytrace.m:149): the Bogacki-Shampine 3(2) pair with
    FSAL and the step-size controller described in Shampine & Reichelt, "The MATLAB ODE Suite" (1997):
    A = [1/2 3/4 1], B = [1/2 0 2/9; 0 3/4 1/3; 0 0 4/9], E = [-5/72 1/12 1/9 -1/8], pow = 1/3,
    threshold = atol/rtol, hmax = 0.1*|tf-t0|, err = |h| * ||(f*E) ./ max(|y|,|ynew|,thr)||_inf,
    rejection factor max(0.5, 0.8 (rtol/err)^pow) (then 0.5), growth 1/(1.25 (err/rtol)^pow) capped at 5.
    PARITY UNPINNED: MATLAB is proprietary and absent; no reference test stores an ode23 output (the
    tableau and the dense-output polynomial are cross-checked against scipy's independent RK23 in
    tests/test_oracle_kat.py).
    ``tspan = [t0 tf]`` returns (y_final, stats).  A longer ``tspan`` (SW_zero_background_raytracing.m:73-78)
    returns (Y, stats) with one row per requested time: the steps are chosen exactly as before and the
    rows come from the cubic dense output ``ntrp23`` (BI = [1 -4/3 5/9; 0 1 -2/3; 0 4/3 -8/9; 0 -1 1]),
    or ``ynew`` itself where an output time coincides with a step end."""
    tspan = np.asarray(tspan, dtype=np.float64)
    t0, tfinal = float(tspan[0]), float(tspan[-1])
    dense = tspan.size > 2
    y = np.array(y0, dtype=np.float64)
    if dense:
        Y = np.zeros((tspan.size, y.size)); Y[0] = y; nxt = 1
    pw = 1.0 / 3.0
    threshold = atol / rtol
    hmax = min(abs(tfinal - t0), abs(0.1 * (tfinal - t0)))
    t = t0
    f1 = odefun(t, y)
    nfevals = 1
    hmin = 16 * np.spacing(abs(t))
    # MATLAB (odearguments / ode23): htspan = |tspan(2) - tspan(1)|, absh = min(hmax, htspan) -- for a dense tspan the FIRST
    # output interval, not the whole span, bounds the initial step
    absh = min(hmax, abs(float(tspan[1]) - float(tspan[0])))
    rh = np.max(np.abs(f1) / np.maximum(np.abs(y), threshold)) / (0.8 * rtol ** pw)
    if absh * rh > 1:
        absh = 1 / rh
    absh = max(absh, hmin)
    nsteps = nfailed = 0
    done = False
    while not done:
        hmin = 16 * np.spacing(abs(t))
        absh = min(hmax, max(hmin, absh))
        h = absh
        if 1.1 * absh >= abs(tfinal - t):
            h = tfinal - t; absh = abs(h); done = True
        nofailed = True
        while True:
            f2 = odefun(t + 0.5 * h, y + f1 * (h * 0.5))
            f3 = odefun(t + 0.75 * h, y + f2 * (h * 0.75))
            tnew = tfinal if done else t + h
            ynew = y + (f1 * (h * (2.0 / 9.0)) + f2 * (h * (1.0 / 3.0)) + f3 * (h * (4.0 / 9.0)))      # y + f*hB(:,3), hB = h*B
            f4 = odefun(tnew, ynew)
            nfevals += 3
            fE = f1 * (-5 / 72) + f2 * (1 / 12) + f3 * (1 / 9) + f4 * (-1 / 8)
            err = absh * np.max(np.abs(fE) / np.maximum(np.maximum(np.abs(y), np.abs(ynew)), threshold))
            if not (err <= rtol):
                nfailed += 1
                if absh <= hmin:
                    raise RuntimeError("ode23: step size below hmin")
                if nofailed:
                    nofailed = False
                    absh = max(hmin, absh * max(0.5, 0.8 * (rtol / err) ** pw))
                else:
                    absh = max(hmin, 0.5 * absh)
                h = absh; done = False
            else:
                break
        nsteps += 1
        if dense:
            while nxt < tspan.size and tnew - tspan[nxt] >= 0:
                if tspan[nxt] == tnew:
                    Y[nxt] = ynew
                else:
                    sfrac = (tspan[nxt] - t) / h
                    s2, s3 = sfrac * sfrac, sfrac * sfrac * sfrac
                    Y[nxt] = y + (f1 * (h * (sfrac - 4.0 / 3.0 * s2 + 5.0 / 9.0 * s3)) + f2 * (h * (s2 - 2.0 / 3.0 * s3))
                                  + f3 * (h * (4.0 / 3.0 * s2 - 8.0 / 9.0 * s3)) + f4 * (h * (-s2 + s3)))
                nxt += 1
        if nofailed:
            temp = 1.25 * (err / rtol) ** pw
            absh = absh / temp if temp > 0.2 else 5.0 * absh
        t = tnew; y = ynew; f1 = f4
    stats = {"nsteps": nsteps, "nfailed": nfailed, "nfevals": nfevals, "t": t}
    return (Y, stats) if dense else (y, stats)


def generate_raytracing_ode(bf1, bf2, Npackets, f, Cg, tmax, h, eval6=None, bump=BUMP_QG):
    """qgsw_raytrace.m:258-268: odefun(t, y) on y = [x; y; k; l].  ``eval6(x, y, alpha)`` overrides the
    Lagrange interpolate_U evaluation (used for the SPECTRAL mode oracle)."""
    n = Npackets

    def odefun(t, y):
        x, yy, k, l = y[0:n], y[n:2 * n], y[2 * n:3 * n], y[3 * n:4 * n]
        if eval6 is None:
            d = odefun_rhs(x, yy, k, l, t / tmax, bf1, bf2, f, Cg, h, bump)
        else:
            d = rhs_from_eval(eval6(x, yy, t / tmax), k, l, f, Cg)
        return np.concatenate(d)

    return odefun


# --------------------------------------------------------------------------------------------
# One-layer QG flow solver of the drivers (producer of the background-flow frames)
# --------------------------------------------------------------------------------------------

def qg_filter(kx_, ky_, dx):
    """qgsw_raytrace.m:222-230: exponential cutoff filter Ef."""
    Ef = np.ones_like(kx_)
    kstar = np.sqrt((kx_ * dx) ** 2 + (ky_ * dx) ** 2)
    kc = 0.75 * np.pi
    const = np.log(1e-15) / (0.25 * np.pi) ** 4
    res = np.exp(const * (kstar - kc) ** 4)
    Ef[kstar >= kc] = res[kstar >= kc]
    return Ef


def qg_inertial_ring(force_strength, K2, f, Cg):
    """qgsw_raytrace.m:216-220"""
    om = np.sqrt(f ** 2 + Cg ** 2 * K2)
    forces = np.zeros_like(K2)
    forces[(0.9 * f < om) & (om < 1.1 * f)] = force_strength
    return forces


def qg_update(qk, K2, K_d2, beta, r_drag, surface_forces, kx_, ky_):
    """qgsw_raytrace.m:270-286 ``update`` (including ``r_drag * K2`` exactly as written on :285)."""
    psik = -qk / (K_d2 + K2)
    psikx = 1j * kx_ * psik; psiky = 1j * ky_ * psik
    qkx = 1j * kx_ * qk; qky = 1j * ky_ * qk
    J = k2g(psikx) * k2g(qky) - k2g(psiky) * k2g(qkx)
    return g2k(J) - beta * psikx + r_drag * K2 + surface_forces


def qg_run(qk, nsteps, dt, nx, L, K_d2, f, Cg, beta=0.0, r_drag=0.1, force_strength=0.1):
    """qgsw_raytrace.m:111-137: Euler / AB2 start-up then AB3, filter after every step."""
    kx_, ky_ = wavenumbers(nx)
    kap = 2 * np.pi / L
    kx_, ky_ = kap * kx_, kap * ky_
    K2 = kx_ ** 2 + ky_ ** 2
    Ef = qg_filter(kx_, ky_, L / nx)
    forces = qg_inertial_ring(force_strength, K2, f, Cg)
    Qm = [np.zeros_like(qk), np.zeros_like(qk)]
    qk = np.array(qk, dtype=np.complex128)
    for step in range(1, nsteps + 1):
        Qn = qg_update(qk, K2, K_d2, beta, r_drag, forces, kx_, ky_)
        if step == 1:
            dq = dt * Qn
        elif step == 2:
            dq = dt / 2 * (3 * Qn - Qm[0])
        else:
            dq = dt / 12 * (23 * Qn - 16 * Qm[0] + 5 * Qm[1])
        Qm[1] = Qm[0]; Qm[0] = Qn
        qk = Ef * (qk + dq)
    return qk


# --------------------------------------------------------------------------------------------
# The scripts BASELINE.json's configs name, restated (checkers for swraytracing_b200/drivers.py)
# --------------------------------------------------------------------------------------------

def childress_soward_as_written(nx, L, U0, km, a):
    """ray_trace_sw/raytrace.m:31-37 literally: line 36 reads ``a*cos(km*x_)*cos(km*y_)`` -- a MATRIX
    product -- so the reference's v_x differs from the closed form when a ~= 0 (``childress_soward``
    above is the intended element-wise form)."""
    psi, U, G = childress_soward(nx, L, U0, km, a)
    dx = L / nx
    x = np.arange(nx) * dx
    x_, y_ = np.meshgrid(x, x, indexing="ij")
    G = dict(G)
    G["v_x"] = -km * U0 * (np.sin(km * x_) * np.sin(km * y_) + (a * np.cos(km * x_)) @ np.cos(km * y_))
    return psi, U, G


def raytrace_driver(C0=1.0, Fr=0.1, f=4.0, a=0.25, np_=5, nx=256, nsteps=None, seed=5489):
    """ray_trace_sw/raytrace.m:1-54 with the packet-major loops kept (one packet at a time through
    ``step_packet``).  ``seed`` 5489 = MATLAB's start-up mt19937ar state (no rng call in the script);
    ``rand*L`` is drawn x then y per packet (:45-46).  Returns x,y,k,l histories (np, nsteps)."""
    U0 = Fr; L = 2 * np.pi
    kd = f / C0 ** 2; km = kd; ki = km * 10
    dx = L / nx
    dt = 0.3 * dx / max(C0, U0)
    Tend = 1 / (f * Fr ** 2)
    nsteps = int(round(Tend / dt)) if nsteps is None else int(nsteps)
    _, U, GradU = childress_soward_as_written(nx, L, U0, km, a)
    rs = matlab_rand_stream(seed)
    hist = {n: np.zeros((np_, nsteps)) for n in ("x", "y", "k", "l")}
    for i in range(1, np_ + 1):
        hist["x"][i - 1, 0] = rs.rand() * L
        hist["y"][i - 1, 0] = rs.rand() * L
        hist["k"][i - 1, 0] = ki * np.cos(2 * np.pi * i / np_)
        hist["l"][i - 1, 0] = ki * np.sin(2 * np.pi * i / np_)
    for i in range(np_):
        for j in range(1, nsteps):
            P = {n: hist[n][i, j - 1] for n in hist}
            out = step_packet(P, U, GradU, C0, f, dx, dx, dt)
            for n in hist:
                hist[n][i, j] = out[n]
    return hist, dt, nsteps


def geostrophic_fields(S, f, Cg):
    """ray_trace_sw/raytrace_sw.m:14-52: geostrophic mode of S(:,:,1:3) = [u,v,eta] and its gradients."""
    nx = S.shape[0]
    kx_, ky_ = wavenumbers(nx)
    K2_ = kx_ ** 2 + ky_ ** 2
    gH0 = Cg ** 2
    sig2_ = f ** 2 + gH0 * K2_
    uk, vk, etak = g2k(S[:, :, 0]), g2k(S[:, :, 1]), g2k(S[:, :, 2])
    zetak = 1j * (kx_ * vk - ky_ * uk)
    etagk = (f * etak - zetak) * f / sig2_
    ugk = -1j * ky_ * (gH0 / f * etagk)
    vgk = 1j * kx_ * (gH0 / f * etagk)
    H = 1 + k2g(etagk)
    U = {"u": k2g(ugk), "v": k2g(vgk)}
    GradU = {"u_x": k2g(1j * kx_ * ugk), "u_y": k2g(1j * ky_ * ugk), "v_x": k2g(1j * kx_ * vgk), "v_y": k2g(1j * ky_ * vgk)}
    return U, GradU, H


def raytrace_sw_driver(S, f, Cg, np_=10, nsteps=None, seed=5489):
    """ray_trace_sw/raytrace_sw.m:80-130 (packet-major loops, ``step_packet_xka`` one packet at a time)."""
    nx = S.shape[0]
    C0 = Cg
    U, GradU, H = geostrophic_fields(S, f, Cg)
    L = 2 * np.pi
    kd = f / C0; ki = kd * 10
    U0 = float(np.sqrt(U["u"] ** 2 + U["v"] ** 2).max())
    Fr = U0 / C0
    dx = L / nx
    dt = 0.3 * dx / max(C0, U0)
    if nsteps is None:
        nsteps = int(round(20 / (f * Fr ** 2) / dt))
    rs = matlab_rand_stream(seed)
    hist = {n: np.zeros((np_, nsteps)) for n in ("x", "y", "k", "l", "a")}
    for i in range(1, np_ + 1):
        hist["x"][i - 1, 0] = rs.rand() * L
        hist["y"][i - 1, 0] = rs.rand() * L
        hist["k"][i - 1, 0] = ki * np.cos(2 * np.pi * i / np_)
        hist["l"][i - 1, 0] = ki * np.sin(2 * np.pi * i / np_)
        hist["a"][i - 1, 0] = 1.0
    for i in range(np_):
        for j in range(1, nsteps):
            P = {n: hist[n][i, j - 1] for n in hist}
            out = step_packet_xka(P, U, GradU, H, C0, f, dx, dx, dt)
            for n in hist:
                hist[n][i, j] = out[n]
    return hist, {"dt": dt, "nsteps": nsteps, "U0": U0, "Fr": Fr, "U": U, "GradU": GradU, "H": H}


def frozen_flow_setup(q, nx, f, Cg, Nparticles, grid_lo, mode="lagrange", seed=123):
    """symplectic_full_fourier.m:5-38 / SW_zero_background_raytracing.m:6-50: scheme from a PV frame, ring
    of packets (rng(123)), U0 = max speed over the nx^2 points of ``meshgrid(linspace(lo, lo+L, nx))``."""
    L = 2 * np.pi
    K_d2 = f / Cg
    kx_, ky_ = wavenumbers(nx)
    K2 = kx_ ** 2 + ky_ ** 2
    rs = matlab_rand_stream(seed)
    X = matlab_linspace(grid_lo, grid_lo + L, nx)
    XX, YY = np.meshgrid(X, X)
    scheme = SpectralScheme(L, nx, k2g(-g2k(q) / (K_d2 + K2)), mode=mode)
    x = np.zeros((1, 2, Nparticles)); k = np.zeros((1, 2, Nparticles))
    for i in range(1, Nparticles + 1):
        k[0, :, i - 1] = 3 * np.array([np.cos(2 * np.pi * i / Nparticles), np.sin(2 * np.pi * i / Nparticles)])
        x[0, :, i - 1] = L * rs.rand(2) - L / 2
    U = scheme.U(np.stack([XX.ravel(order="F"), YY.ravel(order="F")], axis=1))
    U0 = float(np.sqrt((U ** 2).sum(axis=1)).max())
    gH = Cg ** 2
    return L, gH, scheme, x, k, U0, U0 / Cg, 0.1 * (L / nx) / max(Cg, U0)


def omega_abs_history(scheme, x, k, f, gH):
    """omega(k,f,gH) + dot(scheme.U(x), k, 2) (symplectic_full_fourier.m:41,55,62-64)"""
    return np.sqrt(f * f + gH * (k ** 2).sum(axis=1)) + (scheme.U(x) * k).sum(axis=1)


def symplectic_full_fourier_driver(q, nx, f, Cg, Nparticles=10, Tend=None, mode="lagrange", seed=123):
    """symplectic_full_fourier.m:1-60 from the PV frame on."""
    L, gH, scheme, x, k, U0, Fr, dt = frozen_flow_setup(q, nx, f, Cg, Nparticles, 0.0, mode, seed)
    Tend = 10 / (f * Fr ** 2) if Tend is None else Tend
    Omega_0 = omega_abs_history(scheme, x, k, f, gH)
    sx, sk, st = ode_symplectic(x, k, dt, Tend, f, gH, scheme)
    err = (omega_abs_history(scheme, sx, sk, f, gH) - Omega_0) / Omega_0
    return {"solver_x": sx, "solver_k": sk, "solver_t": st, "solver_error": err, "U0": U0, "Fr": Fr, "dt": dt, "Tend": Tend}


def sw_zero_background_driver(q, nx, f, Cg, Nparticles=10, Tend=None, rtol=1e-6, atol=1e-7, mode="lagrange", seed=123):
    """SW_zero_background_raytracing.m:1-132 from the PV frame on: ode23 with output at dt*(0:Nsteps),
    RHS dx/dt = U + gH k/omega, dk/dt = -(grad U)^T k (:134-145,182-184)."""
    L, gH, scheme, x, k, U0, Fr, dt = frozen_flow_setup(q, nx, f, Cg, Nparticles, -np.pi, mode, seed)
    Tend = 1 / (f * Fr ** 2) if Tend is None else Tend
    Nsteps = int(math.floor(Tend / dt))
    n = Nparticles

    def odefun(t, y):
        xa = np.stack([y[0:n], y[n:2 * n]], axis=1)
        ka = np.stack([y[2 * n:3 * n], y[3 * n:4 * n]], axis=1)
        cg = gH * ka / np.sqrt(f * f + gH * (ka ** 2).sum(axis=1))[:, None]
        dx = scheme.U(xa) + cg
        dk = -scheme.grad_U_times_k(xa, ka)
        return np.concatenate([dx[:, 0], dx[:, 1], dk[:, 0], dk[:, 1]])

    y0 = np.concatenate([x[0, 0], x[0, 1], k[0, 0], k[0, 1]])
    t_hist = dt * np.arange(0, Nsteps + 1)
    Y, stats = ode23(odefun, t_hist, y0, rtol=rtol, atol=atol)
    sx = np.stack([Y[:, 0:n], Y[:, n:2 * n]], axis=1)
    sk = np.stack([Y[:, 2 * n:3 * n], Y[:, 3 * n:4 * n]], axis=1)
    Omega_0 = omega_abs_history(scheme, x, k, f, gH)[0]
    err = (omega_abs_history(scheme, sx, sk, f, gH) - Omega_0) / Omega_0
    return {"t_hist": t_hist, "solver_x": sx, "solver_k": sk, "solver_error": err, "U0": U0, "Fr": Fr, "dt": dt, "Nsteps": Nsteps,
            "stats": stats}


# --------------------------------------------------------------------------------------------
# Two-layer QG solver and driver loop of qg2layersw_raytrace.m
# --------------------------------------------------------------------------------------------

def qg2_operators(kx_, ky_, K_d2, beta, shear_strength, r, nu, alpha):
    """qg2layersw_raytrace.m:136-150: B (2,2,nkx,nky), factor_L, and its page-wise eigendecomposition
    ``[LV,LD] = pageeig(factor_L); LV1 = pageinv(LV)`` (numpy.linalg.eig per page; eigenvector scaling and
    order are arbitrary in both and cancel in V exp(D t) V^-1)."""
    K2 = kx_ ** 2 + ky_ ** 2
    F = K_d2 / 2
    B = np.zeros((2, 2) + K2.shape)
    B[0, 0] = -F - K2; B[0, 1] = -F; B[1, 0] = -F; B[1, 1] = -F - K2
    detB = K2 * (K2 + 2 * F)
    with np.errstate(divide="ignore"):
        detB = np.where(K2 == 0, np.inf, detB)
    B = B / detB
    diffusion_factor = (nu * K2 ** alpha + r) * K2 - 1j * kx_ * beta
    diffusion_terms = B * diffusion_factor
    shear_factor = 1j * kx_ * shear_strength
    M = np.einsum("ij,jkab->ikab", np.array([[-1.0, 0.0], [0.0, 1.0]]), np.eye(2)[:, :, None, None] + 2 * F * B)
    factor_L = shear_factor * M + diffusion_terms
    pages = np.moveaxis(factor_L, (0, 1), (2, 3))                      # (nkx, nky, 2, 2)
    LD, LV = np.linalg.eig(pages)
    LV1 = np.linalg.inv(LV)
    return B, factor_L, LV, LD, LV1


def qg2_expL(LV, LD, LV1, t):
    """pagemtimes(pagemtimes(LV, diag_exp(LD, t)), LV1) (:149-150,341-343) -> (2,2,nkx,nky)"""
    E = np.einsum("abij,abj,abjk->abik", LV, np.exp(t * LD), LV1)
    return np.moveaxis(E, (2, 3), (0, 1))


def mmult3(A, x):
    """qg2layersw_raytrace.m:333-338: y(:,:,i) = A(i,1,:,:).*x(:,:,1) + A(i,2,:,:).*x(:,:,2); x: (nkx,nky,2)"""
    return np.stack([A[i, 0] * x[:, :, 0] + A[i, 1] * x[:, :, 1] for i in range(2)], axis=2)


def qg2_update(qk, B, kx_, ky_):
    """qg2layersw_raytrace.m:309-323"""
    psik = mmult3(B, qk)
    out = []
    for i in range(2):
        psix = k2g(1j * kx_ * psik[:, :, i]); psiy = k2g(1j * ky_ * psik[:, :, i])
        qx = k2g(1j * kx_ * qk[:, :, i]); qy = k2g(1j * ky_ * qk[:, :, i])
        out.append(g2k(psix * qy - psiy * qx))
    return np.stack(out, axis=2)


def qg2_max_speed(qk, K_d2, K2, kx_, ky_, shear_strength):
    """:155-157: grid_U applied to the 3-D qk (one-layer inversion per layer, shear added to u), max speed"""
    m = 0.0
    for i in range(2):
        flow = grid_U(qk[:, :, i], K_d2, K2, kx_, ky_, shear_strength)
        m = max(m, float((flow["u"] ** 2 + flow["v"] ** 2).max()))
    return math.sqrt(m)


def qg2layersw_driver(nx, Npackets, near_inertial_factor, T_Fr_days, packet_delay_Fr_days, U_g, f, Cg, max_steps, k_max=30,
                      seed=5, eval_mode="lagrange"):
    """qg2layersw_raytrace.m:12-196 without the I/O and plotting: returns the state after ``max_steps`` passes of
    the while loop.  ``eval_mode``: 'lagrange' (interpolate_U, the reference) or 'spectral' (exact trig sum of the
    same six planes, the oracle of the SPECTRAL product mode)."""
    L = 20.0
    dx = L / nx
    xg = matlab_linspace(-L / 2, L / 2, nx)
    X, Y = np.meshgrid(xg, xg, indexing="ij")
    kx_, ky_ = wavenumbers(nx)
    kx_ = kx_ * (2 * np.pi / L); ky_ = ky_ * (2 * np.pi / L)
    K2 = kx_ ** 2 + ky_ ** 2
    rs = matlab_rand_stream(seed)
    beta = 0.0; K_d2 = f / Cg; shear_strength = 0.5
    T_Fr = T_Fr_days / f
    packet_delay_steps = (packet_delay_Fr_days / f) / f
    CFL_fraction = 0.25; alpha = 4; r = 0.4; nutune = 0.1
    q1 = initial_q(X, Y, U_g, K_d2, rs, k_min=10, k_max=k_max)
    qk = np.stack([g2k(q1), g2k(-q1)], axis=2)
    wf = math.sqrt((near_inertial_factor ** 2 - 1) * f ** 2 / Cg ** 2)
    i = np.arange(1, Npackets + 1)
    pk = wf * np.cos(2 * np.pi * i / Npackets); pl = wf * np.sin(2 * np.pi * i / Npackets)
    rr = rs.rand(Npackets, 2)
    px, py = L * rr[:, 0] - L / 2, L * rr[:, 1] - L / 2
    U0 = qg2_max_speed(qk, K_d2, K2, kx_, ky_, shear_strength)
    Fr = U0 / Cg
    T = T_Fr / Fr ** 2
    dt = CFL_fraction * dx / U0
    nu = nutune * dx ** (2 * alpha)
    B, _, LV, LD, LV1 = qg2_operators(kx_, ky_, K_d2, beta, shear_strength, r, nu, alpha)
    expLdt = qg2_expL(LV, LD, LV1, dt); expL2dt = qg2_expL(LV, LD, LV1, 2 * dt)
    Qm = [np.zeros_like(qk), np.zeros_like(qk)]
    t = 0.0; step = 0
    stats = {"packet_steps": 0, "ode23_steps": 0, "ode23_failed": 0, "dt_changes": 0}
    while t <= T and step < max_steps:
        step += 1
        U0 = qg2_max_speed(qk, K_d2, K2, kx_, ky_, shear_strength)
        CFL_condition = CFL_fraction * dx / U0
        if CFL_condition < dt or dt < CFL_condition / 4:
            dt = CFL_fraction / 2 * dx / U0
            stats["dt_changes"] += 1
            expLdt = qg2_expL(LV, LD, LV1, dt); expL2dt = qg2_expL(LV, LD, LV1, 2 * dt)
        prev_qk = qk
        Qn = qg2_update(qk, B, kx_, ky_)
        if step == 1:
            dq = dt * Qn
        elif step == 2:
            dq = dt / 2 * (3 * Qn - mmult3(expLdt, Qm[0]))
        else:
            dq = dt / 12 * (23 * Qn - 16 * mmult3(expLdt, Qm[0]) + 5 * mmult3(expL2dt, Qm[1]))
        t = t + dt
        Qm = [Qn, Qm[0]]
        qk = mmult3(expLdt, qk + dq)
        if Npackets > 0 and t > packet_delay_steps:
            if eval_mode == "lagrange":
                bf1 = grid_U(prev_qk[:, :, 0], K_d2, K2, kx_, ky_, shear_strength)
                bf2 = grid_U(qk[:, :, 0], K_d2, K2, kx_, ky_, shear_strength)
                ode = generate_raytracing_ode(bf1, bf2, Npackets, f, Cg, dt, dx)
            else:
                p1 = grid_U_planes_k(prev_qk[:, :, 0], K_d2, K2, kx_, ky_, shear_strength)
                p2 = grid_U_planes_k(qk[:, :, 0], K_d2, K2, kx_, ky_, shear_strength)
                ev = lambda x, y, a: spectral_eval_planes(x, y, [(1 - a) * c1 + a * c2 for c1, c2 in zip(p1, p2)], dx, nx)
                ode = generate_raytracing_ode(None, None, Npackets, f, Cg, dt, dx, eval6=ev)
            y, st = ode23(ode, [0.0, dt], np.concatenate([px, py, pk, pl]))
            px, py, pk, pl = (y[j * Npackets:(j + 1) * Npackets] for j in range(4))
            stats["packet_steps"] += 1; stats["ode23_steps"] += st["nsteps"]; stats["ode23_failed"] += st["nfailed"]
    return {"qk": qk, "t": t, "dt": dt, "U0": U0, "Fr": Fr, "T": T, "steps": step, "packets": (px, py, pk, pl), **stats}
