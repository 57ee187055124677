"""The on-device QG frame producers (swrt_qg.inc) at the production grids -- C3's one layer at 256^2, C4's two layers at
512^2 -- against extended-precision references (qg_ld_oracle.py) and the float64 oracle.

* CPU: each long-double helper against mpmath or the float64 oracle.
* Linear regime: a PV spectrum scaled by 2^-700 makes every product of the Jacobian underflow to exactly 0, so a step
  is exactly its linear propagator -- exp(dt factor_L) for two layers (both branches of expm2, the dt rebuild, the
  nu K^8 hyperviscosity), the filtered Euler / AB2 / AB3 recurrence for one layer -- with a reference at every mode.
* Nonlinear parity at 256^2 and 512^2 against the float64 oracle loops, one step against the long-double update().
* The hand-off to the flow slots (swrt_set_flow_from_qg / _qg2), get_grid, and swrt_g2k / swrt_k2g above 64^2.

Errors are measured per mode relative to the largest |q| of the reference, and per mode relative to its own |q| for
every mode within 1e-8 of the largest."""
import functools

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
from oracle import c_oracle as CO
from oracle import swrt_oracle as O
import qg_ld_oracle as Q
from test_spectral_large_grids import edge_positions, scaled_err

pytestmark = pytest.mark.skipif(not Q.EXTENDED, reason="np.longdouble has no more precision than float64 here")

K_D2, F0, CG = 3.0, 3.0, 1.0                     # f / Cg of C3 and C4
L1 = 2 * np.pi                                   # C3
L2, SHEAR, R2, ALPHA = 20.0, 0.5, 0.4, 4         # C4: qg2layersw_raytrace.m:26-33
TINY, TINY_SHIFT = 2.0 ** -700, 60               # the linear regime; the scaling guard runs at 2^-640 as well
TOL_LIN = 1e-13                                  # linear regime: of max|q_ref|
TOL_LIN_MODE = 1e-11                             # linear regime: of |q_ref| at modes above 1e-8 max|q_ref|
TOL_NONLIN = 1e-12                               # nonlinear parity: of max|q|
TOL_ONE_STEP_LD = 1e-14                          # one step against the long-double update(): of max|q|


def nu(nx):
    return 0.1 * (L2 / nx) ** 8                  # nutune * dx^(2 alpha)


def random_spectrum(nx, seed, layers=1):
    """every mode of the half plane, unit amplitude, real-field symmetry on ky = 0"""
    rs = np.random.RandomState(seed)
    out = [O.symmetrise_ky0(rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) for _ in range(layers)]
    return out if layers > 1 else out[0]


def errors(got, ref):
    """(max |got - ref| / max |ref|, max |got - ref| / |ref| over modes with |ref| >= 1e-8 max |ref|)"""
    got, ref = np.asarray(got).astype(Q.CLD), np.asarray(ref).astype(Q.CLD)
    d, a = np.abs(got - ref), np.abs(ref)
    scale = a.max()
    big = a >= 1e-8 * scale
    return float(d.max() / scale), float((d[big] / a[big]).max())


@functools.lru_cache(maxsize=None)
def factor_L(nx, beta):
    kx, ky = Q.wavenumbers(nx, L2)
    return Q.qg2_factor_ld(kx, ky, K_D2, beta, SHEAR, R2, nu(nx), ALPHA)


@functools.lru_cache(maxsize=None)
def expL(nx, beta, dt):
    return Q.expm2_ld(factor_L(nx, beta), dt)


def branch_dt(nx, beta):
    """a dt that puts >= 100 modes (all there are at 32^2: 105) on either side of expm2's series threshold: |dt D| in
    [3e-5, 1e-4) and in [1e-4, 3e-4]"""
    D = np.abs(Q.discriminant(factor_L(nx, beta))).ravel()
    D = np.sort(D[D > 0])
    best = max(np.geomspace(D[0], D[-1], 400),
               key=lambda c: min(((D >= 0.3 * c) & (D < c)).sum(), ((D >= c) & (D <= 3 * c)).sum()))
    return 1e-4 / best


def series_dt(nx, beta):
    """a dt that keeps every mode on expm2's series branch, |dt D| < 1e-4: half the threshold over the largest |D|.
    (No fixed dt does that at every size: max|D| is ~290 at 32^2 for C4's operator, ~20 at 256^2 and ~40 at 512^2.)"""
    return 0.5e-4 / np.abs(Q.discriminant(factor_L(nx, beta))).max()


def qg2_handle(nx, q, beta):
    return S.QG2Flow(nx, L2, q[0], q[1], K_D2, beta, SHEAR, R2, nu(nx), ALPHA)


def c3_state(nx):
    """C3: initial_q(U_g = 0.5, rng(146)) on L = 2 pi, dt = 0.05 dx / U0 (qgsw_raytrace.m:29,70)"""
    xg = O.matlab_linspace(-L1 / 2, L1 / 2, nx)
    X, Y = np.meshgrid(xg, xg)
    qk = O.g2k(O.initial_q(X, Y, 0.5, K_D2, O.matlab_rand_stream(146)))
    kx, ky = Q.wavenumbers(nx, L1)
    fl = O.grid_U(qk, K_D2, kx ** 2 + ky ** 2, kx, ky)
    return qk, 0.05 * (L1 / nx) / np.sqrt((fl["u"] ** 2 + fl["v"] ** 2).max())


def c4_state(nx):
    """C4's field (the benchmark's: workloads.make_workload('C4'), k up to 30, seed 5) as PV of both layers, q2 = -q1
    (qg2layersw_raytrace.m:57), and the driver's first dt = 0.25 dx / U0"""
    w = W.make_workload("C4", n_packets=1, nx=nx)
    kx, ky = Q.wavenumbers(nx, L2)
    K2 = kx ** 2 + ky ** 2
    q1 = O.symmetrise_ky0(-(K_D2 + K2) * w.psik)
    qk = np.stack([q1, -q1], axis=2)
    return qk, 0.25 * (L2 / nx) / O.qg2_max_speed(qk, K_D2, K2, kx, ky, SHEAR)


# ------------------------------------------------------------------------------------------------
# CPU: the long-double helpers
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [0.0, 0.3])
@pytest.mark.parametrize("dt", [2e-5, 0.05])
def test_expm2_ld_against_mpmath(beta, dt):
    """~200 modes of C4's operator at 512^2: K = 0, the kx = 0 column, both top corners, the 50 smallest |D| (near the
    neutral curve, where the 2x2 matrix is close to a Jordan block) and 60 random ones, against mpmath at 40 digits"""
    nx = 512
    M = factor_L(nx, beta)
    E = expL(nx, beta, dt)
    nkx, nky = M.shape[2:]
    kmax = (nkx - 1) // 2
    D = np.abs(Q.discriminant(M))
    modes = {(kmax, 0), (0, nky - 1), (nkx - 1, nky - 1)}
    modes |= {(kmax, j) for j in range(0, nky, 2)}
    modes |= set(zip(*np.unravel_index(np.argsort(D, axis=None)[:50], D.shape)))
    rs = np.random.RandomState(3)
    modes |= set(zip(rs.randint(0, nkx, 60), rs.randint(0, nky, 60)))
    assert len(modes) >= 200
    worst = max(Q.expm2_mp_error(E[:, :, a, b], M[:, :, a, b], dt) for a, b in modes)
    assert worst < 1e-17, worst


@pytest.mark.parametrize("nx,dt", [(64, 0.05), (256, 0.02), (512, 0.01)])
def test_expm2_ld_against_eig_oracle(nx, dt):
    """the float64 oracle's exp(L t) = V exp(D t) V^-1 (pageeig) agrees to its own noise, ~2.5e-13 of each mode's
    max|E| (modes whose exponential is below 1e-200 have lost their digits to float64's range and are left out)"""
    kx, ky = Q.wavenumbers(nx, L2)
    _, FL, LV, LDg, LV1 = O.qg2_operators(kx, ky, K_D2, 0.3, SHEAR, R2, nu(nx), ALPHA)
    assert np.abs(FL - factor_L(nx, 0.3)).max() <= 1e-15 * np.abs(FL).max()
    E = expL(nx, 0.3, dt)
    Eo = O.qg2_expL(LV, LDg, LV1, dt)
    scale = np.abs(E).max(axis=(0, 1))
    keep = scale > 1e-200
    err = (np.abs(Eo - E).max(axis=(0, 1))[keep] / scale[keep]).astype(np.float64)
    assert err.max() < 1e-12, err.max()


@pytest.mark.parametrize("nx", [50, 256])
def test_qg_linear_ld_against_qg_run(nx):
    """qg_run at 2^-700 (its Jacobian underflows to 0) is the linear recurrence: Euler, AB2, AB3 and the filter"""
    q0 = random_spectrum(nx, 1) * TINY
    kx, ky = O.wavenumbers(nx)
    assert np.abs(O.qg_update(q0, kx ** 2 + ky ** 2, K_D2, 0.0, 0.0, np.zeros(kx.shape), kx, ky)).max() == 0.0
    for n in (1, 2, 3, 40):
        ref = O.qg_run(q0, n, 0.05, nx, L1, K_D2, F0, CG, beta=0.3, r_drag=0.0, force_strength=0.0)
        e, _ = errors(ref, Q.qg_linear_ld(q0, n, 0.05, nx, L1, K_D2, 0.3))
        assert e < 5e-15, (n, e)          # numpy rounds the filter's exp(cst (kstar - kc)^4) at arguments up to ~35


@pytest.mark.parametrize("nx", [64, 130, 256])
def test_g2k_k2g_ld_against_numpy(nx):
    rs = np.random.RandomState(nx)
    kx, ky = O.wavenumbers(nx)
    fk = O.symmetrise_ky0((rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx ** 2 + ky ** 2))
    fg = Q.k2g_ld(fk)
    assert np.abs(fg - O.k2g(fk)).max() < 1e-15 * np.abs(fg).max()
    back = Q.g2k_ld(fg)
    assert np.abs(back - fk).max() < 1e-18 * np.abs(fk).max()           # g2k(k2g(fk)) = fk: the ld round trip
    assert np.abs(back - O.g2k(fg.astype(np.float64))).max() < 1e-15 * np.abs(fk).max()


# ------------------------------------------------------------------------------------------------
# linear regime: the producers are exactly their propagators
# ------------------------------------------------------------------------------------------------
LIN2_SIZES = [32, 50, 256, 512]
LIN2_DTS = ["series", 2e-5, 1e-3, 1e-2, 0.05, "branch"]


@pytest.mark.gpu
@pytest.mark.parametrize("nx", LIN2_SIZES)
@pytest.mark.parametrize("beta", [0.0, 0.3])
@pytest.mark.parametrize("dt", LIN2_DTS)
def test_qg2_linear_propagator(nx, beta, dt):
    """q_N = exp(dt factor_L)^N q0 for N = 1, 3, 50"""
    if dt == "branch":
        dt = branch_dt(nx, beta)
    if dt == "series":
        dt = series_dt(nx, beta)
        assert np.abs(Q.discriminant(factor_L(nx, beta))).max() * dt < 1e-4           # series branch everywhere
    q0 = np.stack(random_spectrum(nx, 7, layers=2)) * TINY
    E = expL(nx, beta, dt)
    ref = q0.astype(Q.CLD)
    qg = qg2_handle(nx, q0, beta)
    done, worst = 0, (0.0, 0.0)
    for n in (1, 3, 50):
        while done < n:
            qg.step(dt)
            ref = Q.apply2(E, ref)
            done += 1
        e = errors(np.stack([qg.get(0), qg.get(1)]), ref)
        worst = max(worst[0], e[0]), max(worst[1], e[1])
    qg.close()
    print(f"qg2 linear nx={nx} beta={beta} dt={dt:.3g}: {worst[0]:.2e} of max, {worst[1]:.2e} per mode")
    assert worst[0] < TOL_LIN and worst[1] < TOL_LIN_MODE, worst


@pytest.mark.gpu
@pytest.mark.parametrize("nx", LIN2_SIZES)
def test_qg2_dt_change_rebuilds_the_exponentials(nx):
    """dt1, dt2, dt1 gives E(dt1) E(dt2) E(dt1) q0: a stale expLdt would give E(dt1)^3 or E(dt2)^2 E(dt1)"""
    beta, dt1, dt2 = 0.3, 1e-2, branch_dt(nx, 0.3)
    q0 = np.stack(random_spectrum(nx, 8, layers=2)) * TINY
    ref = q0.astype(Q.CLD)
    qg = qg2_handle(nx, q0, beta)
    for dt in (dt1, dt2, dt1):
        qg.step(dt)
        ref = Q.apply2(expL(nx, beta, dt), ref)
    e = errors(np.stack([qg.get(0), qg.get(1)]), ref)
    qg.close()
    print(f"qg2 dt sequence nx={nx}: {e[0]:.2e} of max, {e[1]:.2e} per mode")
    assert e[0] < TOL_LIN and e[1] < TOL_LIN_MODE, e


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [50, 256, 512])
def test_qg_linear_recurrence(nx):
    """one layer, beta = 0.3, r_drag = 0, no forcing: Euler, AB2, AB3 and the filter against qg_linear_ld"""
    dt = 0.05
    q0 = random_spectrum(nx, 9) * TINY
    qg = S.QGFlow(nx, L1, q0, K_D2, dt, F0, CG, beta=0.3, r_drag=0.0, force_strength=0.0)
    done, worst = 0, (0.0, 0.0)
    for n in (1, 2, 3, 40):
        qg.step(n - done)
        done = n
        e = errors(qg.get(), Q.qg_linear_ld(q0, n, dt, nx, L1, K_D2, 0.3))
        worst = max(worst[0], e[0]), max(worst[1], e[1])
    qg.close()
    print(f"qg linear nx={nx}: {worst[0]:.2e} of max, {worst[1]:.2e} per mode")
    assert worst[0] < TOL_LIN and worst[1] < TOL_LIN_MODE, worst


def assert_scaled_identical(a, b, shift):
    """a * 2^shift == b bit for bit wherever b's components are far above the subnormal range of a's run; below, a's
    run rounded to subnormals and only an absolute bound far under either scale is asserted"""
    a = np.ldexp(np.stack([np.asarray(a).real, np.asarray(a).imag]), shift)
    b = np.stack([np.asarray(b).real, np.asarray(b).imag])
    normal = np.abs(b) >= 2.0 ** -900
    assert normal.mean() > 0.5
    assert np.array_equal(a[normal], b[normal])
    assert np.abs(a[~normal] - b[~normal]).max(initial=0.0) <= 2.0 ** -950


@pytest.mark.gpu
def test_linear_regime_scales_exactly():
    """the runs at 2^-700 and 2^-640 agree bit for bit after the factor 2^60: no term but the linear one ran"""
    nx, dt = 512, 1e-3
    q0 = np.stack(random_spectrum(nx, 10, layers=2))
    out = []
    for sc in (TINY, TINY * 2.0 ** TINY_SHIFT):
        qg = qg2_handle(nx, q0 * sc, 0.3)
        for _ in range(3):
            qg.step(dt)
        out.append(np.stack([qg.get(0), qg.get(1)]))
        qg.close()
    comps = np.abs(np.stack([out[0].real, out[0].imag]))
    assert np.all(comps[comps != 0] >= 2.0 ** -1022)                   # no subnormals: bit identity holds everywhere
    assert np.array_equal(np.ldexp(out[0].real, TINY_SHIFT), out[1].real)
    assert np.array_equal(np.ldexp(out[0].imag, TINY_SHIFT), out[1].imag)
    nx = 256
    q0 = random_spectrum(nx, 11)
    out = []
    for sc in (TINY, TINY * 2.0 ** TINY_SHIFT):
        qg = S.QGFlow(nx, L1, q0 * sc, K_D2, 0.05, F0, CG, beta=0.3, r_drag=0.0, force_strength=0.0)
        qg.step(3)
        out.append(qg.get())
        qg.close()
    assert_scaled_identical(out[0], out[1], TINY_SHIFT)


# ------------------------------------------------------------------------------------------------
# nonlinear parity at the production sizes
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nx,nsteps", [(256, 500), (512, 100)])
def test_qg_nonlinear_against_qg_run(nx, nsteps):
    """C3's run (beta 0.3, forcing 0.1, r_drag 0) against the oracle; step(N) equals N calls of step(1) bit for bit.
    A 1-ulp change of q0 moves qg_run by ~2.5e-16 of max|q| after 100 steps at 256^2, so 1e-12 is a real bound."""
    qk0, dt = c3_state(nx)
    kw = dict(beta=0.3, r_drag=0.0, force_strength=0.1)
    qg, one = S.QGFlow(nx, L1, qk0, K_D2, dt, F0, CG, **kw), S.QGFlow(nx, L1, qk0, K_D2, dt, F0, CG, **kw)
    qg.step(nsteps)
    for _ in range(nsteps):
        one.step(1)
    got = qg.get()
    assert np.array_equal(got, one.get())
    ref = O.qg_run(qk0, nsteps, dt, nx, L1, K_D2, F0, CG, **kw)
    e = np.abs(got - ref).max() / np.abs(ref).max()
    grid = qg.get_grid()
    eg = np.abs(grid - O.k2g(got)).max() / np.abs(grid).max()
    qg.close(); one.close()
    print(f"qg nonlinear nx={nx} {nsteps} steps: {e:.2e} of max; get_grid {eg:.2e}")
    assert e < TOL_NONLIN and eg < 1e-13, (e, eg)


@pytest.mark.gpu
def test_qg_r_drag_source_256():
    """the r_drag K2 source of update() as written, 12 steps (Euler, AB2, AB3).  The source grows with K2 (0.01 K2 reaches
    328 at 256^2), and with r_drag = 0.01 C3's state blows up to |q| ~ 1e43 within 12 steps, where a 1-ulp change of q0
    already moves qg_run by 3.5e-12.  r_drag = 1e-4 keeps the run well conditioned (that spread is 2.4e-16) while the
    source changes q by ~11% of max|q|."""
    nx = 256
    qk0, dt = c3_state(nx)
    kw = dict(beta=0.3, r_drag=1e-4, force_strength=0.1)
    qg = S.QGFlow(nx, L1, qk0, K_D2, dt, F0, CG, **kw)
    qg.step(12)
    ref = O.qg_run(qk0, 12, dt, nx, L1, K_D2, F0, CG, **kw)
    without = O.qg_run(qk0, 12, dt, nx, L1, K_D2, F0, CG, **dict(kw, r_drag=0.0))
    assert np.abs(ref - without).max() > 0.05 * np.abs(ref).max()       # the source is not lost in the bound
    e = np.abs(qg.get() - ref).max() / np.abs(ref).max()
    qg.close()
    print(f"qg r_drag nx=256: {e:.2e} of max")
    assert e < TOL_NONLIN, e


@pytest.mark.gpu
def test_qg_one_step_against_long_double_update():
    """update() + Euler + filter at 256^2 with g2k_ld / k2g_ld in place of the FFTs"""
    nx = 256
    qk0, dt = c3_state(nx)
    qg = S.QGFlow(nx, L1, qk0, K_D2, dt, F0, CG, beta=0.3, r_drag=0.0, force_strength=0.1)
    qg.step(1)
    got = qg.get()
    qg.close()
    kx, ky = Q.wavenumbers(nx, L1)
    forces = O.qg_inertial_ring(0.1, kx ** 2 + ky ** 2, F0, CG)
    Qn = Q.qg_update_ld(qk0, nx, L1, K_D2, 0.3, 0.0, forces)
    ref = Q.qg_filter_ld(kx, ky, L1 / nx) * (qk0.astype(Q.CLD) + Q.LD(dt) * Qn)
    e, _ = errors(got, ref)
    print(f"qg one step vs long double nx=256: {e:.2e} of max")
    assert e < TOL_ONE_STEP_LD, e


@pytest.mark.gpu
def test_qg2_nonlinear_512():
    """C4's two layers for 30 steps at the driver's CFL dt, halved at step 11, against the oracle's loop with
    exp(dt factor_L) from expm2_ld rounded to complex128; max_speed against the oracle at every step; a second handle
    driven through the same dts agrees bit for bit"""
    nx, beta = 512, 0.0
    qk, dt0 = c4_state(nx)
    kx, ky = Q.wavenumbers(nx, L2)
    K2 = kx ** 2 + ky ** 2
    B = O.qg2_operators(kx, ky, K_D2, beta, SHEAR, R2, nu(nx), ALPHA)[0]
    qg, twin = qg2_handle(nx, [qk[:, :, 0], qk[:, :, 1]], beta), qg2_handle(nx, [qk[:, :, 0], qk[:, :, 1]], beta)
    Qm = [np.zeros_like(qk), np.zeros_like(qk)]
    worst, worst_u = 0.0, 0.0
    for step in range(1, 31):
        dt = dt0 if step <= 10 else dt0 / 2
        U0 = O.qg2_max_speed(qk, K_D2, K2, kx, ky, SHEAR)
        worst_u = max(worst_u, abs(qg.max_speed() - U0) / U0)
        E1 = expL(nx, beta, dt).astype(np.complex128)
        E2 = expL(nx, beta, 2 * dt).astype(np.complex128)
        Qn = O.qg2_update(qk, B, kx, ky)
        if step == 1:
            dq = dt * Qn
        elif step == 2:
            dq = dt / 2 * (3 * Qn - O.mmult3(E1, Qm[0]))
        else:
            dq = dt / 12 * (23 * Qn - 16 * O.mmult3(E1, Qm[0]) + 5 * O.mmult3(E2, Qm[1]))
        Qm = [Qn, Qm[0]]
        qk = O.mmult3(E1, qk + dq)
        qg.step(dt); twin.step(dt)
        for layer in range(2):
            ref = qk[:, :, layer]
            worst = max(worst, np.abs(qg.get(layer) - ref).max() / np.abs(ref).max())
    for layer in range(2):
        assert np.array_equal(qg.get(layer), twin.get(layer))
    qg.close(); twin.close()
    print(f"qg2 nonlinear 512: {worst:.2e} of max per layer; max_speed {worst_u:.2e}")
    assert worst < TOL_NONLIN and worst_u < 1e-13, (worst, worst_u)


@pytest.mark.gpu
def test_qg2_max_speed_over_the_whole_512_grid():
    """max_speed of C4's field and of the same field moved by half the domain in y (q-hat times (-1)^ky): one of the two
    has its maximum in the upper half of the grid, past the first grid-stride chunk of the reduction"""
    nx = 512
    qk, _ = c4_state(nx)
    kx, ky = Q.wavenumbers(nx, L2)
    K2 = kx ** 2 + ky ** 2
    sign = (-1.0) ** O.wavenumbers(nx)[1]
    rows = []
    for q in (qk, qk * sign[:, :, None]):
        U0 = O.qg2_max_speed(q, K_D2, K2, kx, ky, SHEAR)
        qg = qg2_handle(nx, [q[:, :, 0], q[:, :, 1]], 0.0)
        got = qg.max_speed()
        qg.close()
        assert abs(got - U0) < 1e-13 * U0, (got, U0)
        s2 = [(lambda fl: fl["u"] ** 2 + fl["v"] ** 2)(O.grid_U(q[:, :, i], K_D2, K2, kx, ky, SHEAR)) for i in range(2)]
        s2 = s2[int(np.argmax([a.max() for a in s2]))]
        rows.append(np.unravel_index(np.argmax(s2), s2.shape)[1])
    assert max(rows) >= nx // 2, rows                          # column-major index >= nx^2/2


# ------------------------------------------------------------------------------------------------
# hand-off to the flow slots at production size
# ------------------------------------------------------------------------------------------------
def eval_points(L, dx, n=2000, seed=21):
    rs = np.random.RandomState(seed)
    xe, ye = edge_positions(L, dx)
    return np.concatenate([rs.uniform(-3 * L, 3 * L, n), xe]), np.concatenate([rs.uniform(-3 * L, 3 * L, n), ye])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [S.MODE_SPECTRAL, S.MODE_NUFFT])
def test_set_flow_from_qg_256(mode):
    nx, u_mean = 256, 0.3
    qk0, dt = c3_state(nx)
    qg = S.QGFlow(nx, L1, qk0, K_D2, dt, F0, CG, beta=0.3, r_drag=0.0, force_strength=0.1)
    qg.step(5)
    qk = qg.get()
    kx, ky = Q.wavenumbers(nx, L1)
    x, y = eval_points(L1, L1 / nx)
    with S.Engine(nx, L1, F0, CG ** 2, mode) as e:
        qg.to_flow(e, 0, u_mean=u_mean)
        got = e.eval_at(x, y)
    qg.close()
    ref = CO.spectral_eval(x, y, O.grid_U_planes_k(qk, K_D2, kx ** 2 + ky ** 2, kx, ky, u_mean), L1 / nx, nx, precise=True)
    err = scaled_err(got, ref)
    print(f"set_flow_from_qg 256 mode={mode}: {err:.2e} of max|plane|")
    assert err < 1e-12, err


def qg2_c4_after(nx, nsteps):
    qk, dt = c4_state(nx)
    qg = qg2_handle(nx, [qk[:, :, 0], qk[:, :, 1]], 0.0)
    for _ in range(nsteps):
        qg.step(dt)
    return qg


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [S.MODE_SPECTRAL, S.MODE_NUFFT])
def test_set_flow_from_qg2_512(mode):
    nx = 512
    qg = qg2_c4_after(nx, 3)
    q1 = qg.get(0)
    kx, ky = Q.wavenumbers(nx, L2)
    x, y = eval_points(L2, L2 / nx)
    with S.Engine(nx, L2, F0, CG ** 2, mode) as e:
        qg.to_flow(e, 0)
        got = e.eval_at(x, y)
    qg.close()
    ref = CO.spectral_eval(x, y, O.grid_U_planes_k(q1, K_D2, kx ** 2 + ky ** 2, kx, ky, SHEAR), L2 / nx, nx, precise=True)
    err = scaled_err(got, ref)
    print(f"set_flow_from_qg2 512 mode={mode}: {err:.2e} of max|plane|")
    assert err < 1e-12, err


def _ndev():
    try:
        return S.load_library().swrt_device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < 2, reason="needs >= 2 CUDA devices (the in-library multi-device handle)")
def test_set_flow_from_qg2_512_on_two_devices():
    nx = 512
    qg = qg2_c4_after(nx, 3)
    x, y = eval_points(L2, L2 / nx, n=3001)
    res = []
    for ngpu in (1, 2):
        with S.Engine(nx, L2, F0, CG ** 2, S.MODE_SPECTRAL, ngpu=ngpu) as e:
            qg.to_flow(e, 0)
            e.set_packets(x, y, np.ones_like(x), np.zeros_like(x))
            res.append(e.eval())
    qg.close()
    assert np.array_equal(res[0], res[1])


# ------------------------------------------------------------------------------------------------
# swrt_g2k / swrt_k2g above 64^2
# ------------------------------------------------------------------------------------------------
def u_plane(nx, seed=7):
    """the u plane of test_gpu_parity.make_flow: -i ky psi-hat, psi-hat ~ 0.3 randn / (1 + K^2)^1.5"""
    rs = np.random.RandomState(seed)
    kx, ky = O.wavenumbers(nx)
    psik = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx ** 2 + ky ** 2) ** 1.5 * 0.3
    return -1j * ky * psik


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [128, 130, 256, 258, 384, 512, 1024])
def test_device_g2k_k2g_large(nx):
    """the bounds of test_gpu_parity.test_device_g2k_k2g_grid_U; long-double references up to 512^2, numpy at 1024^2"""
    fk = u_plane(nx)
    fg = S.k2g_dev(fk)
    ref_g = Q.k2g_ld(fk) if nx <= 512 else O.k2g(fk)
    eg = float(np.abs(fg - ref_g).max())
    back = S.g2k_dev(fg)
    ref_k = Q.g2k_ld(fg) if nx <= 512 else O.g2k(fg)
    ek = float(np.abs(back - ref_k).max())
    print(f"g2k/k2g nx={nx}: k2g {eg:.2e} (max|fg| {np.abs(fg).max():.2e}), g2k {ek:.2e}")
    assert eg < 1e-13 * max(1.0, float(np.abs(ref_g).max())) and ek < 1e-15, (eg, ek)
