"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs, against the committed golden fixture, and -- at BASELINE.json's full sizes -- through
size-independent properties.  Parity contract: SURVEY.md 8c P1-P6.

Tolerances (fp64):  field / RHS values 1e-12 relative to max|plane|;  trajectories over <= 100
steps 1e-9 absolute;  histogram counts bit-exact."""
from pathlib import Path

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from swraytracing_b200 import workloads as W
from oracle import swrt_oracle as O
from oracle import c_oracle as CO

pytestmark = pytest.mark.gpu

GOLD = np.load(Path(__file__).parent / "golden" / "hotpath_nx32.npz")
TOL_FIELD = 1e-12
TOL_TRAJ = 1e-9
F0, GH0 = 3.0, 1.0


def scaled_err(got, ref):
    got = np.asarray(got); ref = np.asarray(ref)
    scale = np.abs(ref).reshape(ref.shape[0], -1).max(axis=1)
    scale = np.where(scale > 0, scale, 1.0)
    return float((np.abs(got - ref).reshape(ref.shape[0], -1).max(axis=1) / scale).max())


def make_flow(nx, seed=7, slope=1.5, amp=0.3):
    rs = np.random.RandomState(seed)
    kx_, ky_ = O.wavenumbers(nx)
    psik = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx_ ** 2 + ky_ ** 2) ** slope * amp
    planes = O.velocity_planes_k(psik, kx_, ky_)
    return psik, planes


def make_packets(n, L, seed=5):
    rs = np.random.RandomState(seed)
    i = np.arange(n)
    return rs.uniform(-3 * L, 3 * L, n), rs.uniform(-3 * L, 3 * L, n), 3 * np.cos(0.37 * i), 3 * np.sin(0.37 * i)


# ------------------------------------------------------------------------------------------------
# P2: SPECTRAL kernel vs exact-sum oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nx", [16, 32, 36, 48, 64, 128])
@pytest.mark.parametrize("mt", [1, 2])
@pytest.mark.parametrize("psi", [True, False])
def test_spectral_eval_vs_exact_sum(nx, mt, psi):
    # psi=True: three psi-hat moment planes contracted, six planes assembled in stage 2;
    # psi=False: the six planes contracted directly.  Same oracle, same tolerance.
    L = 2 * np.pi; dx = L / nx
    psik, planes = make_flow(nx)
    n = 517 if nx <= 64 else 300
    x, y, k, l = make_packets(n, L)
    ref = CO.spectral_eval(x, y, planes, dx, nx, precise=True)
    with S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as e:
        e.set_tuning(mt, use_psi_moments=psi)
        e.set_flow_spectral(psik)
        assert e.contracted_planes() == (3 if psi else 6)
        e.set_packets(x, y, k, l)
        got = e.eval()
        assert scaled_err(got, ref) < TOL_FIELD
        got2 = e.eval_at(x[::-1].copy(), y[::-1].copy())
        assert np.array_equal(got2[:, ::-1], got)      # a packet's value does not depend on its tile slot


def test_spectral_full_spectrum_flat_is_within_tolerance():
    # white (slope 0) spectrum up to the truncation: the hardest case for the twiddle recurrences
    nx = 128; L = 2 * np.pi; dx = L / nx
    psik, planes = make_flow(nx, slope=0.0, amp=1e-3)
    x, y, k, l = make_packets(200, L, seed=9)
    ref = CO.spectral_eval(x, y, planes, dx, nx, precise=True)
    with S.Engine(nx, L, F0, GH0) as e:
        e.set_flow_planes_spectral(planes)
        got = e.eval_at(x, y)
    assert scaled_err(got, ref) < TOL_FIELD


def test_spectral_planes_upload_and_domain_L20():
    # qg2layersw_raytrace.m:13,19-22: L = 20, wavenumbers scaled by 2*pi/L, mean shear on u
    nx = 32; L = 20.0; dx = L / nx
    rs = np.random.RandomState(3)
    kx_, ky_ = O.wavenumbers(nx)
    kap = 2 * np.pi / L
    psik = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx_ ** 2 + ky_ ** 2)
    planes = O.velocity_planes_k(psik, kap * kx_, kap * ky_)
    planes[0] = planes[0].copy(); planes[0][nx // 2 - 1, 0] += 0.5
    x, y, k, l = make_packets(333, L)
    ref = CO.spectral_eval(x, y, planes, dx, nx)
    with S.Engine(nx, L, F0, GH0) as e:
        e.set_flow_spectral(psik, u_mean=0.5)
        assert e.contracted_planes() == 3
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD
        e.set_tuning(0, use_psi_moments=False)
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD
        e.set_tuning(0, use_psi_moments=True)
        e.set_flow_planes_spectral(planes)
        assert e.contracted_planes() == 6          # arbitrary planes: no psi-hat to take moments of
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD


# ------------------------------------------------------------------------------------------------
# P1: LAGRANGE6 kernel vs restated interpolate / interpolate_U
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nx", [16, 32, 64])
def test_lagrange_eval_vs_interpolate(nx):
    L = 2 * np.pi; dx = L / nx
    psik, planes = make_flow(nx)
    grids = [O.k2g(p) for p in planes]
    x, y, k, l = make_packets(777, L)
    ref = CO.interpolate6(x, y, grids, dx)
    with S.Engine(nx, L, F0, GH0, S.MODE_LAGRANGE6) as e:
        e.set_flow_grid(*grids)
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD
    with S.Engine(nx, L, F0, GH0, S.MODE_LAGRANGE6) as e:      # grid_U on the device (k2g via cuFFT)
        e.set_flow_spectral(psik)
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD
    # standalone interpolate(x,y,F,dx,dy) and the bump = 1e-10 variant
    assert np.abs(S.interpolate_dev(x, y, grids[0], dx, dx) - ref[0]).max() / np.abs(ref[0]).max() < TOL_FIELD
    par = O.interpolate_par(x, y, grids[1], dx, dx)
    assert np.abs(R.interpolate_par(x, y, grids[1], dx, dx) - par).max() / np.abs(par).max() < TOL_FIELD


def test_interpolate_U_time_blend_both_modes():
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx
    alpha = float(GOLD["alpha"])
    kx_, ky_ = O.wavenumbers(nx)
    g1 = [O.k2g(p) for p in O.velocity_planes_k(GOLD["psik"], kx_, ky_)]
    g2 = [O.k2g(p) for p in O.velocity_planes_k(GOLD["psik2"], kx_, ky_)]
    names = ("u", "v", "ux", "uy", "vx", "vy")
    bf1 = dict(zip(names, g1)); bf2 = dict(zip(names, g2))
    xy = np.stack([GOLD["x"], GOLD["y"]], axis=1)
    U, nab = R.interpolate_U(bf1, bf2, alpha, xy, dx)                  # binds to qg_flow_ray_trace/interpolate.m: bump 1e-10
    got = np.stack([U[:, 0], U[:, 1], nab["u_x"], nab["u_y"], nab["v_x"], nab["v_y"]])
    Uo, nabo = O.interpolate_U(bf1, bf2, alpha, xy, dx)
    assert scaled_err(got, np.stack([Uo[:, 0], Uo[:, 1], nabo["u_x"], nabo["u_y"], nabo["v_x"], nabo["v_y"]])) < TOL_FIELD
    U, nab = R.interpolate_U(bf1, bf2, alpha, xy, dx, bump=R.BUMP_LIVE)    # the same function beside ray_trace_sw's copy
    got = np.stack([U[:, 0], U[:, 1], nab["u_x"], nab["u_y"], nab["v_x"], nab["v_y"]])
    assert scaled_err(got, GOLD["interpU_lagrange"]) < TOL_FIELD
    with S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(GOLD["psik"], slot=0)
        e.set_flow_spectral(GOLD["psik2"], slot=1)
        assert scaled_err(e.eval_at(GOLD["x"], GOLD["y"], alpha), GOLD["interpU_spectral"]) < TOL_FIELD
        assert scaled_err(e.eval_at(GOLD["x"], GOLD["y"], 0.0), GOLD["eval_spectral"]) < TOL_FIELD
        with pytest.raises(S.SwrtError):
            S.Engine(nx, L, F0, GH0).eval_at(GOLD["x"], GOLD["y"], 0.0)       # no flow set


# ------------------------------------------------------------------------------------------------
# P3: SPECTRAL kernel vs the reference's Lagrange stencil
# ------------------------------------------------------------------------------------------------
def test_spectral_vs_reference_lagrange_at_grid_nodes_and_bound_off_grid():
    nx = 64; L = 2 * np.pi; dx = L / nx
    rs = np.random.RandomState(1)
    kx_, ky_ = O.wavenumbers(nx)
    kcut = 8
    psik = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) * ((np.abs(kx_) <= kcut) & (ky_ <= kcut)) * 0.01
    planes = O.velocity_planes_k(psik, kx_, ky_)
    grids = [O.k2g(p) for p in planes]
    ix, iy = np.meshgrid(np.arange(nx), np.arange(nx), indexing="ij")
    xn = (ix * dx).ravel(); yn = (iy * dx).ravel()
    with S.Engine(nx, L, F0, GH0) as e:
        e.set_flow_spectral(psik)
        got = e.eval_at(xn, yn)
        ref = CO.interpolate6(xn, yn, grids, dx)          # reference semantics at grid nodes
        assert scaled_err(got, ref) < TOL_FIELD
        x, y, _, _ = make_packets(500, L)
        gap = np.abs(e.eval_at(x, y) - CO.interpolate6(x, y, grids, dx))
        for c in range(6):
            # degree-5 Lagrange bound per direction (3.52/720) (kmax dx)^6 * sum|coefficients|
            csum = 2 * np.abs(planes[c]).sum()
            assert gap[c].max() <= 2 * (3.52 / 720) * (kcut * dx) ** 6 * csum


# ------------------------------------------------------------------------------------------------
# P4: RHS and short trajectories, each mode against its oracle
# ------------------------------------------------------------------------------------------------
def test_rhs_both_modes():
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx
    alpha = float(GOLD["alpha"])
    x, y, k, l = GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"]
    with S.Engine(nx, L, F0, GH0, S.MODE_LAGRANGE6) as e:
        e.set_flow_spectral(GOLD["psik"], slot=0); e.set_flow_spectral(GOLD["psik2"], slot=1)
        e.set_packets(x, y, k, l)
        assert scaled_err(np.stack(e.rhs(alpha)), GOLD["rhs_lagrange"]) < TOL_FIELD
    ref = np.stack(O.rhs_from_eval(GOLD["interpU_spectral"], k, l, F0, 1.0))
    with S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(GOLD["psik"], slot=0); e.set_flow_spectral(GOLD["psik2"], slot=1)
        e.set_packets(x, y, k, l)
        assert scaled_err(np.stack(e.rhs(alpha)), ref) < TOL_FIELD
    # generate_raytracing_ode closure (qgsw_raytrace.m:258-268), y = [x;y;k;l]
    kx_, ky_ = O.wavenumbers(nx)
    names = ("u", "v", "ux", "uy", "vx", "vy")
    bf1 = dict(zip(names, [O.k2g(p) for p in O.velocity_planes_k(GOLD["psik"], kx_, ky_)]))
    bf2 = dict(zip(names, [O.k2g(p) for p in O.velocity_planes_k(GOLD["psik2"], kx_, ky_)]))
    ode = R.generate_raytracing_ode(bf1, bf2, x.size, F0, 1.0, 2.0, dx, bump=R.BUMP_LIVE)
    dydt = ode(alpha * 2.0, np.concatenate([x, y, k, l]))
    assert scaled_err(dydt.reshape(4, -1), GOLD["rhs_lagrange"]) < TOL_FIELD
    ode = R.generate_raytracing_ode(bf1, bf2, x.size, F0, 1.0, 2.0, dx)        # as the QG drivers run it: bump 1e-10
    want = O.generate_raytracing_ode(bf1, bf2, x.size, F0, 1.0, 2.0, dx)(alpha * 2.0, np.concatenate([x, y, k, l]))
    assert scaled_err(ode(alpha * 2.0, np.concatenate([x, y, k, l])).reshape(4, -1), want.reshape(4, -1)) < TOL_FIELD


@pytest.mark.parametrize("mt", [1, 2])
@pytest.mark.parametrize("psi", [True, False])
def test_leapfrog_trajectory_spectral_golden_and_oracle(mt, psi):
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx; dt = float(GOLD["dt"])
    with S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as e:
        e.set_tuning(mt, use_psi_moments=psi)
        e.set_flow_spectral(GOLD["psik"])
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        e.step(S.SCHEME_LEAPFROG, dt, 20)
        assert np.abs(np.stack(e.get_packets()) - GOLD["leapfrog20_spectral"]).max() < TOL_TRAJ
        # 100 steps, fused (one launch) == 100 single-step launches, and both match the oracle
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        e.step(S.SCHEME_LEAPFROG, dt, 100)
        fused = np.stack(e.get_packets())
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        for _ in range(100):
            e.step(S.SCHEME_LEAPFROG, dt, 1)
        assert np.array_equal(fused, np.stack(e.get_packets()))
    kx_, ky_ = O.wavenumbers(nx)
    ref = CO.leapfrog_spectral(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"], O.velocity_planes_k(GOLD["psik"], kx_, ky_),
                               dx, nx, F0, GH0, dt, 100, precise=True)
    assert np.abs(fused - np.stack(ref)).max() < TOL_TRAJ


def test_leapfrog_trajectory_lagrange():
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx; dt = float(GOLD["dt"])
    with S.Engine(nx, L, F0, GH0, S.MODE_LAGRANGE6) as e:
        e.set_flow_grid(*list(GOLD["grids"]))
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        e.step(S.SCHEME_LEAPFROG, dt, 20)
        assert np.abs(np.stack(e.get_packets()) - GOLD["leapfrog20_lagrange"]).max() < TOL_TRAJ
        e.step(S.SCHEME_LEAPFROG, dt, 80)
        ref = CO.leapfrog_lagrange(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"], list(GOLD["grids"]), dx, F0, GH0, dt, 100)
        assert np.abs(np.stack(e.get_packets()) - np.stack(ref)).max() < TOL_TRAJ


def test_leapfrog_time_dependent_flow_blend_on_device():
    # swrt_step(alpha0, dalpha): step j evaluates (1-a_j) frame0 + a_j frame1, a_j = alpha0 + j*dalpha
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx; dt = float(GOLD["dt"])
    kx_, ky_ = O.wavenumbers(nx)
    p1 = O.velocity_planes_k(GOLD["psik"], kx_, ky_); p2 = O.velocity_planes_k(GOLD["psik2"], kx_, ky_)
    m = 8
    st = (GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
    for j in range(m):
        a = (j + 0.5) / m
        pl = [(1 - a) * u + a * v for u, v in zip(p1, p2)]
        st = O.leapfrog_step(*st, dt, F0, GH0, lambda xx, yy: CO.spectral_eval(xx, yy, pl, dx, nx))
    with S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(GOLD["psik"], slot=0); e.set_flow_spectral(GOLD["psik2"], slot=1)
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        e.step(S.SCHEME_LEAPFROG, dt, m, alpha0=0.5 / m, dalpha=1.0 / m)
        assert np.abs(np.stack(e.get_packets()) - np.stack(st)).max() < TOL_TRAJ
        with pytest.raises(S.SwrtError):
            e2 = S.Engine(nx, L, F0, GH0); e2.set_flow_spectral(GOLD["psik"]); e2.set_packets(*st)
            e2.step(S.SCHEME_LEAPFROG, dt, 2, alpha0=0.25, dalpha=0.5)         # slot 1 never set


@pytest.mark.parametrize("xka", [False, True])
def test_rk4_packet_steps_lagrange(xka):
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx; dt = float(GOLD["dt"])
    key = "rk4x3_xka_lagrange" if xka else "rk4x3_packet_lagrange"
    g = list(GOLD["grids"])
    with S.Engine(nx, L, F0, 1.0, S.MODE_LAGRANGE6) as e:
        e.set_flow_grid(*g, H=GOLD["H"] if xka else None)
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        e.step(S.SCHEME_RK4_XKA if xka else S.SCHEME_RK4_PACKET, dt, 3)
        got = np.stack(e.get_packets(with_a=True))
    ref = GOLD[key]
    assert np.abs(got[:4] - ref[:4]).max() < TOL_TRAJ
    if xka:
        assert np.abs(got[4] - ref[4]).max() < TOL_TRAJ
    # reference calling surface: Pout = step_packet(_xka)(P, U, GradU, [H,] C0, f, dx, dy, dt), one packet
    U = {"u": g[0], "v": g[1]}; G = {"u_x": g[2], "u_y": g[3], "v_x": g[4], "v_y": g[5]}
    P = {"x": float(GOLD["x"][0]), "y": float(GOLD["y"][0]), "k": float(GOLD["k"][0]), "l": float(GOLD["l"][0]), "a": 1.0}
    if xka:
        Pg = R.step_packet_xka(P, U, G, GOLD["H"], 1.0, F0, dx, dx, dt)
        Po = O.step_packet_xka(P, U, G, GOLD["H"], 1.0, F0, dx, dx, dt)
    else:
        Pg = R.step_packet(P, U, G, 1.0, F0, dx, dx, dt)
        Po = O.step_packet(P, U, G, 1.0, F0, dx, dx, dt)
    for name in Po:
        assert abs(Pg[name] - Po[name]) < 1e-12


@pytest.mark.parametrize("xka", [False, True])
def test_rk4_packet_steps_spectral(xka):
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx; dt = float(GOLD["dt"])
    kx_, ky_ = O.wavenumbers(nx)
    planes = O.velocity_planes_k(GOLD["psik"], kx_, ky_)
    Hk = O.g2k(GOLD["H"])
    n = 120
    st = tuple(GOLD[q][:n] for q in ("x", "y", "k", "l")) + (np.ones(n),)
    ref = st
    for _ in range(2):
        ref = O.rk4_step_batch(*ref, dt, 1.0, F0, None, dx, xka, mode="spectral", planes_k=planes + [Hk], nx=nx)
    with S.Engine(nx, L, F0, 1.0, S.MODE_SPECTRAL) as e:
        e.set_flow_planes_spectral(planes + ([Hk] if xka else []))
        e.set_packets(*st)
        e.step(S.SCHEME_RK4_XKA if xka else S.SCHEME_RK4_PACKET, dt, 2)
        got = np.stack(e.get_packets(with_a=True))
    assert np.abs(got - np.stack(ref)).max() < TOL_TRAJ
    if not xka:
        with pytest.raises(S.SwrtError):       # xka without an H plane is a state error, not a crash
            with S.Engine(nx, L, F0, 1.0) as e:
                e.set_flow_planes_spectral(planes); e.set_packets(*st); e.step(S.SCHEME_RK4_XKA, dt, 1)


# ------------------------------------------------------------------------------------------------
# P5 / properties at full size
# ------------------------------------------------------------------------------------------------
def test_zero_flow_analytic_dispersion_C1():
    w = W.make_workload("C1")
    for mode in (S.MODE_SPECTRAL, S.MODE_LAGRANGE6):
        with S.Engine(w.nx, w.L, w.f, w.gH, mode) as e:
            e.set_flow_spectral(w.psik)
            e.set_packets(w.x, w.y, w.k, w.l)
            e.step(S.SCHEME_LEAPFROG, w.dt, 100)
            x, y, k, l = e.get_packets()
        om = np.sqrt(w.f ** 2 + w.gH * (w.k ** 2 + w.l ** 2))
        assert np.array_equal(k, w.k) and np.array_equal(l, w.l)
        assert np.abs(x - (w.x + w.gH * w.k / om * 100 * w.dt)).max() < 1e-12
        assert np.abs(y - (w.y + w.gH * w.l / om * 100 * w.dt)).max() < 1e-12


def test_C2_full_size_against_cpu_port_and_sharding_identity():
    w = W.make_workload("C2")                      # 128^2, 65,536 packets: BASELINE configs[1]
    planes = W.planes_from_psik(w.psik, w.L)
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(w.psik)
        e.set_packets(w.x, w.y, w.k, w.l)
        got = e.eval()
        ref = CO.spectral_eval(w.x, w.y, planes, w.dx, w.nx, precise=False)     # double sums: 1e-11 is their own accuracy
        assert scaled_err(got, ref) < 1e-11
        sub = np.arange(0, w.n_packets, 97)
        refp = CO.spectral_eval(w.x[sub], w.y[sub], planes, w.dx, w.nx, precise=True)
        assert scaled_err(got[:, sub], refp) < TOL_FIELD
        e.step(S.SCHEME_LEAPFROG, w.dt, 10)
        full = np.stack(e.get_packets())
        # the same packets split into two unequal shards give bit-identical states (SURVEY.md section 4)
        cut = 30011
        parts = []
        for sl in (slice(0, cut), slice(cut, None)):
            e.set_packets(w.x[sl], w.y[sl], w.k[sl], w.l[sl])
            e.step(S.SCHEME_LEAPFROG, w.dt, 10)
            parts.append(np.stack(e.get_packets()))
        assert np.array_equal(np.concatenate(parts, axis=1), full)
        ref10 = CO.leapfrog_spectral(w.x[sub], w.y[sub], w.k[sub], w.l[sub], planes, w.dx, w.nx, w.f, w.gH, w.dt, 10)
        assert np.abs(full[:, sub] - np.stack(ref10)).max() < TOL_TRAJ
        assert np.all(np.isfinite(full))


def test_C3_full_size_two_frame_blend():
    # BASELINE configs[2]: 256^2, time-evolving flow (two frames blended on the device), 1M packets
    w = W.make_workload("C3")
    m = 2
    p1 = W.planes_from_psik(w.psik, w.L); p2 = W.planes_from_psik(w.psik2, w.L)
    sub = np.arange(0, w.n_packets, 9973)
    st = tuple(a[sub] for a in (w.x, w.y, w.k, w.l))
    for j in range(m):
        al = (j + 0.5) / m
        pl = [(1 - al) * u + al * v for u, v in zip(p1, p2)]
        st = CO.leapfrog_spectral(*st, pl, w.dx, w.nx, w.f, w.gH, w.dt / m, 1, precise=True)
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(w.psik, slot=0); e.set_flow_spectral(w.psik2, slot=1)
        assert e.contracted_planes() == 3
        e.set_packets(w.x, w.y, w.k, w.l)
        e.step(S.SCHEME_LEAPFROG, w.dt / m, m, alpha0=0.5 / m, dalpha=1.0 / m)
        got = np.stack(e.get_packets())
        assert np.abs(got[:, sub] - np.stack(st)).max() < TOL_TRAJ
        assert np.all(np.isfinite(got))
        # histogram of all 1M packets: counts add up, and equal the host histogram of the returned k,l
        om = np.sqrt(w.f ** 2 + w.gH * (got[2] ** 2 + got[3] ** 2))
        edges = O.matlab_linspace(0, om.max(), 300)
        c = e.hist_omega(edges)
        assert int(c.sum()) == w.n_packets and np.array_equal(c, O.histcounts(om, edges))


def test_C4_shard_size_L20_shear():
    # BASELINE configs[3]: 512^2, L = 20, mean shear on u (qg2layersw_raytrace.m:13,28,187-188); one GPU's
    # shard of the 16M packets (2M).  Checked on a subsample against the long-double CPU sum.
    w = W.make_workload("C4", n_packets=2 * 1024 * 1024)
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean)
    sub = np.arange(0, w.n_packets, 40009)
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(w.psik, u_mean=w.u_mean)
        e.set_packets(w.x, w.y, w.k, w.l)
        got = e.eval()
        ref = CO.spectral_eval(w.x[sub], w.y[sub], planes, w.dx, w.nx, precise=True)
        assert scaled_err(got[:, sub], ref) < TOL_FIELD
        assert abs(got[0].mean() - w.u_mean) < 0.05           # the mean shear is there
        e.step(S.SCHEME_LEAPFROG, w.dt, 1)
        st = CO.leapfrog_spectral(w.x[sub], w.y[sub], w.k[sub], w.l[sub], planes, w.dx, w.nx, w.f, w.gH, w.dt, 1)
        assert np.abs(np.stack(e.get_packets())[:, sub] - np.stack(st)).max() < TOL_TRAJ


@pytest.mark.parametrize("mode", [S.MODE_LAGRANGE6, S.MODE_SPECTRAL])
def test_C5_step_packet_xka_large(mode):
    # BASELINE configs[4]: step_packet_xka with amplitude transport on a geostrophic [u,v,eta] state
    # (synthetic: the bundled wavevort restart frame is not in the reference tree), 256^2.
    n = 4 * 1024 * 1024 if mode == S.MODE_LAGRANGE6 else 256 * 1024
    w = W.make_workload("C5", n_packets=n)
    planes = W.planes_from_psik(w.psik, w.L, etak=w.extra["etak"])
    sub = np.arange(0, n, max(1, n // 150))
    a0 = np.ones(n)
    with S.Engine(w.nx, w.L, w.f, w.gH, mode) as e:
        e.set_flow_planes_spectral(planes)
        e.set_packets(w.x, w.y, w.k, w.l, a0)
        e.step(S.SCHEME_RK4_XKA, w.dt, 2)
        got = np.stack(e.get_packets(with_a=True))
    st = tuple(v[sub] for v in (w.x, w.y, w.k, w.l, a0))
    if mode == S.MODE_LAGRANGE6:
        grids = [O.k2g(p) for p in planes]
        ref = CO.rk4_lagrange(*st, grids, w.dx, w.f, w.Cg, w.dt, 2, True)
    else:
        ref = st
        for _ in range(2):
            ref = O.rk4_step_batch(*ref, w.dt, w.Cg, w.f, None, w.dx, True, mode="spectral", planes_k=planes, nx=w.nx)
    assert np.abs(got[:, sub] - np.stack(ref)).max() < TOL_TRAJ
    assert np.all(np.isfinite(got)) and np.abs(got[4] - 1).max() > 1e-6      # wave action does evolve


def test_omega_drift_and_conserved_absolute_frequency():
    # steady flow: Omega = omega + U.k is conserved by the ray equations; the leapfrog keeps the drift
    # bounded and shrinking with dt (images/Symplectic_error: <~ 5e-3 at dt = 0.01 for a weak flow)
    w = W.make_workload("C2", n_packets=4096, nx=64, kind="band")
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(w.psik)
        worst = {}
        for dt, nst in ((0.01, 100), (0.005, 200)):
            e.set_packets(w.x, w.y, w.k, w.l)
            om0, Om0 = e.omega()
            worst[dt] = 0.0
            for _ in range(4):
                e.step(S.SCHEME_LEAPFROG, dt, nst)
                om, Om = e.omega()
                worst[dt] = max(worst[dt], np.abs((Om - Om0) / Om0).max())
        assert worst[0.01] < 5e-2                      # U_g = 0.5, |k| <= 8: a strong, sharp flow
        # the reference's phi2 is an explicit Euler step of H2 = U.k (ode_symplectic.m:18-21: x and k both
        # advance from the same x1), so the composite is FIRST order: the drift halves with dt
        # (CPU oracle on the same inputs: 1.6e-2, 8.4e-3, 4.3e-3 at dt = 0.01, 0.005, 0.0025)
        assert 0.35 * worst[0.01] < worst[0.005] < 0.65 * worst[0.01]
        assert np.abs(om - om0).max() > 1e-3           # intrinsic frequency does change (refraction happens)
        d = e.diag()
        assert d[4] == 0 and d[6] == 4096 and abs(d[0] - om.sum()) < 1e-8 * om.sum() and abs(d[1] - Om.sum()) < 1e-8 * abs(Om.sum())
        assert d[2] == om.max() and d[3] == om.min()


# ------------------------------------------------------------------------------------------------
# P6: histogram
# ------------------------------------------------------------------------------------------------
def test_histogram_bit_exact():
    nx = int(GOLD["nx"]); L = float(GOLD["L"])
    with S.Engine(nx, L, F0, GH0) as e:
        e.set_flow_spectral(GOLD["psik"])
        e.set_packets(GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"])
        c = e.hist_omega(GOLD["hist_edges"])
        assert np.array_equal(c, GOLD["hist_counts"])
        c2 = e.hist_omega(GOLD["hist_edges"], counts=c.copy())      # accumulate
        assert np.array_equal(c2, 2 * GOLD["hist_counts"])
        # larger, after stepping: identical states -> identical counts (load_data.m:33-49 rule)
        rs = np.random.RandomState(4)
        n = 200000
        k = rs.normal(0, 3, n); l = rs.normal(0, 3, n)
        e.set_packets(rs.uniform(-3, 3, n), rs.uniform(-3, 3, n), k, l)
        om, Om = e.omega()
        assert np.array_equal(om, np.sqrt(F0 * F0 + GH0 * (k * k + l * l)))
        edges = O.matlab_linspace(0, om.max(), 300)
        assert np.array_equal(e.hist_omega(edges), O.histcounts(om, edges))
        assert int(e.hist_omega(edges).sum()) == n                  # max lands in the closed last bin
        edges_abs = O.matlab_linspace(Om.min(), Om.max(), 300)
        assert np.array_equal(e.hist_omega(edges_abs, kind=S.HIST_ABSOLUTE), O.histcounts(Om, edges_abs))


# ------------------------------------------------------------------------------------------------
# edge cases and error behaviour
# ------------------------------------------------------------------------------------------------
def test_edge_cases_empty_single_ragged_nonfinite():
    nx = 32; L = 2 * np.pi
    psik, planes = make_flow(nx)
    for mode in (S.MODE_SPECTRAL, S.MODE_LAGRANGE6, S.MODE_NUFFT):
        with S.Engine(nx, L, F0, GH0, mode) as e:
            e.set_flow_spectral(psik)
            z = np.zeros(0)
            e.set_packets(z, z, z, z)
            e.step(S.SCHEME_LEAPFROG, 0.01, 3)                     # empty: no-op
            assert e.eval().shape == (6, 0)
            for n in (1, 7, 8, 63, 64, 65, 129):                    # around the 8/64/128 tile edges
                x, y, k, l = make_packets(n, L, seed=n)
                e.set_packets(x, y, k, l)
                ref = (CO.spectral_eval(x, y, planes, L / nx, nx) if mode != S.MODE_LAGRANGE6
                       else CO.interpolate6(x, y, [O.k2g(p) for p in planes], L / nx))
                assert scaled_err(e.eval(), ref) < TOL_FIELD
            # huge and negative positions reduce exactly like mod(x/dx, nx)
            x = np.array([1e6 + 0.123, -1e6 - 0.456, 0.0, -1e-20, L, -L]); y = x[::-1].copy()
            ref = (CO.spectral_eval(x, y, planes, L / nx, nx) if mode != S.MODE_LAGRANGE6
                   else CO.interpolate6(x, y, [O.k2g(p) for p in planes], L / nx))
            assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD
            # a non-finite packet is counted by the sentinel and does not poison the others
            x, y, k, l = make_packets(100, L)
            k2 = k.copy(); k2[17] = np.nan
            e.set_packets(x, y, k2, l)
            e.step(S.SCHEME_LEAPFROG, 0.01, 2)
            d = e.diag()
            assert d[4] == 1 and d[6] == 100
            xs, _, ks, _ = e.get_packets()
            assert np.isfinite(np.delete(ks, 17)).all() and np.isfinite(np.delete(xs, 17)).all()
            # non-finite POSITIONS (the quad kernels index the grid from them): no fault, neighbours untouched
            x2 = x.copy(); x2[3] = np.inf; x2[40] = np.nan; x2[77] = 1e300
            e.set_packets(x2, y, k, l)
            e.step(S.SCHEME_LEAPFROG, 0.01, 2)
            xs, ys, ks, _ = e.get_packets()
            good = np.ones(100, bool); good[[3, 40]] = False
            assert np.isfinite(xs[good]).all() and np.isfinite(ks[good]).all() and not np.isfinite(xs[~good]).any()


def test_error_behaviour():
    with pytest.raises(S.SwrtError) as ei:
        S.Engine(33, 1.0, 1.0, 1.0)
    assert ei.value.code == -1
    with S.Engine(32, 2 * np.pi, F0, GH0) as e:
        z = np.zeros(4)
        e.set_packets(z, z, z, z)
        with pytest.raises(S.SwrtError) as ei:
            e.step(S.SCHEME_LEAPFROG, 0.1, 1)                       # no flow
        assert ei.value.code == -2
        with pytest.raises(S.SwrtError):
            e.set_flow_spectral(np.zeros((15, 8), dtype=complex))    # wrong shape
        e.set_flow_spectral(np.zeros((31, 16), dtype=complex))
        with pytest.raises(S.SwrtError):
            e.step(99, 0.1, 1)
        with pytest.raises(S.SwrtError):
            e.hist_omega(np.array([1.0]))
        assert e.launch_count() > 0


# ------------------------------------------------------------------------------------------------
# the reference calling surface (SpectralScheme / ode_symplectic / grid_U / g2k / k2g)
# ------------------------------------------------------------------------------------------------
def test_reference_surface_spectral_scheme_and_ode_symplectic():
    nx = 32; L = 2 * np.pi
    psik, planes = make_flow(nx)
    psi = O.k2g(psik)
    n = 41
    x0 = np.zeros((1, 2, n)); k0 = np.zeros((1, 2, n))
    x0[0, 0], x0[0, 1], k0[0, 0], k0[0, 1] = make_packets(n, L)
    dt = 0.02; T = 0.5
    for mode, omode in ((S.MODE_SPECTRAL, "spectral"), (S.MODE_LAGRANGE6, "lagrange")):
        sch = R.SpectralScheme(L, nx, psi, mode=mode)
        osch = O.SpectralScheme(L, nx, psi, mode=omode)
        assert np.abs(sch.U(x0) - osch.U(x0)).max() < 1e-12
        g, og = sch.grad_U(x0), osch.grad_U(x0)
        for name in og:
            assert np.abs(g[name] - og[name]).max() < 1e-11
        assert np.abs(sch.grad_U_times_k(x0, k0) - osch.grad_U_times_k(x0, k0)).max() < 1e-11
        xs, ks, ts = R.ode_symplectic(x0, k0, dt, T, F0, GH0, sch)
        xo, ko, to = O.ode_symplectic(x0, k0, dt, T, F0, GH0, osch)
        assert xs.shape == xo.shape == (25, 2, n) and np.allclose(ts, to)
        assert np.abs(xs - xo).max() < TOL_TRAJ and np.abs(ks - ko).max() < TOL_TRAJ
        xs5, ks5, ts5 = R.ode_symplectic(x0, k0, dt, T, F0, GH0, sch, save_stride=5)
        assert np.array_equal(xs5, xs[::5]) and np.allclose(ts5, ts[::5])
    assert np.abs(sch.streamfunction(x0[0, 0], x0[0, 1]) - osch.streamfunction(x0[0, 0], x0[0, 1])).max() < 1e-12


def test_device_g2k_k2g_grid_U():
    nx = 64
    psik, planes = make_flow(nx)
    fg = O.k2g(planes[0])
    assert np.abs(S.k2g_dev(planes[0]) - fg).max() < 1e-13 * max(1, np.abs(fg).max())
    assert np.abs(S.g2k_dev(fg) - O.symmetrise_ky0(planes[0])).max() < 1e-15
    kx_, ky_ = O.wavenumbers(nx)
    K2 = kx_ ** 2 + ky_ ** 2
    qk = -(3.0 + K2) * psik
    bf = R.grid_U(qk, 3.0, K2, kx_, ky_, 0.5)
    ref = O.grid_U(qk, 3.0, K2, kx_, ky_, 0.5)
    for name in ref:
        assert np.abs(bf[name] - ref[name]).max() < 1e-12


# ------------------------------------------------------------------------------------------------
# "next" row f2: the production drivers' ode23 solve (qgsw_raytrace.m:143-150)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [S.MODE_LAGRANGE6, S.MODE_SPECTRAL])
def test_ode23_flow_step_matches_oracle(mode):
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx
    kx_, ky_ = O.wavenumbers(nx)
    p1 = O.velocity_planes_k(GOLD["psik"], kx_, ky_); p2 = O.velocity_planes_k(GOLD["psik2"], kx_, ky_)
    names = ("u", "v", "ux", "uy", "vx", "vy")
    bf1 = dict(zip(names, [O.k2g(p) for p in p1])); bf2 = dict(zip(names, [O.k2g(p) for p in p2]))
    x, y, k, l = GOLD["x"], GOLD["y"], GOLD["k"], GOLD["l"]
    n = x.size
    tmax = 0.4                                # one (long) flow step, so that the controller takes several steps
    if mode == S.MODE_LAGRANGE6:
        ode = O.generate_raytracing_ode(bf1, bf2, n, F0, 1.0, tmax, dx, bump=O.BUMP_LIVE)     # the engine below runs its default bump
    else:
        ev = lambda xx, yy, al: CO.spectral_eval(xx, yy, [(1 - al) * a + al * b for a, b in zip(p1, p2)], dx, nx)
        ode = O.generate_raytracing_ode(None, None, n, F0, 1.0, tmax, dx, eval6=ev)
    yref, sref = O.ode23(ode, [0, tmax], np.concatenate([x, y, k, l]))
    with S.Engine(nx, L, F0, GH0, mode) as e:
        e.set_flow_spectral(GOLD["psik"], slot=0); e.set_flow_spectral(GOLD["psik2"], slot=1)
        e.set_packets(x, y, k, l)
        st = R.ode23(e, [0, tmax], tmax)
        got = np.concatenate(e.get_packets())
        assert (st["nsteps"], st["nfailed"], st["nfevals"]) == (sref["nsteps"], sref["nfailed"], sref["nfevals"])
        assert st["nsteps"] >= 10              # MaxStep = 0.1*(tf - t0)
        assert np.abs(got - yref).max() < TOL_TRAJ
        # tighter tolerances: more steps, same agreement
        e.set_packets(x, y, k, l)
        st2 = R.ode23(e, [0, tmax], tmax, rtol=1e-6, atol=1e-7)      # SW_zero_background_raytracing.m:71-72
        yref2, sref2 = O.ode23(ode, [0, tmax], np.concatenate([x, y, k, l]), rtol=1e-6, atol=1e-7)
        # At RelTol 1e-6 the estimator sits at the kinks of the piecewise-polynomial Lagrange interpolant, so
        # accept/reject decisions hinge on 1e-16-level differences: the two runs may take slightly different
        # step sequences, each a valid solution to the requested tolerance.
        assert st2["nsteps"] > st["nsteps"] and abs(st2["nsteps"] - sref2["nsteps"]) <= 0.1 * sref2["nsteps"]
        assert np.abs(np.concatenate(e.get_packets()) - yref2).max() < (TOL_TRAJ if mode == S.MODE_SPECTRAL else 1e-5)
        with pytest.raises(S.SwrtError):
            e.set_packets(x, y, k, l)
            e.bs23_attempt(0.1, [0, 0, 0], 1e-3)          # attempt without begin after new packets


def test_ode23_error_norm_couples_all_packets():
    # one stiff packet (huge k) shrinks everybody's step: the reference solves ONE 4*Np system
    nx = int(GOLD["nx"]); L = float(GOLD["L"])
    x, y, k, l = (GOLD[q].copy() for q in ("x", "y", "k", "l"))
    with S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(GOLD["psik"] * 20)
        e.set_packets(x, y, k, l)
        base = R.ode23(e, [0, 0.5], np.inf)              # steady flow: alpha = t/inf = 0
        k[3] *= 300.0
        e.set_packets(x, y, k, l)
        stiff = R.ode23(e, [0, 0.5], np.inf)
        assert stiff["nsteps"] > base["nsteps"]


def test_ideal_omega_distribution_theoretical_pdf():
    # "next" row f4 (ideal_omega_distribution.m:3-11): counts over (grid point, angle), bit-exact against a host
    # histogram of the same U; pdf integrates to one; mean sits at omega_0 (the flow has zero mean)
    nx = 64; L = 2 * np.pi; f, Cg, k0 = 3.0, 1.0, 3.0
    psik, planes = make_flow(nx)
    psi = O.k2g(psik)
    for mode in (S.MODE_SPECTRAL, S.MODE_LAGRANGE6):
        sch = R.SpectralScheme(L, nx, psi, mode=mode)
        X = O.matlab_linspace(0.0, L, nx); XX, YY = np.meshgrid(X, X)
        U = sch.U(np.stack([XX.ravel(order="F"), YY.ravel(order="F")], axis=1))
        t = O.matlab_linspace(0, 2 * np.pi, 100)
        om0 = np.sqrt(f * f + Cg * Cg * k0 * k0)
        om_abs = om0 + (np.outer(U[:, 0], k0 * np.cos(t)) + np.outer(U[:, 1], k0 * np.sin(t)))
        edges = O.matlab_linspace(om_abs.min(), om_abs.max(), 61)
        counts, pdf = R.ideal_omega_distribution(sch, f, Cg, k0, edges)
        assert np.array_equal(counts, O.histcounts(om_abs, edges))
        assert int(counts.sum()) == nx * nx * 100
        assert abs((pdf * np.diff(edges)).sum() - 1.0) < 1e-12
        centre = (edges[1:] + edges[:-1]) / 2
        assert abs((pdf * np.diff(edges) * centre).sum() - om0) < 0.05


def test_device_qg_frame_producer_and_time_evolving_run():
    # "next" row f3: the one-layer QG solver of qgsw_raytrace.m:111-137,270-286 on the device, feeding the two
    # flow slots without a host copy; packets advanced per flow step with frame blending (config C3's shape)
    nx = 64; L = 2 * np.pi; f, Cg = 3.0, 1.0; K_d2 = f / Cg
    xg = O.matlab_linspace(-L / 2, L / 2, nx)
    X, Y = np.meshgrid(xg, xg)
    q0 = O.initial_q(X, Y, 0.5, K_d2, O.matlab_rand_stream(146))
    qk0 = O.g2k(q0)
    kx_, ky_ = O.wavenumbers(nx); K2 = kx_ ** 2 + ky_ ** 2
    flow = O.grid_U(qk0, K_d2, K2, kx_, ky_)
    U0 = np.sqrt((flow["u"] ** 2 + flow["v"] ** 2).max())
    dt = 0.05 * (L / nx) / U0                                  # qgsw_raytrace.m:29,70
    # update() as written adds the constant source r_drag*K2 to every mode (qgsw_raytrace.m:285); with the
    # driver's r_drag = 0.1 the restated solver overflows within ~12 steps on this grid, so the parity run uses
    # r_drag = 0.01 (12 steps: Euler, AB2, then AB3; |q| grows 3x) -- the term itself is still exercised
    rd = 0.01
    qg = S.QGFlow(nx, L, qk0, K_d2, dt, f, Cg, r_drag=rd)
    nsteps = 12
    ref = O.qg_run(qk0, nsteps, dt, nx, L, K_d2, f, Cg, r_drag=rd)
    qg.step(nsteps)
    got = qg.get()
    assert np.abs(got - ref).max() < 1e-10 * np.abs(ref).max()
    # flow slots straight from the device state == uploading psi-hat from the host
    x, y, k, l = make_packets(300, L)
    with S.Engine(nx, L, f, Cg ** 2) as e, S.Engine(nx, L, f, Cg ** 2) as e2:
        qg.to_flow(e, 0)
        e2.set_flow_spectral(-got / (K_d2 + K2))
        assert np.abs(e.eval_at(x, y) - e2.eval_at(x, y)).max() < 1e-13
        # one flow step of the production loop: frame 0 = prev_qk, frame 1 = qk (qgsw_raytrace.m:141-143)
        qg.step(1)
        qg.to_flow(e, 1)
        e.set_packets(x, y, k, l)
        st = R.ode23(e, [0, dt], dt)
        p1 = O.velocity_planes_k(-got / (K_d2 + K2), kx_, ky_)
        p2 = O.velocity_planes_k(-O.qg_run(qk0, nsteps + 1, dt, nx, L, K_d2, f, Cg, r_drag=rd) / (K_d2 + K2), kx_, ky_)
        ev = lambda xx, yy, al: CO.spectral_eval(xx, yy, [(1 - al) * a + al * b for a, b in zip(p1, p2)], L / nx, nx)
        yref, sref = O.ode23(O.generate_raytracing_ode(None, None, x.size, f, Cg, dt, L / nx, eval6=ev), [0, dt], np.concatenate([x, y, k, l]))
        assert st["nsteps"] == sref["nsteps"] and np.abs(np.concatenate(e.get_packets()) - yref).max() < TOL_TRAJ
    qg.close()


def test_qgsw_raytrace_driver_on_device(tmp_path):
    # the reference's production driver signature (qgsw_raytrace.m:1) end to end: QG frames, flow slots and the
    # per-step ode23 packet solve on the GPU, packet frames in the reference's file format
    from swraytracing_b200 import drivers, fieldio
    nx, Np, nif, U_g, f, Cg = 32, 12, 2.0, 0.5, 3.0, 1.0
    nst = 6
    out = drivers.qgsw_raytrace(nx, Np, nif, 6000, 0, U_g, f, Cg, outdir=str(tmp_path), max_steps=nst, r_drag=0.01, log=lambda s: None)
    # --- oracle-side restatement of the same loop
    L = 2 * np.pi; K_d2 = f / Cg
    xg = O.matlab_linspace(-L / 2, L / 2, nx); X, Y = np.meshgrid(xg, xg)
    rs = O.matlab_rand_stream(146)
    qk0 = O.g2k(O.initial_q(X, Y, U_g, K_d2, rs))
    x, y, k, l = O.init_packets(Np, L, np.sqrt((nif ** 2 - 1) * f ** 2 / Cg ** 2), rs)
    kx_, ky_ = O.wavenumbers(nx); K2 = kx_ ** 2 + ky_ ** 2
    fl = O.grid_U(qk0, K_d2, K2, kx_, ky_)
    U0 = np.sqrt((fl["u"] ** 2 + fl["v"] ** 2).max()); dt = 0.05 * (L / nx) / U0
    assert abs(out["dt"] - dt) < 1e-15 and abs(out["U0"] - U0) < 1e-13
    yv = np.concatenate([x, y, k, l])
    for step in range(1, nst + 1):
        p1 = O.velocity_planes_k(-O.qg_run(qk0, step - 1, dt, nx, L, K_d2, f, Cg, r_drag=0.01) / (K_d2 + K2), kx_, ky_)
        p2 = O.velocity_planes_k(-O.qg_run(qk0, step, dt, nx, L, K_d2, f, Cg, r_drag=0.01) / (K_d2 + K2), kx_, ky_)
        ev = lambda xx, yy, al: CO.spectral_eval(xx, yy, [(1 - al) * a + al * b for a, b in zip(p1, p2)], L / nx, nx)
        yv, _ = O.ode23(O.generate_raytracing_ode(None, None, Np, f, Cg, dt, L / nx, eval6=ev), [0, dt], yv)
    assert np.abs(np.concatenate(out["packets"]) - yv).max() < TOL_TRAJ
    assert out["packet_steps"] == nst and out["ode23_steps"] >= 10 * nst
    # files: initial frame + one frame when mod(step - packet_step_start + 1, 5) == 0, i.e. step 4 with
    # packet_step_start = ceil(0/dt) = 0 (qgsw_raytrace.m:73,153); wrapped positions
    t, xs, ks = fieldio.load_packet_frames(tmp_path, Np)
    assert xs.shape == (Np, 2, 2) and abs(t[1] - 4 * dt) < 1e-12 and np.abs(xs).max() <= L / 2
    assert np.array_equal(ks[:, 0, 0], k)


@pytest.mark.gpu
def test_hist_pipeline_matches_blocking_histogram(small_flow, packets):
    """HistPipeline (non-blocking histogram launch + snapshot, results two rotations later) returns exactly the
    counts of the blocking swrt_hist_omega for every interval, in order"""
    import swraytracing_b200 as S
    from swraytracing_b200.distributed import ShardedEnsemble
    eng = S.Engine(small_flow["nx"], small_flow["L"], 3.0, 1.0, S.MODE_SPECTRAL)
    eng.set_flow_spectral(small_flow["psik"])
    eng.set_packets(packets["x"], packets["y"], packets["k"], packets["l"])
    ens = ShardedEnsemble(eng, packets["n"])
    edges = np.linspace(0.0, 9.0, 300)
    pipe = ens.hist_pipeline(edges)
    want, got = [], []
    for it in range(5):
        eng.step_async(S.SCHEME_LEAPFROG, 0.01, 3)
        r = pipe.rotate()
        if r is not None:
            got.append(r)
        pipe.launch()
        want.append(eng.hist_omega(edges))            # blocking reference of the same state
    got += pipe.drain()
    assert len(got) == 5
    for g, w_ in zip(got, want):
        assert np.array_equal(g, w_) and int(g.sum()) <= packets["n"]
    eng.close()


# ------------------------------------------------------------------------------------------------
# LAGRANGE6 = the reference's double arithmetic, operation for operation (steady flow): bit-identical
# ------------------------------------------------------------------------------------------------
def _bit_equal(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _ulps(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float((np.abs(a - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)))).max())


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [16, 64])
def test_lagrange_mode_is_bit_identical_to_the_restatement(nx):
    """interpolate.m's weights (multiply by (a-j+bump), divide by (j-i), five times), the i-outer/j-inner 36-term sum
    without fused multiply-adds, ode_symplectic's drift/kick expressions, step_packet's and step_packet_xka's RK4
    stages: the kernel executes the same IEEE operations in the same order as the line-by-line restatement, so every
    output double is the same double -- not merely within 1e-12."""
    L = 2 * np.pi; dx = L / nx
    psik, planes = make_flow(nx)
    grids = [O.k2g(p) for p in planes]
    n = 513
    rs = np.random.RandomState(nx)
    x = rs.uniform(-3 * L, 3 * L, n); y = rs.uniform(-3 * L, 3 * L, n)
    x[:4] = [0.0, -dx, 5 * dx, L]; y[:4] = [0.0, 2 * dx, -L, 7 * dx - 1e-14]        # grid nodes, wrap, negative side
    k = 3 * np.cos(np.arange(n) * 0.37); l = 3 * np.sin(np.arange(n) * 0.37)
    # (1) interpolate(x,y,F,dx,dy), both bumps
    for bump, ref_fn in ((1e-13, O.interpolate), (1e-10, O.interpolate_par)):
        got = S.interpolate_dev(x, y, grids[0], dx, dx, bump)
        assert _bit_equal(got, ref_fn(x, y, grids[0], dx, dx)), _ulps(got, ref_fn(x, y, grids[0], dx, dx))
    with S.Engine(nx, L, F0, GH0, S.MODE_LAGRANGE6) as e:
        e.set_flow_grid(*grids)
        # (2) the six planes of SpectralScheme.U / grad_U
        got = e.eval_at(x, y)
        for c in range(6):
            assert _bit_equal(got[c], O.interpolate(x, y, grids[c], dx, dx)), (c, _ulps(got[c], O.interpolate(x, y, grids[c], dx, dx)))
        # (3) ode_symplectic: 25 leapfrog steps
        dt = 0.1 * dx
        e.set_packets(x, y, k, l)
        e.step(S.SCHEME_LEAPFROG, dt, 25)
        got = e.get_packets()
        ev = lambda xx, yy: tuple(O.interpolate(xx, yy, g, dx, dx) for g in grids)
        ref = (x, y, k, l)
        for _ in range(25):
            ref = O.leapfrog_step(*ref, dt, F0, GH0, ev)
        for g_, r_, name in zip(got, ref, "xykl"):
            assert _bit_equal(g_, r_), (name, _ulps(g_, r_))
    # (3b) two flow frames: interpolate_U interpolates BOTH frames and blends the results (interpolate_U.m:19-23); odefun
    psik2, planes2 = make_flow(nx, seed=8)
    grids2 = [O.k2g(p) for p in planes2]
    names = ("u", "v", "ux", "uy", "vx", "vy")
    bf1 = dict(zip(names, grids)); bf2 = dict(zip(names, grids2))
    with S.Engine(nx, L, F0, 1.0, S.MODE_LAGRANGE6) as e:
        e.set_flow_grid(*grids, slot=0); e.set_flow_grid(*grids2, slot=1)
        for alpha in (0.0, 0.37, 1.0):
            U, nab = O.interpolate_U(bf1, bf2, alpha, np.stack([x, y], axis=1), dx, bump=O.BUMP_LIVE)
            got = e.eval_at(x, y, alpha)
            want = [U[:, 0], U[:, 1], nab["u_x"], nab["u_y"], nab["v_x"], nab["v_y"]]
            for c in range(6):
                assert _bit_equal(got[c], want[c]), (alpha, c, _ulps(got[c], want[c]))
        e.set_packets(x, y, k, l)
        d = e.rhs(0.37)
        ref = O.odefun_rhs(x, y, k, l, 0.37, bf1, bf2, F0, 1.0, dx, bump=O.BUMP_LIVE)
        for g_, r_, name in zip(d, ref, ("dxdt", "dydt", "dkdt", "dldt")):
            assert _bit_equal(g_, r_), (name, _ulps(g_, r_))
        # the pre-blend tuning (one blended grid, half the gathers) agrees to rounding, not to the bit
        e.set_tuning(0, preblend_grid=True)
        fast = e.eval_at(x, y, 0.37)
        U, nab = O.interpolate_U(bf1, bf2, 0.37, np.stack([x, y], axis=1), dx, bump=O.BUMP_LIVE)
        assert scaled_err(fast, np.stack([U[:, 0], U[:, 1], nab["u_x"], nab["u_y"], nab["v_x"], nab["v_y"]])) < 1e-13
    # (4) step_packet / step_packet_xka: 3 RK4 steps of a few packets through the reference's own per-packet functions
    H = 1.0 + 0.2 * grids[0] / np.abs(grids[0]).max()
    U = {"u": grids[0], "v": grids[1]}; G = {"u_x": grids[2], "u_y": grids[3], "v_x": grids[4], "v_y": grids[5]}
    dt = 0.3 * dx
    for xka in (False, True):
        with S.Engine(nx, L, F0, 1.0, S.MODE_LAGRANGE6) as e:
            e.set_flow_grid(*grids, H=H if xka else None)
            m = 12
            e.set_packets(x[:m], y[:m], 10 * k[:m], 10 * l[:m], np.ones(m))
            e.step(S.SCHEME_RK4_XKA if xka else S.SCHEME_RK4_PACKET, dt, 3)
            got = e.get_packets(with_a=True)
        for p in range(m):
            P = {"x": x[p], "y": y[p], "k": 10 * k[p], "l": 10 * l[p], "a": 1.0}
            for _ in range(3):
                P = {**P, **(O.step_packet_xka(P, U, G, H, 1.0, F0, dx, dx, dt) if xka else O.step_packet(P, U, G, 1.0, F0, dx, dx, dt))}
            for j, name in enumerate(("x", "y", "k", "l") + (("a",) if xka else ())):
                assert got[j][p] == P[name], (xka, p, name, got[j][p], P[name])


@pytest.mark.gpu
def test_scheme_diagnostics_and_difference_scheme_cross_check():
    """product SpectralScheme (device) vs the reference's independent DifferenceScheme on the analytic
    Childress-Soward streamfunction, and the inherited RaytracingScheme diagnostics vs the oracle scheme"""
    nx, L, U0, km, a = 64, 2 * np.pi, 0.1, 4.0, 0.25
    psi, _, _ = O.childress_soward(nx, L, U0, km, a)
    ds = O.DifferenceScheme(lambda x, y, t: U0 / km * (np.sin(km * x) * np.sin(km * y) + a * np.cos(km * x) * np.cos(km * y)))
    x = np.random.RandomState(0).uniform(-5, 5, (200, 2))
    for mode, omode, tolU in ((S.MODE_SPECTRAL, "spectral", 1e-10), (S.MODE_LAGRANGE6, "lagrange", 1e-4)):
        sch = R.SpectralScheme(L, nx, psi, mode=mode)
        osch = O.SpectralScheme(L, nx, psi, mode=omode)
        assert np.abs(sch.U(x) - ds.U(x)).max() < tolU
        assert np.abs(sch.vorticity(x) - osch.vorticity(x)).max() < 1e-12
        assert np.abs(sch.strain(x) - osch.strain(x)).max() < 1e-12
        assert np.abs(sch.okuboWeiss(x) - osch.okuboWeiss(x)).max() < 1e-12
    zeta = -2 * km ** 2 * ds.streamfunction(x[:, 0], x[:, 1])
    assert np.abs(R.SpectralScheme(L, nx, psi).vorticity(x) - zeta).max() < 1e-12


# ------------------------------------------------------------------------------------------------
# NUFFT mode: the same exact Fourier series as SPECTRAL (P2 contract), evaluated by a type-2 non-uniform FFT
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nx", [16, 32, 36, 48, 64, 128, 256])
def test_nufft_eval_vs_exact_sum(nx):
    L = 2 * np.pi; dx = L / nx
    psik, planes = make_flow(nx)
    n = 517 if nx <= 64 else 200
    x, y, k, l = make_packets(n, L)
    x[:4] = [0.0, -dx, 5 * dx, L]; y[:4] = [0.0, 2 * dx, -L, 7 * dx]                 # grid nodes: kernel argument hits |z| = 1
    ref = CO.spectral_eval(x, y, planes, dx, nx, precise=True)
    with S.Engine(nx, L, F0, GH0, S.MODE_NUFFT) as e:
        e.set_flow_spectral(psik)
        e.set_packets(x, y, k, l)
        got = e.eval()
        assert scaled_err(got, ref) < TOL_FIELD, [float(np.abs(got[c] - ref[c]).max() / np.abs(ref[c]).max()) for c in range(6)]
        assert np.array_equal(e.eval_at(x[::-1].copy(), y[::-1].copy())[:, ::-1], got)
        # the six planes handed over explicitly (grid_U output as coefficients) and as grids: same flow, same answer
        e.set_flow_planes_spectral(planes)
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD
        e.set_flow_grid(*[O.k2g(p) for p in planes])
        assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD


@pytest.mark.gpu
def test_nufft_white_spectrum_L20_shear_and_time_blend():
    # the hardest spectrum (flat up to the truncation), the two-layer driver's domain (L = 20, mean shear), two frames
    nx = 64; L = 20.0; dx = L / nx
    kap = 2 * np.pi / L
    kx_, ky_ = O.wavenumbers(nx)
    rs = np.random.RandomState(12)
    psis = [(rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) * 1e-3 for _ in range(2)]
    pl = []
    for p in psis:
        q = O.velocity_planes_k(p, kap * kx_, kap * ky_)
        q[0] = q[0].copy(); q[0][nx // 2 - 1, 0] += 0.5
        pl.append(q)
    x, y, k, l = make_packets(300, L, seed=2)
    with S.Engine(nx, L, F0, GH0, S.MODE_NUFFT) as e:
        e.set_flow_spectral(psis[0], slot=0, u_mean=0.5); e.set_flow_spectral(psis[1], slot=1, u_mean=0.5)
        for alpha in (0.0, 0.3, 1.0):
            blend = [(1 - alpha) * a + alpha * b for a, b in zip(pl[0], pl[1])]
            ref = CO.spectral_eval(x, y, blend, dx, nx, precise=True)
            assert scaled_err(e.eval_at(x, y, alpha), ref) < TOL_FIELD, alpha
        e.set_packets(x, y, k, l)
        d = np.stack(e.rhs(0.3))
        blend = [0.7 * a + 0.3 * b for a, b in zip(pl[0], pl[1])]
        want = np.stack(O.rhs_from_eval(CO.spectral_eval(x, y, blend, dx, nx, precise=True), k, l, F0, 1.0))
        assert scaled_err(d, want) < TOL_FIELD


@pytest.mark.gpu
def test_nufft_trajectories_ode23_and_rk4_match_spectral_oracle():
    nx = int(GOLD["nx"]); L = float(GOLD["L"]); dx = L / nx; dt = float(GOLD["dt"])
    psik, planes = make_flow(nx)
    x, y, k, l = make_packets(400, L)
    ref = CO.leapfrog_spectral(x, y, k, l, planes, dx, nx, F0, GH0, dt, 100)
    with S.Engine(nx, L, F0, GH0, S.MODE_NUFFT) as e, S.Engine(nx, L, F0, GH0, S.MODE_SPECTRAL) as es:
        for eng in (e, es):
            eng.set_flow_spectral(psik); eng.set_packets(x, y, k, l)
        e.step(S.SCHEME_LEAPFROG, dt, 100)
        assert np.abs(np.stack(e.get_packets()) - np.stack(ref)).max() < TOL_TRAJ
        # fused 100 steps == 100 single-step launches, bit for bit
        e.set_packets(x, y, k, l)
        for _ in range(100):
            e.step(S.SCHEME_LEAPFROG, dt, 1)
        e2 = np.stack(e.get_packets())
        e.set_packets(x, y, k, l); e.step(S.SCHEME_LEAPFROG, dt, 100)
        assert np.array_equal(e2, np.stack(e.get_packets()))
        # ode23 and step_packet run through the mode-independent stage code: same decisions / states as SPECTRAL mode
        for eng in (e, es):
            eng.set_packets(x, y, k, l)
        st, sts = R.ode23(e, [0.0, 20 * dt], None), R.ode23(es, [0.0, 20 * dt], None)
        assert (st["nsteps"], st["nfailed"]) == (sts["nsteps"], sts["nfailed"])
        assert np.abs(np.stack(e.get_packets()) - np.stack(es.get_packets())).max() < TOL_TRAJ
        for eng in (e, es):
            eng.set_packets(x, y, k, l); eng.step(S.SCHEME_RK4_PACKET, dt, 5)
        assert np.abs(np.stack(e.get_packets()) - np.stack(es.get_packets())).max() < TOL_TRAJ
        edges = np.linspace(0, 9, 300)
        assert np.array_equal(e.hist_omega(edges, kind=S.HIST_ABSOLUTE), es.hist_omega(edges, kind=S.HIST_ABSOLUTE))
        with pytest.raises(S.SwrtError):
            e.step(S.SCHEME_RK4_XKA, dt, 1)                               # this flow has no H plane


@pytest.mark.gpu
def test_nufft_step_packet_xka_matches_dense_spectral():
    """config 5 in NUFFT mode: u, v, H at the four RK4 stage positions and the seven planes at the new position come from
    the (u,v) and H fine grids; states equal the dense-contraction path to 1e-9, H itself to 1e-12"""
    w = W.make_workload("C5", n_packets=3000, nx=64)
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean, etak=w.extra["etak"])
    outs = []
    for mode in (S.MODE_SPECTRAL, S.MODE_NUFFT):
        with S.Engine(w.nx, w.L, w.f, w.gH, mode) as e:
            e.set_flow_planes_spectral(planes)
            ev = e.eval_at(w.x, w.y, with_H=True)
            e.set_packets(w.x, w.y, w.k, w.l, np.ones(w.n_packets))
            e.step(S.SCHEME_RK4_XKA, w.dt, 4)
            outs.append((ev, np.stack(e.get_packets(with_a=True))))
    assert scaled_err(outs[1][0], outs[0][0]) < TOL_FIELD
    assert np.abs(outs[1][1] - outs[0][1]).max() < TOL_TRAJ
    assert np.abs(outs[0][1][4] - 1.0).max() > 1e-6                      # the wave action actually evolved


@pytest.mark.gpu
@pytest.mark.parametrize("xka", [False, True])
def test_nufft_fused_rk4_kernel_equals_the_composed_launches(xka):
    """step_packet / step_packet_xka in NUFFT mode: the fused kernel (stages, evaluations, k / a update in one launch)
    against the evaluation + stage launches the dense mode composes (tuning flag): same expressions, so 1e-13 on the
    state; steady (6 steps in one launch) and two-frame (one launch per step, alpha advancing)"""
    w = W.make_workload("C5", n_packets=2500, nx=48)
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean, etak=w.extra["etak"])
    rs = np.random.RandomState(3)
    planes2 = [pl * np.exp(1j * rs.uniform(-0.05, 0.05, pl.shape)) for pl in planes]
    scheme = S.SCHEME_RK4_XKA if xka else S.SCHEME_RK4_PACKET
    for two_frames in (False, True):
        outs = []
        for unfused in (False, True):
            with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_NUFFT) as e:
                e.set_tuning(unfused_rk4=unfused)
                e.set_flow_planes_spectral(planes)
                if two_frames:
                    e.set_flow_planes_spectral(planes2, 1)
                e.set_packets(w.x, w.y, w.k, w.l, np.ones(w.n_packets))
                n0 = e.launch_count()
                if two_frames:
                    e.step(scheme, w.dt, 6, 1 / 12, 1 / 6)
                else:
                    e.step(scheme, w.dt, 6)
                outs.append((np.stack(e.get_packets(with_a=True)), e.launch_count() - n0))
        (fused, nl_f), (comp, nl_c) = outs
        assert np.abs(fused - comp).max() < 1e-13 * max(1.0, np.abs(comp).max())
        assert nl_f < nl_c
        if not two_frames:
            assert nl_f == 1
        if xka:
            assert np.abs(fused[4] - 1.0).max() > 1e-6


@pytest.mark.gpu
def test_nufft_full_size_C4_shard_agrees_with_dense_contraction():
    """512^2, L = 20, shear, two-frame blend: the dense DMMA contraction and the NUFFT gather are two evaluations of one
    Fourier series; on 4,096 packets of the C4 workload they agree to 1e-12 of max|plane|, and 16 leapfrog steps to 1e-9"""
    w = W.make_workload("C4", n_packets=4096)
    outs = []
    for mode in (S.MODE_SPECTRAL, S.MODE_NUFFT):
        with S.Engine(w.nx, w.L, w.f, w.gH, mode) as e:
            e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
            e.set_packets(w.x, w.y, w.k, w.l)
            ev = e.eval(0.4)
            e.step(S.SCHEME_LEAPFROG, w.dt / 16, 16, 1 / 32, 1 / 16)
            outs.append((ev, np.stack(e.get_packets())))
    assert scaled_err(outs[1][0], outs[0][0]) < TOL_FIELD
    assert np.abs(outs[1][1] - outs[0][1]).max() < TOL_TRAJ


@pytest.mark.gpu
@pytest.mark.parametrize("with_H", [False, True])
def test_lagrange_two_frame_sweep_equals_the_two_single_frame_gathers_bit_for_bit(with_H):
    """interpolate_U.m:5-23 in LAGRANGE6 mode: the two-frame kernels gather both frames in one sweep over the 36 nodes;
    every frame's plane must still be the same doubles as a single-frame gather of that frame (alpha = 0 / alpha = 1), and
    the blend the un-fused (1 - alpha)*F1 + alpha*F2 -- for six planes and for seven (H, odd record length); a 12-step
    two-frame leapfrog equals 12 single-step launches"""
    w = W.make_workload("C5", n_packets=3001, nx=48)
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean, etak=w.extra["etak"])
    rs = np.random.RandomState(11)
    planes2 = [pl * np.exp(1j * rs.uniform(-0.05, 0.05, pl.shape)) for pl in planes]
    if not with_H:
        planes, planes2 = planes[:6], planes2[:6]
    alpha = 0.3
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6) as e:
        e.set_flow_planes_spectral(planes, 0); e.set_flow_planes_spectral(planes2, 1)
        f1 = e.eval_at(w.x, w.y, 0.0, with_H=with_H)
        f2 = e.eval_at(w.x, w.y, 1.0, with_H=with_H)
        fb = e.eval_at(w.x, w.y, alpha, with_H=with_H)
        assert np.array_equal(fb, (1.0 - alpha) * f1 + alpha * f2)
        e.set_packets(w.x, w.y, w.k, w.l)
        e.step(S.SCHEME_LEAPFROG, w.dt, 12, 1 / 24, 1 / 12)
        fused = np.stack(e.get_packets())
        e.set_packets(w.x, w.y, w.k, w.l)
        for j in range(12):
            e.step(S.SCHEME_LEAPFROG, w.dt, 1, 1 / 24 + j * (1 / 12), 0.0)      # the doubles swrt_step forms: alpha0 + j*dalpha
        assert np.array_equal(fused, np.stack(e.get_packets()))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [S.MODE_LAGRANGE6, S.MODE_SPECTRAL, S.MODE_NUFFT])
def test_step_packet_xka_uniform_depth_zero_flow_closed_form_on_device(mode):
    """the closed form of tests/test_oracle_kat.py (rest state over a uniform depth: straight rays at the group velocity,
    k unchanged, wave action times the degree-4 Taylor polynomial of exp(-divC dt) per step) through swrt_step(RK4_XKA) in
    every mode; the flow planes are zero and H-hat has only its (0,0) coefficient"""
    nx = 32; L = 2 * np.pi; H0 = 1.3; gH = 0.81; f = 3.0; dt = 0.05; nsteps = 3
    nkx, nky = nx - 1, nx // 2
    planes = [np.zeros((nkx, nky), complex) for _ in range(7)]
    planes[6][nkx // 2, 0] = H0                                       # (kx, ky) = (0, 0)
    rs = np.random.RandomState(5)
    n = 777
    x = rs.uniform(-L / 2, L / 2, n); y = rs.uniform(-L / 2, L / 2, n)
    k = rs.uniform(-3, 3, n); l = rs.uniform(-3, 3, n); a0 = rs.uniform(0.5, 2.0, n)
    with S.Engine(nx, L, f, gH, mode) as e:
        e.set_flow_planes_spectral(planes)
        e.set_packets(x, y, k, l, a0)
        e.step(S.SCHEME_RK4_XKA, dt, nsteps)
        xo, yo, ko, lo, ao = e.get_packets(with_a=True)
    g = gH * H0
    om = np.sqrt(f ** 2 + g * (k ** 2 + l ** 2))
    Cx, Cy = g * k / om, g * l / om
    z = (Cx ** 2 + Cy ** 2) / om * dt
    tol = 1e-12
    assert np.abs(xo - (x + nsteps * dt * Cx)).max() < tol and np.abs(yo - (y + nsteps * dt * Cy)).max() < tol
    assert np.abs(ko - k).max() < tol and np.abs(lo - l).max() < tol
    assert np.abs(ao / a0 - (1 + z + z ** 2 / 2 + z ** 3 / 6 + z ** 4 / 24) ** nsteps).max() < tol


@pytest.mark.gpu
def test_ode23_in_lagrange_mode_is_bit_identical_to_the_restatement():
    """qgsw_raytrace.m:141-150 in LAGRANGE6 mode: interpolate_U (both frames, blended results), odefun and the
    Bogacki-Shampine stages (y + f*hB, the error estimate f*E) are all executed without fused multiply-adds in the
    restatement's order, so the whole adaptive solve -- every accept/reject decision and the final packets -- is the same
    doubles as oracle.ode23 on the restated odefun, not merely within 1e-9."""
    nx = 32; L = 2 * np.pi; h = L / nx
    _, p1 = make_flow(nx, seed=7); _, p2 = make_flow(nx, seed=8)
    names = ("u", "v", "ux", "uy", "vx", "vy")
    bf1 = {n: O.k2g(p) for n, p in zip(names, p1)}; bf2 = {n: O.k2g(p) for n, p in zip(names, p2)}
    n = 257
    x, y, k, l = make_packets(n, L)
    tmax = 0.05
    ode = O.generate_raytracing_ode(bf1, bf2, n, F0, 1.0, tmax, h)               # bump 1e-10, as the QG drivers run it
    yref, sref = O.ode23(ode, [0.0, tmax], np.concatenate([x, y, k, l]))
    with S.Engine(nx, L, F0, 1.0, S.MODE_LAGRANGE6, bump=O.BUMP_QG) as e:
        e.set_flow_grid(*[bf1[n_] for n_ in names], slot=0); e.set_flow_grid(*[bf2[n_] for n_ in names], slot=1)
        e.set_packets(x, y, k, l)
        st = R.ode23(e, [0.0, tmax], tmax)
        got = np.concatenate(e.get_packets())
    assert (st["nsteps"], st["nfailed"], st["nfevals"]) == (sref["nsteps"], sref["nfailed"], sref["nfevals"]) and st["nsteps"] >= 10
    assert _bit_equal(got, yref), _ulps(got, yref)
    # dense output (SW_zero_background_raytracing.m:73-78) through the same stages
    ts = tmax * np.linspace(0.0, 1.0, 7)
    Yref, _ = O.ode23(ode, ts, np.concatenate([x, y, k, l]))
    with S.Engine(nx, L, F0, 1.0, S.MODE_LAGRANGE6, bump=O.BUMP_QG) as e:
        e.set_flow_grid(*[bf1[n_] for n_ in names], slot=0); e.set_flow_grid(*[bf2[n_] for n_ in names], slot=1)
        e.set_packets(x, y, k, l)
        Y = R.ode23(e, ts, tmax)["Y"].reshape(len(ts), 4 * n)
    assert _bit_equal(Y, Yref), _ulps(Y, Yref)


@pytest.mark.gpu
def test_C2_C3_full_size_lagrange_mode_bit_identical_to_the_cpu_port():
    """The CPU arm of bench.py (--impl reference: oracle/swrt_oracle.c, -ffp-contract=off) and the LAGRANGE6 GPU arm execute
    the same IEEE operations: at BASELINE's full sizes every packet of the two runs is the same four doubles.
    C2: 65,536 packets x 48 steps on 128^2; C3 field (256^2): 1,048,576 packets x 8 steps."""
    for name, nsteps in (("C2", 48), ("C3", 8)):
        w = W.make_workload(name)
        kx_, ky_ = O.wavenumbers(w.nx)
        grids = [O.k2g(p) for p in O.velocity_planes_k(w.psik, kx_, ky_)]
        ref = CO.leapfrog_lagrange(w.x, w.y, w.k, w.l, grids, w.dx, w.f, w.gH, w.dt, nsteps)
        with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6) as e:
            e.set_flow_grid(*grids)
            e.set_packets(w.x, w.y, w.k, w.l)
            e.step(S.SCHEME_LEAPFROG, w.dt, nsteps)
            got = e.get_packets()
        for g_, r_, comp in zip(got, ref, "xykl"):
            assert _bit_equal(g_, r_), (name, comp, _ulps(g_, r_))


@pytest.mark.gpu
def test_randomised_sizes_all_modes_agree_with_their_checkers():
    """differential sweep over awkward sizes: grid sizes that are not powers of two (incl. nx/2 odd and the minimum nx = 8),
    domains L != 2*pi, ragged packet counts (quad / tile tails), positions far outside the domain; every mode against its
    checker, and NUFFT against SPECTRAL"""
    rs = np.random.RandomState(2024)
    for nx in (8, 10, 12, 14, 18, 22, 26, 34, 50, 66, 100):
        L = float(rs.choice([2 * np.pi, 20.0, 1.0, 7.3])); dx = L / nx
        kap = 2 * np.pi / L
        kx_, ky_ = O.wavenumbers(nx)
        psik = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx_ ** 2 + ky_ ** 2) * 0.1
        um = float(rs.choice([0.0, 0.5]))
        planes = O.velocity_planes_k(psik, kap * kx_, kap * ky_)
        planes[0] = planes[0].copy(); planes[0][nx // 2 - 1, 0] += um
        n = int(rs.randint(1, 300))
        x = rs.uniform(-50 * L, 50 * L, n); y = rs.uniform(-50 * L, 50 * L, n)
        k = rs.randn(n) * 3; l = rs.randn(n) * 3
        ref = CO.spectral_eval(x, y, planes, dx, nx, precise=True)
        grids = [O.k2g(p) for p in planes]
        dt = 0.05 * dx
        outs = {}
        for mode in (S.MODE_SPECTRAL, S.MODE_NUFFT, S.MODE_LAGRANGE6):
            with S.Engine(nx, L, F0, GH0, mode) as e:
                e.set_flow_spectral(psik, u_mean=um)
                ev = e.eval_at(x, y)
                if mode == S.MODE_LAGRANGE6:
                    # bit-identical to the restatement when the SAME grids are handed over (device grid_U uses cuFFT)
                    e.set_flow_grid(*grids)
                    ev = e.eval_at(x, y)
                    for c in range(6):
                        assert _bit_equal(ev[c], O.interpolate(x, y, grids[c], dx, dx)), (nx, n, c)
                else:
                    assert scaled_err(ev, ref) < TOL_FIELD, (nx, L, n, mode, scaled_err(ev, ref))
                e.set_packets(x, y, k, l)
                e.step(S.SCHEME_LEAPFROG, dt, 7)
                outs[mode] = np.stack(e.get_packets())
        assert np.abs(outs[S.MODE_NUFFT] - outs[S.MODE_SPECTRAL]).max() < TOL_TRAJ * max(1.0, 50 * L), (nx, n)
        assert np.isfinite(outs[S.MODE_LAGRANGE6]).all()


@pytest.mark.gpu
def test_randomised_schemes_two_frames_awkward_sizes():
    """second differential sweep: two flow frames with random alpha, RK4 steppers with and without H, ode23, at grid sizes
    that are not powers of two and ragged packet counts; NUFFT and SPECTRAL must agree (same series), LAGRANGE6 must match
    the restated RK4 batch stepper"""
    rs = np.random.RandomState(77)
    for nx in (8, 12, 18, 30, 44, 70):
        L = 2 * np.pi; dx = L / nx
        kx_, ky_ = O.wavenumbers(nx)
        amp = 0.05 / (1 + kx_ ** 2 + ky_ ** 2)
        psi1 = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) * amp
        psi2 = (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) * amp
        etak = 3.0 * psi1
        planes7 = W.planes_from_psik(psi1, L, 0.0, etak=etak)
        n = int(rs.randint(1, 200))
        x = rs.uniform(-5 * L, 5 * L, n); y = rs.uniform(-5 * L, 5 * L, n)
        k = rs.randn(n) * 5; l = rs.randn(n) * 5
        alpha = float(rs.uniform(0.05, 0.95)); dt = 0.1 * dx
        res = {}
        for mode in (S.MODE_SPECTRAL, S.MODE_NUFFT):
            with S.Engine(nx, L, F0, 1.0, mode) as e:
                e.set_flow_spectral(psi1, 0); e.set_flow_spectral(psi2, 1)
                e.set_packets(x, y, k, l)
                rhs = np.stack(e.rhs(alpha))
                e.step(S.SCHEME_LEAPFROG, dt, 3, alpha, 0.01)
                e.step(S.SCHEME_RK4_PACKET, dt, 2, alpha)
                st = R.ode23(e, [0.0, 5 * dt], 5 * dt)
                a_ = np.stack(e.get_packets())
                e.set_flow_planes_spectral(planes7, 0)
                e.set_packets(x, y, k, l, np.ones(n))
                e.step(S.SCHEME_RK4_XKA, dt, 2)
                res[mode] = (rhs, a_, (st["nsteps"], st["nfailed"]), np.stack(e.get_packets(with_a=True)))
        a, b = res[S.MODE_SPECTRAL], res[S.MODE_NUFFT]
        assert scaled_err(b[0], a[0]) < 5e-12, (nx, n)
        assert np.abs(b[1] - a[1]).max() < TOL_TRAJ * 50 and a[2] == b[2], (nx, n)
        assert np.abs(b[3] - a[3]).max() < TOL_TRAJ * 50, (nx, n)
        # LAGRANGE6 RK4 (with H) against the restated batch stepper on the same grids
        grids = [O.k2g(p) for p in planes7[:6]]; H = O.k2g(planes7[6])
        fields = {"u": grids[0], "v": grids[1], "u_x": grids[2], "u_y": grids[3], "v_x": grids[4], "v_y": grids[5], "H": H}
        with S.Engine(nx, L, F0, 1.0, S.MODE_LAGRANGE6) as e:
            e.set_flow_grid(*grids, H=H)
            e.set_packets(x, y, k, l, np.ones(n))
            e.step(S.SCHEME_RK4_XKA, dt, 2)
            got = np.stack(e.get_packets(with_a=True))
        st_ = (x, y, k, l, np.ones(n))
        for _ in range(2):
            st_ = O.rk4_step_batch(*st_, dt, 1.0, F0, fields, dx, True)
        assert np.abs(got - np.stack(st_)).max() < TOL_TRAJ, (nx, n)


@pytest.mark.gpu
def test_bench_gpu_arm_prints_one_contract_line():
    """python bench.py (the GPU arm, N = 1) on small ensembles: exactly one JSON line on stdout carrying the contract's
    keys -- value / e2e with host<->device bytes (pinned and pageable), gpu_launches > 0, roofline of the dominant kernel
    (tensor bound against the fp64 peak measured in the run, fraction in (0, 1]), cpu_baseline measured beside it, sampled
    clocks -- a side config under "configs" and the side legs of the other two modes (gather bound, "l2")"""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SWRT_BENCH_TARGET_S="0.3")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "3", "--warmup", "3", "--packets", "9472",
                          "--configs", "C2", "--side-steps", "3"],
                         capture_output=True, text=True, env=env, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "configs", "peaks_measured"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["dtype"] == "f64" and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert d["config"]["name"] == "C4" and d["config"]["nx"] == 512 and d["config"]["packets_total"] == 9472
    assert d["arm"]["mode"] == "SPECTRAL" and d["arm"]["packets_per_gpu"] == 9472
    assert d["value"] > 0 and d["gpu_launches"] >= 3 * 3
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 4 * 8 * 9472 == d["e2e"]["d2h_bytes_per_step"]
    assert d["e2e"]["pageable"]["value"] > 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and 0.0 < r["frac"] <= 1.0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    assert r["kernel_launches_per_step"] == 1                   # the two sub-steps of the two-frame flow run in ONE packet kernel
    assert 25.0 < d["peaks_measured"]["fp64_matmul_tflops"] < 45.0 and r["peak"] == d["peaks_measured"]["fp64_matmul_tflops"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0 and d["cpu_baseline"]["cores"] >= 1
    assert d["clocks"]["sm_max_mhz"] > 0
    c2 = d["configs"]["C2"]
    assert c2["value"] > 0 and c2["e2e"]["value"] > 0 and c2["roofline"]["bound"] == "tensor" and c2["config"]["packets_total"] == 65536
    for m in ("lagrange6", "nufft"):
        assert d[m]["value"] > 0 and d[m]["roofline"]["bound"] == "l2" and d[m]["roofline"]["peak"] == d["peaks_measured"]["gather_probe_gbs"] > 0
    assert d["histogram_total"] <= 9472


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: the packets and omega histogram after warm-up + --steps bench steps, equal to the same
    steps driven through the Engine directly; the same arguments give the same files, one more step gives other ones"""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    n, warmup = 9472, 3

    def bench(steps, tag):
        out = tmp_path / tag
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                            "--packets", str(n), "--configs", "", "--no-side-modes", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, env=env, timeout=900, cwd=root)
        assert r.returncode == 0, r.stderr[-3000:]
        files = sorted(out.glob("*.npy"))
        assert [f.stem for f in files] == ["k", "l", "omega_hist", "x", "y"]
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        return {f.stem: np.load(f) for f in files}

    w = W.make_workload("C4", n_packets=n)
    edges = np.linspace(0.0, float(np.sqrt(w.f ** 2 + w.gH * 4 * (w.k ** 2 + w.l ** 2).max())), 300)
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL) as e:
        e.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
        e.set_packets(w.x, w.y, w.k, w.l)
        want = {}
        for total in range(1, warmup + 3):
            e.step(S.SCHEME_LEAPFROG, w.dt / 2, 2, 0.25, 0.5)            # one C4 bench step: two time-centred sub-steps
            if total - warmup in (1, 2):
                want[total - warmup] = dict(zip("xykl", e.get_packets()), omega_hist=e.hist_omega(edges).astype(np.float64))
    one, again, two = bench(1, "one"), bench(1, "again"), bench(2, "two")
    for name in one:
        assert one[name].dtype == np.float64 and np.array_equal(one[name], again[name]), name
        assert np.array_equal(one[name], want[1][name]) and np.array_equal(two[name], want[2][name]), name
    assert not np.array_equal(one["x"], two["x"]) and one["omega_hist"].sum() == n


def test_nufft_gradients_at_and_next_to_grid_nodes():
    """A packet on a grid node (or within rounding of one: x = i*dx) puts a stencil node at the very end of the NUFFT kernel's
    support, where the analytic derivative phi' = -phi beta z / sqrt(1 - z^2) is singular; before the end node was dropped
    (nufft_kernels.cu:es_kernel) such packets got a spurious 2e-10 of the gradient.  All six planes within 1e-12 of the exact
    sum on nodes, one ulp either side, and at offsets down to 1e-12 of a cell, in SPECTRAL and NUFFT modes."""
    nx = 32; L = 2 * np.pi; dx = L / nx
    psik, planes = make_flow(nx, seed=11)
    ii = np.arange(nx * 3) % nx; jj = (np.arange(nx * 3) * 5 + 3) % nx
    xs, ys = [], []
    for off in (0.0, 1e-12, -1e-12, 1e-9, -1e-9, 3e-7, -3e-7, 1e-4):
        xs.append((ii + off) * dx); ys.append((jj - off) * dx)
        xs.append((ii * 0.5 + off) * dx); ys.append((jj * 0.5 + 0.25 - off) * dx)          # fine-grid nodes between coarse ones
    xs.append(np.nextafter(ii * dx, np.inf)); ys.append(np.nextafter(jj * dx, -np.inf))
    xs.append(np.nextafter(ii * dx, -np.inf)); ys.append(np.nextafter(jj * dx, np.inf))
    x = np.concatenate(xs); y = np.concatenate(ys)
    ref = CO.spectral_eval(x, y, planes, dx, nx)
    for mode in (S.MODE_SPECTRAL, S.MODE_NUFFT):
        with S.Engine(nx, L, F0, GH0, mode) as e:
            e.set_flow_planes_spectral(planes)
            assert scaled_err(e.eval_at(x, y), ref) < TOL_FIELD, mode
