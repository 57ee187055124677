"""swrt_ode23_packets / Engine.ode23_packets: ode23 with an independent step-size controller per packet.  The oracle is
the definition: packet i of an ensemble solved per packet equals swrt_ode23 (Engine.ode23) run on a handle that holds
packet i alone."""
import re

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from oracle import swrt_oracle as O

pytestmark = pytest.mark.gpu

L = 2 * np.pi
F0, GH0 = 3.0, 1.0
MODES = [(S.MODE_SPECTRAL, 32), (S.MODE_SPECTRAL, 64), (S.MODE_LAGRANGE6, 32), (S.MODE_NUFFT, 32)]
THREE = [(S.MODE_SPECTRAL, 32), (S.MODE_LAGRANGE6, 32), (S.MODE_NUFFT, 32)]


def make_psik(nx, seed, amp=0.3):
    rs = np.random.RandomState(seed)
    kx_, ky_ = O.wavenumbers(nx)
    return (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx_ ** 2 + ky_ ** 2) ** 1.5 * amp


def make_packets(n, seed=5):
    rs = np.random.RandomState(seed)
    i = np.arange(n)
    return np.stack([rs.uniform(-L, L, n), rs.uniform(-L, L, n), 3 * np.cos(0.37 * i), 3 * np.sin(0.37 * i)])


def engine(mode, nx, two, ngpu=1, amp=0.3):
    e = S.Engine(nx, L, F0, GH0, mode, ngpu=ngpu)
    e.set_flow_spectral(make_psik(nx, 7, amp), slot=0)
    if two:
        e.set_flow_spectral(make_psik(nx, 8, amp), slot=1)
    return e


def per_packet(e, pk, tspan, tmax, rtol=1e-3, atol=1e-6):
    e.set_packets(*pk)
    st = e.ode23_packets(tspan, tmax, rtol, atol)
    return st, np.stack(e.get_packets())


def one_packet_solves(e, pk, tspan, tmax, rtol=1e-3, atol=1e-6):
    """swrt_ode23 on a handle holding packet i alone, for every i: (steps, rejected, final state, Y or None, t of failure)"""
    out = []
    for i in range(pk.shape[1]):
        e.set_packets(*pk[:, i:i + 1])
        try:
            st = e.ode23(tspan, tmax, rtol, atol)
            out.append((st["nsteps"], st["nfailed"], np.stack(e.get_packets())[:, 0], st.get("Y"), None))
        except S.SwrtError as ex:
            t = float(re.search(r"at t = (\S+)", str(ex)).group(1))
            out.append((None, None, np.stack(e.get_packets())[:, 0], None, t))
    return out


def assert_equals_one_packet_solves(st, yp, ref, exact, pk_scale):
    assert np.array_equal(st["steps"], [r[0] for r in ref])
    assert np.array_equal(st["rejected"], [r[1] for r in ref])
    assert st["nsteps"] == st["steps"].sum() and st["nfailed"] == st["rejected"].sum()
    assert st["nfevals"] == yp.shape[1] + 3 * (st["nsteps"] + st["nfailed"]) and st["stopped"] == 0
    assert np.all(st["status"] == 0) and np.all(st["t_end"] == st["t"])
    y1 = np.stack([r[2] for r in ref], axis=1)
    Y1 = np.stack([r[3][:, :, 0] for r in ref], axis=2) if "Y" in st else None
    if exact:
        assert np.array_equal(yp, y1)
        if Y1 is not None:
            assert np.array_equal(st["Y"], Y1)
    else:
        assert np.all(np.abs(yp - y1) <= 1e-12 * pk_scale)
        if Y1 is not None:
            assert np.all(np.abs(st["Y"] - Y1) <= 1e-12 * pk_scale[None])


def scale_of(y):
    return np.abs(y).max(axis=1, keepdims=True)


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("two", [False, True])
@pytest.mark.parametrize("tol", [(1e-3, 1e-6), (1e-6, 1e-7)])
def test_equals_one_packet_solves(mode, nx, two, tol):
    tmax = 0.4
    pk = make_packets(40)
    with engine(mode, nx, two) as e:
        st, yp = per_packet(e, pk, [0.0, tmax], tmax if two else None, *tol)
        ref = one_packet_solves(e, pk, [0.0, tmax], tmax if two else None, *tol)
    assert st["steps"].min() >= 10                    # MaxStep = 0.1*(tf - t0)
    # SPECTRAL between two frames evaluates both frames and blends the planes; swrt_ode23 blends the coefficient stacks
    exact = not (mode == S.MODE_SPECTRAL and two)
    assert_equals_one_packet_solves(st, yp, ref, exact, scale_of(yp))


@pytest.mark.parametrize("mode,nx", MODES)
def test_forced_rejections(mode, nx):
    pk = make_packets(40, seed=9)
    for amp in (3.0, 10.0, 30.0):
        with engine(mode, nx, True, amp=amp) as e:
            st, yp = per_packet(e, pk, [0.0, 0.2], 0.2)
            ref = one_packet_solves(e, pk, [0.0, 0.2], 0.2)
        if st["rejected"].max() > 0:
            break
    assert st["rejected"].max() > 0 and st["steps"].max() <= 400
    assert_equals_one_packet_solves(st, yp, ref, mode != S.MODE_SPECTRAL, scale_of(yp))


@pytest.mark.parametrize("mode", [S.MODE_SPECTRAL, S.MODE_LAGRANGE6, S.MODE_NUFFT])
def test_dense_output_c1_shape(mode):
    # SW_zero_background_raytracing.m:70-78: RelTol 1e-6, AbsTol 1e-7, output at dt*(0:N)
    dt, N = 0.05, 40
    tspan = dt * np.arange(N + 1)
    pk = make_packets(40, seed=3)
    with engine(mode, 32, False) as e:
        st, yp = per_packet(e, pk, tspan, None, 1e-6, 1e-7)
        ref = one_packet_solves(e, pk, tspan, None, 1e-6, 1e-7)
    assert st["Y"].shape == (N + 1, 4, 40)
    assert np.array_equal(st["Y"][0], pk) and np.array_equal(st["Y"][-1], yp)
    assert_equals_one_packet_solves(st, yp, ref, True, scale_of(yp))


@pytest.mark.parametrize("mode,nx", THREE)
def test_ensemble_independence(mode, nx):
    pk = make_packets(300, seed=11)
    rs = np.random.RandomState(2)
    sub = np.sort(rs.choice(pk.shape[1], 37, replace=False))
    perm = rs.permutation(pk.shape[1])
    tspan = 0.04 * np.arange(11)
    with engine(mode, nx, True) as e:
        a, ya = per_packet(e, pk, tspan, 0.4, 1e-6, 1e-7)
        b, yb = per_packet(e, pk[:, sub], tspan, 0.4, 1e-6, 1e-7)
        c, yc = per_packet(e, pk[:, perm], tspan, 0.4, 1e-6, 1e-7)
    assert np.array_equal(yb, ya[:, sub]) and np.array_equal(b["Y"], a["Y"][:, :, sub])
    assert np.array_equal(b["steps"], a["steps"][sub]) and np.array_equal(b["rejected"], a["rejected"][sub])
    assert np.array_equal(yc, ya[:, perm]) and np.array_equal(c["Y"], a["Y"][:, :, perm])
    assert np.array_equal(c["steps"], a["steps"][perm]) and np.array_equal(c["t_end"], a["t_end"][perm])
    assert (c["nsteps"], c["nfailed"], c["nfevals"]) == (a["nsteps"], a["nfailed"], a["nfevals"])


@pytest.mark.parametrize("mode,nx", THREE)
def test_two_devices_equal_one_bit_for_bit(mode, nx):
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two GPUs")
    pk = make_packets(3001, seed=12)
    tspan = 0.04 * np.arange(11)
    res = []
    for ngpu in (1, 2):
        with engine(mode, nx, True, ngpu=ngpu) as e:
            res.append(per_packet(e, pk, tspan, 0.4, 1e-6, 1e-7))
    (a, ya), (b, yb) = res
    assert np.array_equal(ya, yb) and np.array_equal(a["Y"], b["Y"])
    for key in ("steps", "rejected", "status", "t_end"):
        assert np.array_equal(a[key], b[key]), key
    assert (a["nsteps"], a["nfailed"], a["nfevals"]) == (b["nsteps"], b["nfailed"], b["nfevals"])


@pytest.mark.parametrize("mode,nx", THREE)
@pytest.mark.parametrize("bad", [np.inf, np.nan])
def test_blown_up_packet_stops_alone(mode, nx, bad):
    pk = make_packets(100)
    pk[2, 17] = bad
    good = np.delete(np.arange(100), 17)
    with engine(mode, nx, True) as e:
        st, yp = per_packet(e, pk, [0.0, 0.4], 0.4)
        assert st["stopped"] == 1 and st["status"][17] == 1 and st["status"].sum() == 1
        assert np.array_equal(yp[:, 17], pk[:, 17], equal_nan=True)          # its initial state
        (_, _, _, _, t_fail), = one_packet_solves(e, pk[:, 17:18], [0.0, 0.4], 0.4)
        assert t_fail is not None and st["t_end"][17] == t_fail
        s2, y2 = per_packet(e, pk[:, good], [0.0, 0.4], 0.4)
        assert np.array_equal(yp[:, good], y2) and np.array_equal(st["steps"][good], s2["steps"])
        assert np.array_equal(st["rejected"][good], s2["rejected"]) and np.all(st["t_end"][good] == 0.4)
        # the same handle then solves a finite ensemble as a fresh one does
        fin = make_packets(100, seed=8)
        s3, y3 = per_packet(e, fin, [0.0, 0.4], 0.4)
    with engine(mode, nx, True) as e:
        s4, y4 = per_packet(e, fin, [0.0, 0.4], 0.4)
    assert s3["stopped"] == 0 and np.array_equal(y3, y4) and np.array_equal(s3["steps"], s4["steps"])


def test_few_host_waits_and_launches_per_round():
    # the reference's unit of work at 50 packets: one solve over a QG step [0, dt] between two frames (C3 flow, 256^2).
    # LAGRANGE6 round: 3 x (stage, evaluation, RHS) + decide
    from swraytracing_b200 import workloads as W
    w = W.make_workload("C3", n_packets=50)
    per_round, begin = 10, 3                          # begin: evaluation, RHS, per-packet initial step
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6) as e:
        e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
        e.set_packets(w.x, w.y, w.k, w.l)
        e.launch_count(reset=True)
        st = e.ode23_packets([0.0, w.dt], w.dt)
        launches = e.launch_count()
    assert st["host_waits"] <= 3 and st["stopped"] == 0
    rounds, rest = divmod(launches - begin, per_round)
    assert rest == 0 and rounds >= (st["steps"] + st["rejected"]).max()


def test_reference_api_per_packet():
    pk = make_packets(20)
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        e.set_packets(*pk)
        a = R.ode23(e, [0.0, 0.4], 0.4, per_packet=True)
        ya = np.stack(e.get_packets())
        b, yb = per_packet(e, pk, [0.0, 0.4], 0.4)
        with pytest.raises(ValueError):
            R.ode23(e, [0.0, 0.4], 0.4, reduce_max=lambda v: v, per_packet=True)
    assert np.array_equal(ya, yb) and np.array_equal(a["steps"], b["steps"])


def test_qgsw_driver_one_packet_equals_coupled_solve(tmp_path):
    from swraytracing_b200 import drivers, fieldio
    nx, nif, U_g, f, Cg = 64, 2.0, 0.5, 3.0, 1.0
    out = {}
    for integ in ("ode23_device", "ode23_packets"):
        out[integ] = drivers.qgsw_raytrace(nx, 1, nif, 6000, 0, U_g, f, Cg, outdir=str(tmp_path / integ), max_steps=6,
                                           r_drag=0.01, integrator=integ, mode=S.MODE_LAGRANGE6, log=lambda s: None)
    a, b = out["ode23_device"], out["ode23_packets"]
    assert (a["ode23_steps"], a["ode23_failed"]) == (b["ode23_steps"], b["ode23_failed"]) and b["ode23_stopped_packets"] == 0
    assert np.array_equal(np.stack(a["packets"]), np.stack(b["packets"]))
    fa = fieldio.load_packet_frames(tmp_path / "ode23_device", 1)
    fb = fieldio.load_packet_frames(tmp_path / "ode23_packets", 1)
    assert all(np.array_equal(u, v) for u, v in zip(fa, fb))


def test_qgsw_driver_many_packets(tmp_path):
    from swraytracing_b200 import drivers, fieldio
    r = drivers.qgsw_raytrace(64, 20, 2.0, 6000, 0, 0.5, 3.0, 1.0, outdir=str(tmp_path), max_steps=6, r_drag=0.01,
                              integrator="ode23_packets", log=lambda s: None)
    assert r["ode23_steps"] >= 20 * 6 and r["ode23_stopped_packets"] == 0
    t, x, k = fieldio.load_packet_frames(tmp_path, 20)
    assert t.size >= 1 and np.all(np.isfinite(x)) and np.all(np.isfinite(k))


def test_sw_zero_background_driver():
    from swraytracing_b200 import drivers
    nx = 32
    got = drivers.SW_zero_background_raytracing(np.zeros((nx, nx)), nx=nx, f=3.0, Cg=2.0, Nparticles=100, Tend=0.5,
                                                integrator="ode23_packets")
    n = got["solver_x"].shape[2]
    assert got["solver_x"].shape == (got["Nsteps"] + 1, 2, n) and got["solver_k"].shape == got["solver_x"].shape
    assert got["stats"]["steps"].shape == (n,)
    assert got["stats"]["stopped"] == 0 and np.abs(got["solver_k"] - got["solver_k"][0]).max() == 0.0
