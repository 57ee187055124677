"""ode23 backward in time on the device: a decreasing tspan (MATLAB's ``ode23(odefun, [T 0], y0)``) in swrt_ode23
(Engine.ode23), swrt_ode23_packets (Engine.ode23_packets), the host controller on the device building blocks
(reference_api.ode23), the MEX gateway and the swrt_ode23.m shim.

The exact check is the mirror identity: in a steady flow, the backward solve of (x, k) over [T .. 0] with the flow psi and
the forward solve of (x, -k) over [-T .. 0] with the flow -psi perform the same floating-point operations up to sign
(t - absh = -(-t + absh); every evaluation path is linear in psi; the RHS is odd in (U, k) for x and even for k; |.|,
eps(|t|) and the error norm are unchanged), so they agree bit for bit with k and l negated."""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from swraytracing_b200 import workloads as W
from test_ode23_device import Recorder
from test_ode23_packets import (F0, GH0, L, MODES, assert_equals_one_packet_solves, make_packets, make_psik,
                                one_packet_solves, scale_of)

pytestmark = pytest.mark.gpu

T = 0.4
TOLS = [(1e-3, 1e-6), (1e-6, 1e-7)]
NEG = np.array([1.0, 1.0, -1.0, -1.0])


def engine(mode, nx, two, sign=1.0, amp=0.3, ngpu=1):
    e = S.Engine(nx, L, F0, GH0, mode, ngpu=ngpu)
    e.set_flow_spectral(sign * make_psik(nx, 7, amp), slot=0)
    if two:
        e.set_flow_spectral(sign * make_psik(nx, 8, amp), slot=1)
    return e


def solve(kind, e, pk, tspan, tmax, rtol, atol):
    """one solve of `kind` from packets pk: (stats, final packets, launches); stats["h"] holds the signed accepted steps
    where the solve reports them"""
    e.set_packets(*pk)
    e.launch_count(reset=True)
    if kind == "device":
        st = e.ode23(tspan, tmax, rtol, atol, trace=100000)
    elif kind == "packets":
        st = e.ode23_packets(tspan, tmax, rtol, atol)
    else:
        rec = Recorder(e)
        st = R.ode23(rec, tspan, tmax, rtol, atol)
        st["h"] = np.array(rec.h)
    return st, np.stack(e.get_packets()), e.launch_count()


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("kind", ["device", "packets", "host"])
@pytest.mark.parametrize("tol", TOLS)
def test_mirror_identity(mode, nx, kind, tol):
    pk = make_packets(200)
    ts = np.linspace(T, 0.0, 11)
    with engine(mode, nx, False) as e, engine(mode, nx, False, sign=-1.0) as em:
        b, yb, nb = solve(kind, e, pk, ts, None, *tol)
        f, yf, nf = solve(kind, em, pk * NEG[:, None], -ts, None, *tol)
    assert (b["nsteps"], b["nfailed"], b["nfevals"]) == (f["nsteps"], f["nfailed"], f["nfevals"]) and nb == nf
    assert b.get("host_waits") == f.get("host_waits")
    if kind == "packets":
        assert b["steps"].min() >= 10
        for key in ("steps", "rejected", "status"):
            assert np.array_equal(b[key], f[key]), key
        assert np.all(b["t_end"] == 0.0) and np.all(f["t_end"] == 0.0)
    else:
        assert b["nsteps"] >= 10 and np.all(b["h"] < 0) and np.array_equal(b["h"], -f["h"])
    assert np.array_equal(yb, yf * NEG[:, None])
    assert np.array_equal(b["Y"], f["Y"] * NEG[None, :, None]) and np.array_equal(b["Y"][0], pk)


def assert_same_backward_solve(sh, ph, sd, pd, exact_if_same_steps):
    """swrt_ode23 made the host controller's decisions (tests/test_ode23_device.py's bounds, for a solve from T to 0)"""
    assert (sd["nsteps"], sd["nfailed"], sd["nfevals"]) == (sh["nsteps"], sh["nfailed"], sh["nfevals"])
    assert sh["t"] == 0.0 and sd["t"] == 0.0
    hh, hd = sh["h"], sd["h"]
    assert hd.shape == hh.shape and np.all(hd < 0)
    # the device power is correctly rounded; glibc's pow (the host controller's) is off by one ulp on rare arguments
    assert np.all(np.abs(hd - hh) <= 2 * np.spacing(np.abs(hh)))
    assert abs(hd.sum() + T) < 1e-12
    assert np.all(np.abs(pd - ph) <= 1e-12 * scale_of(ph))
    if exact_if_same_steps and np.array_equal(hd, hh):
        assert np.array_equal(pd, ph)


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("tol", TOLS)
def test_two_frames_device_equals_host_controller(mode, nx, tol):
    # alpha = t/tmax runs from 1 to 0
    pk = make_packets(300)
    with engine(mode, nx, True) as e:
        sh, ph, _ = solve("host", e, pk, [T, 0.0], T, *tol)
        sd, pd, _ = solve("device", e, pk, [T, 0.0], T, *tol)
    assert sh["nsteps"] >= 10
    assert_same_backward_solve(sh, ph, sd, pd, mode == S.MODE_LAGRANGE6)


@pytest.mark.parametrize("mode,nx", MODES)
def test_two_frames_rejections_match(mode, nx):
    pk = make_packets(200, seed=9)
    for amp in (3.0, 10.0, 30.0):
        with engine(mode, nx, True, amp=amp) as e:
            sh, ph, _ = solve("host", e, pk, [0.2, 0.0], 0.2, 1e-3, 1e-6)
            sd, pd, _ = solve("device", e, pk, [0.2, 0.0], 0.2, 1e-3, 1e-6)
        if sh["nfailed"] > 0:
            break
    assert sh["nfailed"] > 0 and sh["nsteps"] <= 400
    assert (sd["nsteps"], sd["nfailed"], sd["nfevals"]) == (sh["nsteps"], sh["nfailed"], sh["nfevals"])
    assert np.all(np.abs(sd["h"] - sh["h"]) <= 2 * np.spacing(np.abs(sh["h"]))) and abs(sd["h"].sum() + 0.2) < 1e-12
    assert np.all(np.abs(pd - ph) <= 1e-12 * scale_of(ph))
    if mode == S.MODE_LAGRANGE6 and np.array_equal(sd["h"], sh["h"]):
        assert np.array_equal(pd, ph)


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("tol", TOLS)
def test_two_frames_packets_equal_one_packet_solves(mode, nx, tol):
    pk = make_packets(40)
    ts = np.linspace(T, 0.0, 6)
    with engine(mode, nx, True) as e:
        st, yp, _ = solve("packets", e, pk, ts, T, *tol)
        ref = one_packet_solves(e, pk, ts, T, *tol)
    assert st["steps"].min() >= 10
    # SPECTRAL between two frames evaluates both frames and blends the planes; swrt_ode23 blends the coefficient stacks
    assert_equals_one_packet_solves(st, yp, ref, not (mode == S.MODE_SPECTRAL), scale_of(yp))


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("kind", ["device", "packets"])
def test_round_trip_returns_the_initial_packets(mode, nx, kind):
    """forward 0 -> T, then backward T -> 0.  Each accepted step keeps its local error estimate below
    rtol * max(|y|, atol/rtol) per component; over a short solve in a weak flow the errors of both legs add up without
    much growth, so the packets come back within 10 * rtol * (steps of both legs) * their scale -- while a leg that did not
    run backward would miss by the whole displacement"""
    rtol, atol = 1e-6, 1e-7
    pk = make_packets(200)
    with engine(mode, nx, True) as e:
        a, ya, _ = solve(kind, e, pk, [0.0, T], T, rtol, atol)
        b, yb, _ = solve(kind, e, ya, [T, 0.0], T, rtol, atol)
    steps = (a["steps"] + b["steps"]) if kind == "packets" else a["nsteps"] + b["nsteps"]
    bound = 10 * rtol * np.asarray(steps) * np.maximum(scale_of(pk), atol / rtol)
    assert np.all(np.abs(yb - pk) <= bound)
    assert np.abs(ya - pk).max() > 10 * bound.max()              # the flow moved the packets


@pytest.mark.parametrize("mode,nx", MODES)
def test_packets_backward_ensemble_independence(mode, nx):
    pk = make_packets(300, seed=11)
    rs = np.random.RandomState(2)
    sub = np.sort(rs.choice(pk.shape[1], 37, replace=False))
    perm = rs.permutation(pk.shape[1])
    ts = np.linspace(T, 0.0, 11)
    with engine(mode, nx, True) as e:
        a, ya, _ = solve("packets", e, pk, ts, T, 1e-6, 1e-7)
        b, yb, _ = solve("packets", e, pk[:, sub], ts, T, 1e-6, 1e-7)
        c, yc, _ = solve("packets", e, pk[:, perm], ts, T, 1e-6, 1e-7)
    assert np.array_equal(yb, ya[:, sub]) and np.array_equal(b["Y"], a["Y"][:, :, sub])
    assert np.array_equal(b["steps"], a["steps"][sub]) and np.array_equal(b["rejected"], a["rejected"][sub])
    assert np.array_equal(yc, ya[:, perm]) and np.array_equal(c["Y"], a["Y"][:, :, perm])
    assert np.array_equal(c["steps"], a["steps"][perm]) and np.array_equal(c["t_end"], a["t_end"][perm])


@pytest.mark.parametrize("mode,nx", MODES)
def test_packets_backward_blown_up_packet_stops_alone(mode, nx):
    pk = make_packets(100)
    pk[2, 17] = np.inf
    good = np.delete(np.arange(100), 17)
    ts = np.linspace(T, 0.0, 6)
    with engine(mode, nx, True) as e:
        st, yp, _ = solve("packets", e, pk, ts, T, 1e-3, 1e-6)
        s2, y2, _ = solve("packets", e, pk[:, good], ts, T, 1e-3, 1e-6)
    assert st["stopped"] == 1 and st["status"][17] == 1 and st["status"].sum() == 1
    assert 0.0 < st["t_end"][17] <= T and np.all(st["t_end"][good] == 0.0)
    assert np.all(np.isnan(st["Y"][1:, :, 17])) and np.isfinite(st["Y"][:, :, good]).all()
    assert np.array_equal(yp[:, good], y2) and np.array_equal(st["Y"][:, :, good], s2["Y"])
    assert np.array_equal(st["steps"][good], s2["steps"]) and np.array_equal(st["rejected"][good], s2["rejected"])


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("kind", ["device", "packets"])
def test_two_devices_equal_one_bit_for_bit(mode, nx, kind):
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two GPUs")
    pk = make_packets(3001, seed=12)
    ts = np.linspace(T, 0.0, 11)
    res = []
    for ngpu in (1, 2):
        with engine(mode, nx, True, ngpu=ngpu) as e:
            res.append(solve(kind, e, pk, ts, T, 1e-6, 1e-7))
    (a, ya, _), (b, yb, _) = res
    assert (a["nsteps"], a["nfailed"], a["nfevals"]) == (b["nsteps"], b["nfailed"], b["nfevals"])
    assert np.array_equal(ya, yb) and np.array_equal(a["Y"], b["Y"], equal_nan=True)
    for key in ("h",) if kind == "device" else ("steps", "rejected", "status", "t_end"):
        assert np.array_equal(a[key], b[key]), key


@pytest.mark.parametrize("tspan", [[0.0, 0.2, 0.1, T], [T, 0.1, 0.2, 0.0], [0.2, T, 0.0]])
def test_tspan_against_its_direction_is_refused_and_the_handle_survives(tspan):
    import ctypes as C
    lib = S.load_library()
    pk = make_packets(50)
    ts = np.asarray(tspan, dtype=np.float64)
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        ref_d, yref_d, _ = solve("device", e, pk, [T, 0.0], T, 1e-3, 1e-6)
        ref_p, yref_p, _ = solve("packets", e, pk, [T, 0.0], T, 1e-3, 1e-6)
        e.set_packets(*pk)
        st = (C.c_int64 * 5)()
        pts = ts.ctypes.data_as(C.POINTER(C.c_double))
        assert lib.swrt_ode23(e._h, pts, ts.size, T, 1e-3, 1e-6, None, st, None, 0) == -1        # SWRT_ERR_ARG
        assert lib.swrt_ode23_packets(e._h, pts, ts.size, T, 1e-3, 1e-6, None, None, None, st) == -1
        assert np.array_equal(np.stack(e.get_packets()), pk)
        with pytest.raises(S.SwrtError, match="monotonic"):
            e.ode23(ts, T)
        with pytest.raises(ValueError, match="monotonic"):
            R.ode23(e, ts, T)
        got_d, y_d, _ = solve("device", e, pk, [T, 0.0], T, 1e-3, 1e-6)
        got_p, y_p, _ = solve("packets", e, pk, [T, 0.0], T, 1e-3, 1e-6)
    assert np.array_equal(y_d, yref_d) and np.array_equal(got_d["h"], ref_d["h"])
    assert np.array_equal(y_p, yref_p) and np.array_equal(got_p["steps"], ref_p["steps"])


# ---- the MEX gateway and the MATLAB shim -----------------------------------------------------------------------------
@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    from test_mex_gateway import Mex
    return Mex(request.param)


def _gateway_setup(mex, n, blow_up=False):
    w = W.make_workload("C3", n_packets=n, nx=32)
    k = w.k.copy()
    if blow_up:
        k[3] = np.inf
    h = mex("create", float(w.nx), w.L, w.f, w.gH, float(S.MODE_LAGRANGE6))
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6)
    for slot, psik in ((0.0, w.psik), (1.0, w.psik2)):
        mex("set_flow_spectral", h, slot, psik, nlhs=0)
        eng.set_flow_spectral(psik, int(slot))
    mex("set_packets", h, w.x, w.y, k, w.l, nlhs=0)
    eng.set_packets(w.x, w.y, k, w.l)
    return w, h, eng


def test_gateway_ode23_backward(mex):
    w, h, eng = _gateway_setup(mex, 301)
    tspan = w.dt * np.linspace(1.0, 0.0, 6)
    st, Y = mex("ode23", h, tspan, w.dt, 1e-6, 1e-7, nlhs=2)
    ref = eng.ode23(tspan, w.dt, 1e-6, 1e-7)
    assert np.array_equal(np.ravel(st)[:3], [ref["nsteps"], ref["nfailed"], ref["nfevals"]]) and ref["nsteps"] >= 10
    assert np.array_equal(Y.reshape(301, 4, tspan.size, order="F"), ref["Y"].transpose(2, 1, 0))
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()))
    mex("destroy", h, nlhs=0); eng.close()


def test_gateway_ode23_packets_backward(mex):
    w, h, eng = _gateway_setup(mex, 301, blow_up=True)
    tspan = w.dt * np.linspace(1.0, 0.0, 6)
    st, Y, pstat, t_end = mex("ode23_packets", h, tspan, w.dt, 1e-6, 1e-7, nlhs=4)
    ref = eng.ode23_packets(tspan, w.dt, 1e-6, 1e-7)
    assert np.array_equal(np.ravel(st)[:4], [ref["nsteps"], ref["nfailed"], ref["nfevals"], ref["stopped"]]) and ref["stopped"] == 1
    assert np.array_equal(pstat, np.stack([ref["steps"], ref["rejected"], ref["status"]], axis=1))
    assert np.array_equal(t_end, ref["t_end"])
    assert np.array_equal(Y.reshape(301, 4, tspan.size, order="F"), ref["Y"].transpose(2, 1, 0), equal_nan=True)
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()), equal_nan=True)
    mex("destroy", h, nlhs=0); eng.close()


def test_ode23_shim_backward_makes_the_host_controllers_decisions():
    """matlab/shims/swrt_ode23.m run by minimat with [tmax 0] through the gateway: the Python host controller's decisions
    over the same device stages, and the same packets"""
    from test_shims_executed import NAMES, Mex as ShimMex, interp, read_in, workspace
    mex = ShimMex(False)
    I = interp(mex)
    fr, nx, n = workspace()
    I.run(r"""
        eng = swrt_mex('create', nx, L, f, 1, 1, 0, 1e-10);
        swrt_mex('set_flow_grid', eng, 0, bf1.u, bf1.v, bf1.ux, bf1.uy, bf1.vx, bf1.vy);
        swrt_mex('set_flow_grid', eng, 1, bf2.u, bf2.v, bf2.ux, bf2.uy, bf2.vx, bf2.vy);
        swrt_mex('set_packets', eng, x, y, k, l);
        tmax = 0.4;
        stats = swrt_ode23(eng, [tmax 0], tmax);
        [px, py, pk, pl] = swrt_mex('get_packets', eng);
        swrt_mex('destroy', eng);
    """, fr)
    v = fr.vars
    bf1 = {nm: read_in(f"bf1_{nm}", nx, nx) for nm in NAMES}; bf2 = {nm: read_in(f"bf2_{nm}", nx, nx) for nm in NAMES}
    x, y, k, l = (read_in(c, n) for c in "xykl")
    with S.Engine(nx, float(v["L"]), float(v["f"]), 1.0, S.MODE_LAGRANGE6, bump=1e-10) as e:
        e.set_flow_grid(*[bf1[nm] for nm in NAMES], slot=0); e.set_flow_grid(*[bf2[nm] for nm in NAMES], slot=1)
        e.set_packets(x, y, k, l)
        st = R.ode23(e, [0.4, 0.0], 0.4)
        want = e.get_packets()
    assert (v["stats"].f["nsteps"], v["stats"].f["nfailed"]) == (float(st["nsteps"]), float(st["nfailed"])) and st["nsteps"] >= 5
    assert float(v["stats"].f["t"]) == 0.0
    for got, ref in zip((v["px"], v["py"], v["pk"], v["pl"]), want):
        assert np.array_equal(np.asarray(got).ravel(), ref)
