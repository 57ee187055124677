"""swrt_ode23_packets_events / Engine.ode23_packets(events=...): level crossings of the packet state located on every
accepted step of the per-packet ode23 solve.  The oracle is ode23_events_oracle.ode23 on one packet with the mode's
oracle RHS; the solve itself must be swrt_ode23_packets' bit for bit."""
import ctypes as C

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from swraytracing_b200 import workloads as W
import ode23_events_oracle as E
from oracle import swrt_oracle as O
from test_ode23_packets import F0, GH0, L, MODES, THREE, engine, make_packets, make_psik
from test_mex_gateway import Mex

pytestmark = pytest.mark.gpu

T = 2.0
TSPAN = np.linspace(0.0, T, 11)
# crossings that some of make_packets' packets make within T: |k| starts at 3, omega at sqrt(18)
EVENTS = [(S.EVENT_X, 0.0, 0, 0), (S.EVENT_Y, 0.5, -1, 0), (S.EVENT_KMAG, 3.05, 0, 0), (S.EVENT_OMEGA, 4.3, 1, 0)]
KEYS = ("steps", "rejected", "status", "t_end")


def solve(e, pk, events=None, tspan=TSPAN, two=True, **kw):
    e.set_packets(*pk)
    e.launch_count(reset=True)
    st = e.ode23_packets(tspan, T if two else None, events=events, **kw)
    st["launches"] = e.launch_count()
    return st, np.stack(e.get_packets())


def oracle_rhs(mode, nx, two):
    """odefun of one packet with the mode's oracle RHS: the exact series (SPECTRAL, NUFFT) or the Lagrange stencil"""
    kx_, ky_ = O.wavenumbers(nx)
    planes = [O.velocity_planes_k(make_psik(nx, s), kx_, ky_) for s in (7, 8)]
    dx = L / nx
    if mode == S.MODE_LAGRANGE6:
        names = ("u", "v", "ux", "uy", "vx", "vy")
        bf = [{k: O.k2g(p) for k, p in zip(names, pl)} for pl in planes]
        def e6(x, y, al):
            U, g = O.interpolate_U(bf[0], bf[1] if two else bf[0], al, np.stack([x, y], axis=1), dx, 1e-13)
            return U[:, 0], U[:, 1], g["u_x"], g["u_y"], g["v_x"], g["v_y"]
    else:
        def e6(x, y, al):
            a = O.spectral_eval_planes(x, y, planes[0], dx, nx)
            return a if al == 0.0 else (1 - al) * a + al * O.spectral_eval_planes(x, y, planes[1], dx, nx)

    def odefun(t, y):
        return np.concatenate(O.rhs_from_eval(e6(y[0:1], y[1:2], t / T if two else 0.0), y[2:3], y[3:4], F0, 1.0))
    return odefun


def assert_same_solve(a, ya, b, yb):
    assert np.array_equal(ya, yb, equal_nan=True) and np.array_equal(a["Y"], b["Y"], equal_nan=True)
    for key in KEYS + ("nfevals", "nsteps", "nfailed", "launches", "host_waits"):
        assert np.array_equal(a[key], b[key]), key


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("two", [False, True])
def test_records_against_oracle_and_solve_unchanged(mode, nx, two):
    pk = make_packets(40)
    with engine(mode, nx, two) as e:
        solve(e, pk, two=two)                             # the first solve on a handle also prepares the flow
        a, ya = solve(e, pk, two=two)
        b, yb = solve(e, pk, EVENTS, two=two, ev_cap=8)
    assert_same_solve(a, ya, b, yb)
    assert b["terminated"] == 0 and b["events"] == b["ne"].sum() and (b["ne"] > 0).sum() >= 4
    assert len(set(b["ie"][b["ie"] > 0])) >= 3 and b["ne"].max() <= 8
    odefun = oracle_rhs(mode, nx, two)
    scale = np.maximum(np.abs(ya).max(axis=0), 1.0)
    for i in range(pk.shape[1]):
        _, ref = E.ode23(odefun, TSPAN, pk[:, i], events=EVENTS, f=F0, gH=GH0)
        m = b["ne"][i]
        assert m == ref["te"].size, i
        assert np.array_equal(b["ie"][:m, i], ref["ie"]) and np.all(b["ie"][m:, i] == 0)
        assert np.all(np.abs(b["te"][:m, i] - ref["te"]) <= 1e-12 * T), i
        assert np.all(np.abs(b["ye"][:m, :, i] - ref["ye"]) <= 1e-12 * scale[i]), i
        assert np.isnan(b["te"][m:, i]).all() and np.isnan(b["ye"][m:, :, i]).all()
        for r in range(m):                                # g_j(ye) is 0 or has the post-crossing sign
            j = b["ie"][r, i] - 1
            kind, level, d, _ = EVENTS[j]
            g = E.event_g(kind, level, b["ye"][r, :, i], F0, GH0)
            # a crossing the direction allows; without one, the sign alternates from the side of y0
            post = d if d else -np.sign(E.event_g(kind, level, pk[:, i], F0, GH0)) * (-1) ** (b["ie"][:r, i] == j + 1).sum()
            assert g == 0.0 or np.sign(g) == post, (i, r)


@pytest.mark.parametrize("mode,nx", MODES)
def test_terminal_omega_level(mode, nx):
    pk = make_packets(200, seed=4)
    ev = [(S.EVENT_X, 0.0, 0, 0), (S.EVENT_OMEGA, 4.4, 1, 1)]
    with engine(mode, nx, True) as e:
        a, ya = solve(e, pk)
        b, yb = solve(e, pk, ev)
    stop = b["status"] == 2
    assert 0 < stop.sum() < pk.shape[1] and b["terminated"] == stop.sum() and b["stopped"] == 0
    free = ~stop
    assert np.array_equal(yb[:, free], ya[:, free])
    for key in KEYS:
        assert np.array_equal(b[key][free], a[key][free]), key
    assert np.array_equal(b["Y"][:, :, free], a["Y"][:, :, free])
    for i in np.flatnonzero(stop):
        r = b["ne"][i] - 1                               # the terminal record is the packet's last
        assert b["ie"][r, i] == 2 and b["t_end"][i] == b["te"][r, i] and np.array_equal(yb[:, i], b["ye"][r, :, i])
        reached = TSPAN <= b["te"][r, i]
        assert np.array_equal(b["Y"][reached, :, i], a["Y"][reached, :, i]) and np.isnan(b["Y"][~reached, :, i]).all()
        assert b["steps"][i] <= a["steps"][i]


@pytest.mark.parametrize("mode,nx", THREE)
def test_independence(mode, nx):
    pk = make_packets(300, seed=11)
    rs = np.random.RandomState(2)
    sub = np.sort(rs.choice(pk.shape[1], 37, replace=False))
    perm = rs.permutation(pk.shape[1])
    ev = EVENTS[:3] + [(S.EVENT_OMEGA, 4.4, 1, 1)]
    rec = ("te", "ye", "ie", "ne") + KEYS
    with engine(mode, nx, True) as e:
        a, ya = solve(e, pk, ev, ev_cap=8)
        b, yb = solve(e, pk[:, sub], ev, ev_cap=8)
        c, yc = solve(e, pk[:, perm], ev, ev_cap=8)
        d, _ = solve(e, pk, ev + [(S.EVENT_L, 0.0, 0, 0)], ev_cap=8)
        one, _ = solve(e, pk, ev, ev_cap=1)
    assert a["events"] > 0 and a["terminated"] > 0
    assert np.array_equal(yb, ya[:, sub]) and np.array_equal(yc, ya[:, perm])
    for key in rec:
        assert np.array_equal(b[key], a[key][..., sub], equal_nan=True), key
        assert np.array_equal(c[key], a[key][..., perm], equal_nan=True), key
    # another non-terminal event leaves the first events' records as they were
    for i in np.flatnonzero(d["ne"] <= 8):
        sel = d["ie"][:, i] <= len(ev)
        sel &= d["ie"][:, i] > 0
        m = a["ne"][i]
        assert sel.sum() == m and np.array_equal(d["ie"][sel, i], a["ie"][:m, i])
        assert np.array_equal(d["te"][sel, i], a["te"][:m, i]) and np.array_equal(d["ye"][sel, :, i], a["ye"][:m, :, i])
    # ev_cap = 1 keeps the first record and counts every event
    assert np.array_equal(one["ne"], a["ne"]) and np.array_equal(one["te"][0], a["te"][0], equal_nan=True)
    assert np.array_equal(one["ye"][0], a["ye"][0], equal_nan=True) and np.array_equal(one["ie"][0], a["ie"][0])


@pytest.mark.parametrize("mode,nx", THREE)
def test_two_devices_equal_one_bit_for_bit(mode, nx):
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two GPUs")
    pk = make_packets(3001, seed=12)
    ev = EVENTS[:3] + [(S.EVENT_OMEGA, 4.4, 1, 1)]
    res = []
    for ngpu in (1, 2):
        with engine(mode, nx, True, ngpu=ngpu) as e:
            res.append(solve(e, pk, ev))
    (a, ya), (b, yb) = res
    assert np.array_equal(ya, yb) and np.array_equal(a["Y"], b["Y"], equal_nan=True)
    for key in ("te", "ye", "ie", "ne", "events", "terminated") + KEYS:
        assert np.array_equal(a[key], b[key], equal_nan=True), key


@pytest.mark.parametrize("mode,nx", MODES)
def test_zero_flow_x_crossing_is_analytic(mode, nx):
    n = 64
    i = np.arange(n)
    pk = np.stack([np.full(n, -0.5), 0.1 * i, 2.0 + 0.01 * i, np.cos(i)])
    xdot = pk[2] / np.sqrt(F0 ** 2 + GH0 * (pk[2] ** 2 + pk[3] ** 2))
    with S.Engine(nx, L, F0, GH0, mode) as e:
        e.set_flow_spectral(np.zeros((nx - 1, nx // 2), dtype=complex), slot=0)
        st, _ = solve(e, pk, [(S.EVENT_X, 0.0, 0, 0), (S.EVENT_X, 0.25, 1, 0)], two=False)
    te = np.stack([0.5 / xdot, 0.75 / xdot])
    assert np.array_equal(st["ne"], np.full(n, 2)) and np.array_equal(st["ie"][:2], np.tile([[1], [2]], (1, n)))
    assert np.all(np.abs(st["te"][:2] - te) <= 1e-13 * te)


def test_argument_errors_leave_the_handle_usable():
    lib = S.load_library()
    pk = make_packets(30)
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        ref, yref = solve(e, pk, EVENTS)

        def call(evs, nev=None, cap=2, tspan=TSPAN):
            arr = (S.engine._Event * max(len(evs), 1))(*[S.engine._Event(*ev) for ev in evs])
            ts = np.asarray(tspan, dtype=np.float64)
            st = (C.c_int64 * 7)()
            return lib.swrt_ode23_packets_events(e._h, ts.ctypes.data_as(C.POINTER(C.c_double)), ts.size, T, 1e-3, 1e-6, arr,
                                                 len(evs) if nev is None else nev, cap, None, None, None, None, None, None, None, st)
        good = (S.EVENT_X, 0, 0, 0, 0.5)                          # kind, direction, terminal, reserved, level
        assert call([good]) == 0
        bad = [call([good], nev=0), call([good] * 9), call([good], cap=-1), call([(6, 0, 0, 0, 0.5)]), call([(-1, 0, 0, 0, 0.5)]),
               call([(0, 2, 0, 0, 0.5)]), call([(0, -2, 0, 0, 0.5)]), call([(0, 0, 2, 0, 0.5)]), call([(0, 0, 0, 1, 0.5)]),
               call([(0, 0, 0, 0, np.inf)]), call([(0, 0, 0, 0, np.nan)]), call([good], tspan=[0.0, 1.0, 1.0, 2.0]),
               call([good], tspan=[2.0, 0.0])]
        assert bad == [-1] * len(bad)
        got, ygot = solve(e, pk, EVENTS)
    assert np.array_equal(ygot, yref)
    for key in ("te", "ye", "ie", "ne") + KEYS:
        assert np.array_equal(got[key], ref[key], equal_nan=True), key


def test_reference_api_and_sharded_ensemble_pass_events_through():
    from swraytracing_b200.distributed import ShardedEnsemble
    pk = make_packets(20)
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        ref, yref = solve(e, pk, EVENTS)
        e.set_packets(*pk)
        a = R.ode23(e, TSPAN, T, per_packet=True, events=EVENTS)
        ya = np.stack(e.get_packets())
        with pytest.raises(ValueError):
            R.ode23(e, TSPAN, T, events=EVENTS)
    assert np.array_equal(ya, yref)
    for key in ("te", "ye", "ie", "ne"):
        assert np.array_equal(a[key], ref[key], equal_nan=True), key
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        ens = ShardedEnsemble(e, pk.shape[1])
        ens.set_packets_global(*pk)
        b = ens.ode23(TSPAN, T, per_packet=True, events=EVENTS)
        with pytest.raises(ValueError):
            ens.ode23(TSPAN, T, events=EVENTS)
    for key in ("te", "ye", "ie", "ne"):
        assert np.array_equal(b[key], ref[key], equal_nan=True), key


@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    return Mex(request.param)


def test_gateway_ode23_events(mex):
    w = W.make_workload("C3", n_packets=301, nx=32)
    h = mex("create", float(w.nx), w.L, w.f, w.gH, float(S.MODE_LAGRANGE6))
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6)
    for slot, psik in ((0.0, w.psik), (1.0, w.psik2)):
        mex("set_flow_spectral", h, slot, psik, nlhs=0)
        eng.set_flow_spectral(psik, int(slot))
    mex("set_packets", h, w.x, w.y, w.k, w.l, nlhs=0)
    eng.set_packets(w.x, w.y, w.k, w.l)
    tspan = w.dt * np.linspace(0.0, 1.0, 6)
    om = np.sqrt(w.f * w.f + w.gH * (w.k * w.k + w.l * w.l))
    events = [(S.EVENT_X, float(np.median(w.x)), 0, 0), (S.EVENT_OMEGA, float(np.quantile(om, 0.6)), 0, 1)]
    ev = np.array([[k, lv, d, t] for k, lv, d, t in events], dtype=np.float64)
    cap = 3
    st, Y, pstat, t_end, te, ye, ie, ne = mex("ode23_events", h, tspan, w.dt, 1e-6, 1e-7, ev, float(cap), nlhs=8)
    ref = eng.ode23_packets(tspan, w.dt, 1e-6, 1e-7, events=events, ev_cap=cap)
    assert ref["events"] > 0 and ref["terminated"] > 0
    assert np.array_equal(np.ravel(st), [ref[k] for k in ("nsteps", "nfailed", "nfevals", "stopped", "host_waits", "events", "terminated")])
    assert np.array_equal(pstat, np.stack([ref["steps"], ref["rejected"], ref["status"]], axis=1))
    assert np.array_equal(t_end, ref["t_end"])
    assert np.array_equal(Y.reshape(301, 4, tspan.size, order="F"), ref["Y"].transpose(2, 1, 0), equal_nan=True)
    assert np.array_equal(te, ref["te"].T, equal_nan=True) and np.array_equal(ie, ref["ie"].T)
    assert np.array_equal(ye.reshape(301, 4, cap, order="F"), ref["ye"].transpose(2, 1, 0), equal_nan=True)
    assert np.array_equal(np.ravel(ne), ref["ne"])
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()))
    mex("destroy", h, nlhs=0); eng.close()
