"""swrt_ode23_packets_tspans_events / Engine.ode23_packets_tspans_events: events on the per-packet solve with a tspan row
per packet in either direction.  Forward rows must give swrt_ode23_packets_events' results, a backward solve must be the
mirror image of a forward one bit for bit, the records must match ode23_events_tspans_oracle per packet, and apart from
a terminal stop the solve must be swrt_ode23_packets_tspans' bit for bit."""
import ctypes as C

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
import ode23_events_oracle as E
import ode23_events_tspans_oracle as ET
from test_mex_gateway import Mex
from test_ode23_backward import engine as signed_engine
from test_ode23_events import oracle_rhs
from test_ode23_packets import F0, GH0, MODES, THREE, engine, make_packets, scale_of

pytestmark = pytest.mark.gpu

T = 2.0                        # the flow's tmax (alpha = t/T), as oracle_rhs assumes
TOLS = [(1e-3, 1e-6), (1e-6, 1e-7)]
NEG = np.array([1.0, 1.0, -1.0, -1.0])
FWD = np.linspace(0.0, T, 11)
# crossings that some of make_packets' packets make within T: |k| starts at 3, omega at sqrt(18)
EVENTS = [(S.EVENT_X, 0.0, 0, 0), (S.EVENT_Y, 0.5, -1, 0), (S.EVENT_KMAG, 3.05, 0, 0), (S.EVENT_OMEGA, 4.3, 1, 0)]
TERMINAL = EVENTS[:3] + [(S.EVENT_OMEGA, 4.4, 1, 1)]
KEYS = ("steps", "rejected", "status", "t_end")
RECORDS = ("te", "ye", "ie", "ne")
STATS = ("nsteps", "nfailed", "nfevals", "stopped", "host_waits", "events", "terminated")


def ev_solve(e, pk, ts, events, tmax=T, rtol=1e-3, atol=1e-6, ev_cap=4):
    e.set_packets(*pk)
    st = e.ode23_packets_tspans_events(ts, tmax, events, rtol, atol, ev_cap)
    return st, np.stack(e.get_packets())


def fwd_solve(e, pk, ts, events, tmax=T, rtol=1e-3, atol=1e-6, ev_cap=4):
    e.set_packets(*pk)
    st = e.ode23_packets(ts, tmax, rtol, atol, events=events, ev_cap=ev_cap)
    return st, np.stack(e.get_packets())


def rows_solve(e, pk, ts, tmax=T, rtol=1e-3, atol=1e-6):
    e.set_packets(*pk)
    st = e.ode23_packets(ts, tmax, rtol, atol)
    return st, np.stack(e.get_packets())


def assert_same(a, ya, b, yb, cols=slice(None)):
    assert np.array_equal(ya, yb[:, cols], equal_nan=True) and np.array_equal(a["Y"], b["Y"][..., cols], equal_nan=True)
    for key in RECORDS + KEYS:
        assert np.array_equal(a[key], b[key][..., cols], equal_nan=True), key


@pytest.mark.parametrize("mode,nx", THREE)
@pytest.mark.parametrize("two", [False, True])
def test_forward_rows_equal_ode23_packets_events(mode, nx, two):
    pk = make_packets(200, seed=13)
    tmax = T if two else None
    with engine(mode, nx, two) as e:
        a, ya = fwd_solve(e, pk, FWD, TERMINAL, tmax, 1e-6, 1e-7, ev_cap=6)
        b, yb = ev_solve(e, pk, np.repeat(FWD[:, None], 200, axis=1), TERMINAL, tmax, 1e-6, 1e-7, ev_cap=6)
        c, yc = ev_solve(e, pk, FWD, TERMINAL, tmax, 1e-6, 1e-7, ev_cap=6)            # the 1-D form
    assert a["events"] > 0 and a["terminated"] < 200 and (a["terminated"] > 0 or not two)
    assert_same(b, yb, c, yc)
    assert all(b[k] == c[k] for k in STATS)
    for key in ("steps", "rejected", "status", "ie", "ne"):
        assert np.array_equal(a[key], b[key]), key
    assert all(a[k] == b[k] for k in STATS), [(k, a[k], b[k]) for k in STATS]
    if mode == S.MODE_SPECTRAL and two:          # f1 from both frames' planes instead of the blended stack
        sc = scale_of(ya)
        assert np.all(np.abs(ya - yb) <= 1e-12 * sc) and np.all(np.abs(a["Y"] - b["Y"]) <= 1e-12 * sc[None], where=~np.isnan(a["Y"]))
        assert np.array_equal(np.isnan(a["Y"]), np.isnan(b["Y"])) and np.array_equal(np.isnan(a["te"]), np.isnan(b["te"]))
        used = ~np.isnan(a["te"])
        assert np.all(np.abs(a["te"][used] - b["te"][used]) <= 1e-12 * T)
        assert np.all(np.abs(a["ye"] - b["ye"]) <= 1e-12 * sc[None], where=~np.isnan(a["ye"]))
        assert np.all(np.abs(a["t_end"] - b["t_end"]) <= 1e-12 * T)
    else:
        assert_same(a, ya, b, yb)


@pytest.mark.parametrize("mode,nx", THREE)
@pytest.mark.parametrize("tol", TOLS)
@pytest.mark.parametrize("terminal", [False, True])
def test_mirror_identity(mode, nx, tol, terminal):
    """steady flow: backward over [T .. 0] in psi == swrt_ode23_packets_events over [-T .. 0] in -psi with (k, l) negated,
    bit for bit; X, Y, |k| and omega keep their values under the mirror, K's level and direction are negated with k"""
    pk = make_packets(200)
    ts = np.linspace(T, 0.0, 11)
    ev = ([(S.EVENT_X, 0.0, 0, 1)] + EVENTS[1:] if terminal else EVENTS) + [(S.EVENT_K, 1.0, 1, 0)]
    evm = ev[:-1] + [(S.EVENT_K, -1.0, -1, 0)]
    with signed_engine(mode, nx, False) as e, signed_engine(mode, nx, False, sign=-1.0) as em:
        b, yb = ev_solve(e, pk, ts, ev, None, *tol, ev_cap=8)
        f, yf = fwd_solve(em, pk * NEG[:, None], -ts, evm, None, *tol, ev_cap=8)
    assert b["events"] > 0 and (b["terminated"] > 0) == terminal and b["terminated"] < 200
    assert b["steps"][b["status"] == 0].min() >= 10
    assert all(b[k] == f[k] for k in STATS)
    for key in ("steps", "rejected", "status", "ie", "ne"):
        assert np.array_equal(b[key], f[key]), key
    assert np.array_equal(b["t_end"], -f["t_end"]) and np.array_equal(b["te"], -f["te"], equal_nan=True)
    assert np.array_equal(b["ye"], f["ye"] * NEG[None, :, None], equal_nan=True)
    assert np.array_equal(yb, yf * NEG[:, None]) and np.array_equal(b["Y"], f["Y"] * NEG[None, :, None], equal_nan=True)
    for i in range(pk.shape[1]):                          # in order of encounter: te decreasing backward
        assert np.all(np.diff(b["te"][:min(b["ne"][i], 8), i]) <= 0), i


def staggered_rows(n, seed=3):
    """backward rows from a start in [1.2, 2] to 0 and forward rows from a release in [0, 0.8] to T, alternating"""
    rs = np.random.RandomState(seed)
    ts = np.empty((9, n))
    for i in range(n):
        ts[:, i] = np.linspace(rs.uniform(1.2, T), 0.0, 9) if i % 2 == 0 else np.linspace(rs.uniform(0.0, 0.8), T, 9)
    return ts


@pytest.mark.parametrize("mode,nx", MODES)
def test_records_against_oracle(mode, nx):
    pk = make_packets(40)
    ts = staggered_rows(40)
    with engine(mode, nx, True) as e:
        b, yb = ev_solve(e, pk, ts, EVENTS, ev_cap=8)
    assert b["terminated"] == 0 and (b["ne"] > 0).sum() >= 4 and b["ne"].max() <= 8
    assert (b["ne"][0::2] > 0).sum() >= 2 and (b["ne"][1::2] > 0).sum() >= 2
    odefun = oracle_rhs(mode, nx, True)
    scale = np.maximum(np.abs(yb).max(axis=0), 1.0)
    for i in range(pk.shape[1]):
        _, ref = ET.ode23(odefun, ts[:, i], pk[:, i], events=EVENTS, f=F0, gH=GH0)
        m = b["ne"][i]
        assert m == ref["te"].size, i
        assert np.array_equal(b["ie"][:m, i], ref["ie"]) and np.all(b["ie"][m:, i] == 0)
        assert np.all(np.abs(b["te"][:m, i] - ref["te"]) <= 1e-12 * T), i
        assert np.all(np.abs(b["ye"][:m, :, i] - ref["ye"]) <= 1e-12 * scale[i]), i
        assert np.isnan(b["te"][m:, i]).all() and np.isnan(b["ye"][m:, :, i]).all()
        for r in range(m):                                # g_j(ye) is 0 or has the post-crossing sign, in integration order
            j = b["ie"][r, i] - 1
            kind, level, d, _ = EVENTS[j]
            g = E.event_g(kind, level, b["ye"][r, :, i], F0, GH0)
            post = d if d else -np.sign(E.event_g(kind, level, pk[:, i], F0, GH0)) * (-1) ** (b["ie"][:r, i] == j + 1).sum()
            assert g == 0.0 or np.sign(g) == post, (i, r)


def mixed_rows(n):
    """forward, backward and zero-length rows, in turn"""
    ts = np.empty((7, n))
    for i in range(n):
        t0 = 0.1 * (i % 7)
        ts[:, i] = (np.linspace(t0, T, 7), np.linspace(T - t0, 0.0, 7), np.full(7, 0.3 + t0))[i % 3]
    return ts


@pytest.mark.parametrize("mode,nx", THREE)
def test_mixed_rows(mode, nx):
    n = 60
    pk = make_packets(n, seed=4)
    ts = mixed_rows(n)
    with engine(mode, nx, True) as e:
        b, yb = ev_solve(e, pk, ts, TERMINAL, ev_cap=8)
        a, ya = rows_solve(e, pk, ts)
        one = [ev_solve(e, pk[:, i:i + 1], ts[:, i:i + 1], TERMINAL, ev_cap=8) for i in range(0, n, 5)]
    assert b["events"] > 0 and b["terminated"] > 0
    for (s, y), i in zip(one, range(0, n, 5)):            # each packet is its own solve
        assert_same(s, y, b, yb, slice(i, i + 1))
    zero = np.arange(n) % 3 == 2
    assert np.all(b["ne"][zero] == 0) and np.array_equal(yb[:, zero], pk[:, zero]) and np.all(b["steps"][zero] == 1)
    assert np.array_equal(b["t_end"][zero], ts[-1, zero])
    free = b["status"] != 2                               # not stopped by a terminal event: swrt_ode23_packets_tspans
    assert (free & ~zero).sum() > 0
    assert np.array_equal(yb[:, free], ya[:, free]) and np.array_equal(b["Y"][..., free], a["Y"][..., free])
    for key in KEYS:
        assert np.array_equal(b[key][free], a[key][free]), key


@pytest.mark.parametrize("mode,nx", THREE)
def test_terminal_backward_stop(mode, nx):
    n = 200
    pk = make_packets(n, seed=4)
    ts = np.linspace(T, 0.0, 11)
    with engine(mode, nx, True) as e:
        a, ya = rows_solve(e, pk, np.repeat(ts[:, None], n, axis=1))
        b, yb = ev_solve(e, pk, ts, [(S.EVENT_X, 0.0, 0, 0), (S.EVENT_OMEGA, 4.4, 0, 1)], ev_cap=8)
    stop = b["status"] == 2
    assert 0 < stop.sum() < n and b["terminated"] == stop.sum() and b["stopped"] == 0
    free = ~stop
    assert np.array_equal(yb[:, free], ya[:, free]) and np.array_equal(b["Y"][..., free], a["Y"][..., free])
    for i in np.flatnonzero(stop):
        r = b["ne"][i] - 1                                # the terminal record is the packet's last
        assert b["ne"][i] <= 8 and b["ie"][r, i] == 2
        assert b["t_end"][i] == b["te"][r, i] and np.array_equal(yb[:, i], b["ye"][r, :, i])
        assert 0.0 < b["t_end"][i] < T
        reached = ts >= b["te"][r, i]                     # backward: the rows before te* in integration order
        assert np.array_equal(b["Y"][reached, :, i], a["Y"][reached, :, i]) and np.isnan(b["Y"][~reached, :, i]).all()
        assert b["steps"][i] <= a["steps"][i]


@pytest.mark.parametrize("mode,nx", THREE)
def test_independence_and_a_packet_that_blows_up(mode, nx):
    n = 300
    pk = make_packets(n, seed=11)
    ts = mixed_rows(n)
    rs = np.random.RandomState(2)
    sub = np.sort(rs.choice(n, 37, replace=False))
    perm = rs.permutation(n)
    with engine(mode, nx, True) as e:
        a, ya = ev_solve(e, pk, ts, TERMINAL, ev_cap=8)
        b, yb = ev_solve(e, pk[:, sub], ts[:, sub], TERMINAL, ev_cap=8)
        c, yc = ev_solve(e, pk[:, perm], ts[:, perm], TERMINAL, ev_cap=8)
        bad = pk.copy()
        bad[2, 17] = np.inf
        d, yd = ev_solve(e, bad, ts, TERMINAL, ev_cap=8)
    assert a["events"] > 0 and a["terminated"] > 0
    assert_same(b, yb, a, ya, sub)
    assert_same(c, yc, a, ya, perm)
    assert d["status"][17] == 1 and d["stopped"] == 1
    good = np.delete(np.arange(n), 17)
    assert_same({k: v[..., good] for k, v in d.items() if k in RECORDS + KEYS + ("Y",)}, yd[:, good], a, ya, good)


@pytest.mark.parametrize("mode,nx", THREE)
def test_two_devices_equal_one_bit_for_bit(mode, nx):
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two GPUs")
    n = 3001
    pk = make_packets(n, seed=12)
    ts = mixed_rows(n)
    res = []
    for ngpu in (1, 2):
        with engine(mode, nx, True, ngpu=ngpu) as e:
            res.append(ev_solve(e, pk, ts, TERMINAL))
    (a, ya), (b, yb) = res
    assert_same(a, ya, b, yb)
    assert all(a[k] == b[k] for k in ("nsteps", "nfailed", "nfevals", "stopped", "events", "terminated"))


def test_argument_errors_leave_the_packets_untouched_and_the_handle_usable():
    lib = S.load_library()
    n = 30
    pk = make_packets(n)
    ts = mixed_rows(n)
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        ref, yref = ev_solve(e, pk, ts, EVENTS)
        e.set_packets(*pk)

        def call(evs, nev=None, cap=2, tspan=ts):
            arr = (S.engine._Event * max(len(evs), 1))(*[S.engine._Event(*ev) for ev in evs])
            t = np.ascontiguousarray(tspan, dtype=np.float64)
            st = (C.c_int64 * 7)()
            return lib.swrt_ode23_packets_tspans_events(e._h, t.ctypes.data_as(C.POINTER(C.c_double)), t.shape[0], T, 1e-3, 1e-6,
                                                        arr, len(evs) if nev is None else nev, cap, None, None, None, None, None,
                                                        None, None, st)
        good = (S.EVENT_X, 0, 0, 0, 0.5)                          # kind, direction, terminal, reserved, level
        nonfinite, against = ts.copy(), ts.copy()
        nonfinite[3, 7] = np.nan
        against[2, 4] = against[1, 4] - 0.05 if ts[-1, 4] >= ts[0, 4] else against[1, 4] + 0.05
        assert (ts[-1, 4] - ts[0, 4]) * (against[2, 4] - against[1, 4]) < 0
        bad = [call([good], nev=0), call([good] * 9), call([good], cap=-1), call([(6, 0, 0, 0, 0.5)]), call([(-1, 0, 0, 0, 0.5)]),
               call([(0, 2, 0, 0, 0.5)]), call([(0, -2, 0, 0, 0.5)]), call([(0, 0, 2, 0, 0.5)]), call([(0, 0, 0, 1, 0.5)]),
               call([(0, 0, 0, 0, np.inf)]), call([(0, 0, 0, 0, np.nan)]), call([good], tspan=nonfinite),
               call([good], tspan=ts[:1]), call([good], tspan=against)]
        assert bad == [-1] * len(bad) and b"packet 4" in lib.swrt_last_error(e._h)
        assert np.array_equal(np.stack(e.get_packets()), pk)
        got, ygot = ev_solve(e, pk, ts, EVENTS)
    assert_same(got, ygot, ref, yref)


@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    return Mex(request.param)


@pytest.mark.parametrize("matrix", [False, True])
def test_gateway_ode23_tspans_events(mex, matrix):
    n = 301
    w = W.make_workload("C3", n_packets=n, nx=32)
    h = mex("create", float(w.nx), w.L, w.f, w.gH, float(S.MODE_LAGRANGE6))
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6)
    for slot, psik in ((0.0, w.psik), (1.0, w.psik2)):
        mex("set_flow_spectral", h, slot, psik, nlhs=0)
        eng.set_flow_spectral(psik, int(slot))
    mex("set_packets", h, w.x, w.y, w.k, w.l, nlhs=0)
    eng.set_packets(w.x, w.y, w.k, w.l)
    if matrix:                                       # (ntspan, n): half the packets backward, a few zero-length
        ts = w.dt * np.repeat(np.linspace(0.0, 1.0, 6)[:, None], n, axis=1)
        ts[:, 1::2] = ts[::-1, 1::2]
        ts[:, 5::50] = 0.5 * w.dt
    else:
        ts = w.dt * np.linspace(1.0, 0.0, 6)
    om = np.sqrt(w.f * w.f + w.gH * (w.k * w.k + w.l * w.l))
    events = [(S.EVENT_X, float(np.median(w.x)), 0, 0), (S.EVENT_OMEGA, float(np.quantile(om, 0.6)), 0, 1)]
    ev = np.array([[k, lv, d, t] for k, lv, d, t in events], dtype=np.float64)
    cap = 3
    # the gateway takes tspan n x m (row i = packet i) or a vector
    st, Y, pstat, t_end, te, ye, ie, ne = mex("ode23_tspans_events", h, ts.T.copy() if matrix else ts, w.dt, 1e-6, 1e-7, ev,
                                              float(cap), nlhs=8)
    ref = eng.ode23_packets_tspans_events(ts, w.dt, events, 1e-6, 1e-7, cap)
    assert ref["events"] > 0 and ref["terminated"] > 0
    assert np.array_equal(np.ravel(st), [ref[k] for k in STATS])
    assert np.array_equal(pstat, np.stack([ref["steps"], ref["rejected"], ref["status"]], axis=1))
    assert np.array_equal(np.ravel(t_end), ref["t_end"])
    assert np.array_equal(Y.reshape(n, 4, 6, order="F"), ref["Y"].transpose(2, 1, 0), equal_nan=True)
    assert np.array_equal(te, ref["te"].T, equal_nan=True) and np.array_equal(ie, ref["ie"].T)
    assert np.array_equal(ye.reshape(n, 4, cap, order="F"), ref["ye"].transpose(2, 1, 0), equal_nan=True)
    assert np.array_equal(np.ravel(ne), ref["ne"])
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()))
    st2 = mex("ode23_tspans_events", h, ts.T.copy() if matrix else ts, w.dt, 1e-3, 1e-6, ev, 0.0)     # stats only
    assert np.ravel(st2).shape == (7,)
    mex("destroy", h, nlhs=0); eng.close()
