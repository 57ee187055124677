"""swrt_ode23_packets_tspans / Engine.ode23_packets with a 2-D tspan: every packet with its own tspan.  The oracle is the
definition: packet i equals swrt_ode23 (Engine.ode23) run on a handle that holds packet i alone, with tspan[:, i]."""
import re

import numpy as np
import pytest

import swraytracing_b200 as S
from test_ode23_packets import MODES, THREE, engine, make_packets, scale_of

pytestmark = pytest.mark.gpu


def rows_solve(e, pk, ts, tmax, rtol=1e-3, atol=1e-6):
    e.set_packets(*pk)
    st = e.ode23_packets(ts, tmax, rtol, atol)
    return st, np.stack(e.get_packets())


def one_packet_solves(e, pk, ts, tmax, rtol=1e-3, atol=1e-6):
    """swrt_ode23 on a handle holding packet i alone with tspan ts[:, i], for every i: (steps, rejected, final state, Y or
    None, t of failure, signed step sizes)"""
    out = []
    for i in range(pk.shape[1]):
        e.set_packets(*pk[:, i:i + 1])
        try:
            st = e.ode23(ts[:, i], tmax, rtol, atol, trace=4096)
            Y = st["Y"][:, :, 0] if "Y" in st else None
            out.append((st["nsteps"], st["nfailed"], np.stack(e.get_packets())[:, 0], Y, None, st["h"]))
        except S.SwrtError as ex:
            t = float(re.search(r"at t = (\S+)", str(ex)).group(1))
            out.append((None, None, np.stack(e.get_packets())[:, 0], None, t, None))
    return out


def assert_rows_equal_one_packet_solves(st, yp, ref, ts, exact):
    n = yp.shape[1]
    assert np.array_equal(st["steps"], [r[0] for r in ref]) and np.array_equal(st["rejected"], [r[1] for r in ref])
    assert st["nsteps"] == st["steps"].sum() and st["nfailed"] == st["rejected"].sum()
    assert st["nfevals"] == n + 3 * (st["nsteps"] + st["nfailed"]) and st["stopped"] == 0
    assert np.all(st["status"] == 0) and np.array_equal(st["t_end"], ts[-1]) and np.array_equal(st["t"], ts[-1])
    y1 = np.stack([r[2] for r in ref], axis=1)
    tol = 0.0 if exact else 1e-12 * scale_of(yp)
    assert np.all(np.abs(yp - y1) <= tol)
    if "Y" in st:
        Y1 = np.stack([r[3] for r in ref], axis=2)
        assert np.all(np.abs(st["Y"] - Y1) <= (tol if exact else tol[None]))


def staggered(n, seed, t_lo=(0.0, 0.1), t_hi=(0.25, 0.4)):
    rs = np.random.RandomState(seed)
    return np.stack([rs.uniform(*t_lo, n), rs.uniform(*t_hi, n)])


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("two", [False, True])
@pytest.mark.parametrize("tol", [(1e-3, 1e-6), (1e-6, 1e-7)])
def test_each_packet_equals_its_one_packet_solve(mode, nx, two, tol):
    tmax = 0.4
    pk = make_packets(40)
    ts = staggered(40, 1)                       # t0 in [0, 0.1], tfinal in [0.25, 0.4]: inside the frame interval
    with engine(mode, nx, two) as e:
        st, yp = rows_solve(e, pk, ts, tmax if two else None, *tol)
        ref = one_packet_solves(e, pk, ts, tmax if two else None, *tol)
    assert st["steps"].min() >= 10                # MaxStep = 0.1*|tf - t0|
    assert_rows_equal_one_packet_solves(st, yp, ref, ts, not (mode == S.MODE_SPECTRAL and two))


@pytest.mark.parametrize("mode,nx", THREE)
def test_mixed_directions_and_zero_length_rows(mode, nx):
    n, nt = 30, 6
    pk = make_packets(n, seed=6)
    rs = np.random.RandomState(3)
    T = rs.uniform(0.2, 0.4, n)
    kind = np.arange(n) % 3                      # 0 forward [t0 .. T], 1 backward [T .. 0], 2 constant
    ts = np.empty((nt, n))
    for i in range(n):
        if kind[i] == 0:
            ts[:, i] = np.linspace(0.4 - T[i], 0.4, nt)
        elif kind[i] == 1:
            ts[:, i] = np.linspace(T[i], 0.0, nt)
        else:
            ts[:, i] = T[i]
    with engine(mode, nx, True) as e:
        st, yp = rows_solve(e, pk, ts, 0.4, 1e-6, 1e-7)
        ref = one_packet_solves(e, pk, ts, 0.4, 1e-6, 1e-7)
    assert_rows_equal_one_packet_solves(st, yp, ref, ts, mode != S.MODE_SPECTRAL)
    # the one-packet solves step forward, backward and not at all
    for i in range(n):
        h = ref[i][5]
        assert np.all(h > 0) if kind[i] == 0 else np.all(h < 0) if kind[i] == 1 else np.array_equal(h, [0.0])
    # a constant row: one accepted step of size 0, the state unchanged and every dense row y0
    c = kind == 2
    assert np.all(st["steps"][c] == 1) and np.all(st["rejected"][c] == 0)
    assert np.array_equal(yp[:, c], pk[:, c]) and np.array_equal(st["Y"][:, :, c], np.broadcast_to(pk[:, c], (nt, 4, c.sum())))


@pytest.mark.parametrize("mode", [S.MODE_SPECTRAL, S.MODE_LAGRANGE6, S.MODE_NUFFT])
def test_dense_output_c1_shape_with_own_grids(mode):
    # SW_zero_background_raytracing.m:70-78: RelTol 1e-6, AbsTol 1e-7, about 40 outputs, here each packet its own grid
    n, N = 40, 40
    rs = np.random.RandomState(4)
    ts = rs.uniform(0.0, 0.5, n)[None, :] + rs.uniform(0.03, 0.06, n)[None, :] * np.arange(N + 1)[:, None]
    pk = make_packets(n, seed=3)
    with engine(mode, 32, False) as e:
        st, yp = rows_solve(e, pk, ts, None, 1e-6, 1e-7)
        ref = one_packet_solves(e, pk, ts, None, 1e-6, 1e-7)
    assert st["Y"].shape == (N + 1, 4, n)
    assert np.array_equal(st["Y"][0], pk) and np.array_equal(st["Y"][-1], yp)
    assert_rows_equal_one_packet_solves(st, yp, ref, ts, True)
    for i in (0, 17, 39):                        # Y[j, :, i] is the one-packet dense row at ts[j, i]
        assert np.array_equal(st["Y"][:, :, i], ref[i][3])


@pytest.mark.parametrize("mode,nx", THREE)
@pytest.mark.parametrize("two", [False, True])
def test_shared_rows_equal_ode23_packets(mode, nx, two):
    pk = make_packets(200, seed=13)
    tspan = 0.04 * np.arange(11)
    tmax = 0.4 if two else None
    with engine(mode, nx, two) as e:
        a, ya = rows_solve(e, pk, np.repeat(tspan[:, None], 200, axis=1), tmax, 1e-6, 1e-7)
        b, yb = rows_solve(e, pk, tspan, tmax, 1e-6, 1e-7)
    for key in ("steps", "rejected", "status", "t_end"):
        assert np.array_equal(a[key], b[key]), key
    assert (a["nsteps"], a["nfailed"], a["nfevals"], a["stopped"]) == (b["nsteps"], b["nfailed"], b["nfevals"], b["stopped"])
    if mode == S.MODE_SPECTRAL and two:          # f1 from both frames' planes instead of the blended stack
        assert np.all(np.abs(ya - yb) <= 1e-12 * scale_of(yb)) and np.all(np.abs(a["Y"] - b["Y"]) <= 1e-12 * scale_of(yb)[None])
    else:
        assert np.array_equal(ya, yb) and np.array_equal(a["Y"], b["Y"])


@pytest.mark.parametrize("mode,nx", THREE)
def test_independence_and_a_packet_that_blows_up(mode, nx):
    n = 300
    pk = make_packets(n, seed=11)
    rs = np.random.RandomState(2)
    ts = np.sort(rs.uniform(0.0, 0.4, (11, n)), axis=0)
    ts[:, 1::2] = ts[::-1, 1::2]                 # every other packet backward
    perm = rs.permutation(n)
    with engine(mode, nx, True) as e:
        a, ya = rows_solve(e, pk, ts, 0.4, 1e-6, 1e-7)
        c, yc = rows_solve(e, pk[:, perm], ts[:, perm], 0.4, 1e-6, 1e-7)
        assert np.array_equal(yc, ya[:, perm]) and np.array_equal(c["Y"], a["Y"][:, :, perm])
        for key in ("steps", "rejected", "status", "t_end"):
            assert np.array_equal(c[key], a[key][perm]), key
        bad = pk.copy()
        bad[2, 17] = np.inf
        b, yb = rows_solve(e, bad, ts, 0.4, 1e-6, 1e-7)
        (_, _, _, _, t_fail, _), = one_packet_solves(e, bad[:, 17:18], ts[:, 17:18], 0.4, 1e-6, 1e-7)
    assert b["stopped"] == 1 and b["status"][17] == 1 and b["status"].sum() == 1
    assert t_fail is not None and b["t_end"][17] == t_fail
    assert np.array_equal(yb[:, 17], bad[:, 17]) and np.all(np.isnan(b["Y"][1:, :, 17]))
    good = np.delete(np.arange(n), 17)
    assert np.array_equal(yb[:, good], ya[:, good]) and np.array_equal(b["Y"][:, :, good], a["Y"][:, :, good])


@pytest.mark.parametrize("mode,nx", THREE)
def test_two_devices_equal_one_bit_for_bit(mode, nx):
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two GPUs")
    n = 3001
    pk = make_packets(n, seed=12)
    ts = np.sort(np.random.RandomState(5).uniform(0.0, 0.4, (3, n)), axis=0)
    ts[:, ::3] = ts[::-1, ::3]                   # every third packet backward
    res = []
    for ngpu in (1, 2):
        with engine(mode, nx, True, ngpu=ngpu) as e:
            res.append(rows_solve(e, pk, ts, 0.4, 1e-6, 1e-7))
    (a, ya), (b, yb) = res
    assert np.array_equal(ya, yb) and np.array_equal(a["Y"], b["Y"])
    for key in ("steps", "rejected", "status", "t_end"):
        assert np.array_equal(a[key], b[key]), key


def test_refusals_leave_the_packets_untouched():
    n = 10
    pk = make_packets(n)
    ok = np.stack([np.zeros(n), np.full(n, 0.2), np.full(n, 0.4)])
    with engine(S.MODE_LAGRANGE6, 32, True) as e:
        e.set_packets(*pk)
        nonfinite = ok.copy(); nonfinite[1, 3] = np.nan
        with pytest.raises(S.SwrtError, match=r"packet 3: tspan must be finite"):
            e.ode23_packets(nonfinite, 0.4)
        against = ok.copy(); against[:, 6] = [0.4, 0.1, 0.2]          # backward row whose entry 2 goes forward
        with pytest.raises(S.SwrtError, match=r"packet 6: tspan must be monotonic \(entry 2"):
            e.ode23_packets(against, 0.4)
        with pytest.raises(ValueError):
            e.ode23_packets(ok[:, :-1], 0.4)
        assert np.array_equal(np.stack(e.get_packets()), pk)
        st = e.ode23_packets(ok, 0.4)                                  # the handle still solves
    assert st["stopped"] == 0 and np.all(st["t_end"] == 0.4)


@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    from test_mex_gateway import Mex
    return Mex(request.param)


def test_gateway_matrix_tspan(mex):
    from test_mex_ode23 import _setup
    n = 301
    w, h, eng = _setup(mex, n, blow_up=True)
    rs = np.random.RandomState(9)
    ts = np.sort(rs.uniform(0.0, w.dt, (n, 5)), axis=1)                # MATLAB: row i is packet i's tspan
    ts[1::2] = ts[1::2, ::-1]
    st, Y, pstat, t_end = mex("ode23_packets", h, ts, w.dt, 1e-6, 1e-7, nlhs=4)
    ref = eng.ode23_packets(ts.T, w.dt, 1e-6, 1e-7)
    assert np.array_equal(np.ravel(st)[:4], [ref["nsteps"], ref["nfailed"], ref["nfevals"], ref["stopped"]]) and ref["stopped"] == 1
    assert np.array_equal(pstat, np.stack([ref["steps"], ref["rejected"], ref["status"]], axis=1))
    assert np.array_equal(np.ravel(t_end), ref["t_end"])
    assert np.array_equal(Y.reshape(n, 4, 5, order="F"), ref["Y"].transpose(2, 1, 0), equal_nan=True)
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()), equal_nan=True)
    with pytest.raises(Exception, match="n x m"):
        mex("ode23_packets", h, ts[:-1], w.dt, 1e-6, 1e-7)
    mex("destroy", h, nlhs=0); eng.close()
