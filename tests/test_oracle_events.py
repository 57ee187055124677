"""ode23_events_oracle: the restated event semantics of swrt_ode23_packets_events (detection after each accepted step,
Illinois regula falsi on the step's ntrp23 cubic, the terminal rule), checked against known answers on a zero flow and
against scipy's independent RK23 event location on the Childress-Soward flow; its controller is oracle.ode23's, bit for
bit."""
import math

import numpy as np
import pytest

import ode23_events_oracle as E
from oracle import swrt_oracle as O

F0, CG = 3.0, 1.0


def zero_flow(calls=None):
    def odefun(t, y):
        if calls is not None:
            calls.append((t, y.copy()))
        return np.concatenate(O.rhs_from_eval(np.zeros((6, 1)), y[2:3], y[3:4], F0, CG))
    return odefun


def solve(y0, events, tspan=(0.0, 2.0), odefun=None, **kw):
    _, st = E.ode23(odefun or zero_flow(), list(tspan), np.array(y0, dtype=np.float64), events=events, f=F0, gH=CG * CG, **kw)
    return st


def test_zero_flow_x_crossing_is_analytic():
    y0 = [0.1, -0.4, 2.0, 1.0]
    xdot = CG * y0[2] / math.sqrt(F0 ** 2 + CG ** 2 * (y0[2] ** 2 + y0[3] ** 2))
    levels = [0.2, 0.55, 0.9]
    st = solve(y0, [(E.EVENT_X, c, 0, 0) for c in levels])
    assert np.array_equal(st["ie"], [1, 2, 3]) and st["status"] == 0 and st["nsteps"] >= 10
    te = np.array([(c - y0[0]) / xdot for c in levels])
    assert np.all(np.abs(st["te"] - te) <= 1e-13 * te)
    assert np.all(np.abs(st["ye"][:, 0] - levels) <= 1e-13) and np.array_equal(st["ye"][:, 2:], np.tile(y0[2:], (3, 1)))


def test_zero_flow_kmag_and_omega_never_fire():
    y0 = [0.1, -0.4, 2.0, 1.0]
    K = math.hypot(2.0, 1.0)
    w = math.sqrt(F0 ** 2 + CG ** 2 * K ** 2)
    ev = [(E.EVENT_KMAG, K, 0, 0), (E.EVENT_KMAG, K - 0.1, 0, 0), (E.EVENT_OMEGA, w + 0.1, 0, 0), (E.EVENT_OMEGA, w, 0, 1)]
    st = solve(y0, ev)
    assert st["te"].size == 0 and st["status"] == 0 and st["t"] == 2.0


@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_directions_filter(sign):
    y0 = [0.0, 0.0, sign * 2.0, 0.5]                    # x rises (sign +1) or falls (sign -1) through +-0.3
    lvl = sign * 0.3
    ev = [(E.EVENT_X, lvl, 0, 0), (E.EVENT_X, lvl, 1, 0), (E.EVENT_X, lvl, -1, 0)]
    st = solve(y0, ev)
    assert np.array_equal(st["ie"], [1, 2] if sign > 0 else [1, 3])
    assert st["te"][0] == st["te"][1]


def test_zero_at_t0_not_reported_and_step_end_reported_once():
    y0 = [0.25, -0.4, 2.0, 1.0]
    calls = []
    ref = solve(y0, [(E.EVENT_X, 1.0, 0, 0)], odefun=zero_flow(calls))
    # calls: f1, then (f2, f3, f4) per attempt; no rejections on a zero flow, so calls[3 * m] holds the m-th step end
    assert ref["nfailed"] == 0 and len(calls) == 1 + 3 * ref["nsteps"]
    t3, y3 = calls[9]
    st = solve(y0, [(E.EVENT_X, y0[0], 0, 0), (E.EVENT_X, float(y3[0]), 0, 0), (E.EVENT_Y, y0[1], 0, 0)])
    assert np.array_equal(st["ie"], [2]) and st["te"][0] == t3 and np.array_equal(st["ye"][0], y3)
    assert st["nsteps"] == ref["nsteps"]                  # events never change a step decision


def test_terminal_event_stops_the_solve():
    y0 = [0.1, -0.4, 2.0, 1.0]
    tspan = np.linspace(0.0, 2.0, 21)
    free, _ = E.ode23(zero_flow(), tspan, np.array(y0))
    Y, st = E.ode23(zero_flow(), tspan, np.array(y0), events=[(E.EVENT_X, 0.9, 0, 0), (E.EVENT_X, 0.5, 0, 1), (E.EVENT_Y, -0.2, 0, 0)],
                    f=F0, gH=CG * CG)
    assert np.array_equal(st["ie"], [2]) and st["status"] == 2 and st["t"] == st["te"][0]
    reached = tspan <= st["te"][0]
    assert np.array_equal(Y[reached], free[reached]) and np.isnan(Y[~reached]).all()


def cs_odefun(U0=1.0, km=1.0, a=0.5):
    def odefun(t, y):
        e6 = O.childress_soward_point(y[0:1], y[1:2], U0, km, a)
        return np.concatenate(O.rhs_from_eval(e6, y[2:3], y[3:4], F0, CG))
    return odefun


def test_against_scipy_rk23_events_on_childress_soward():
    from scipy.integrate import solve_ivp
    y0 = np.array([0.3, 0.7, 2.0, -1.0])
    ev = [(E.EVENT_X, 0.6, 0, 0), (E.EVENT_Y, 0.9, -1, 0), (E.EVENT_K, 0.0, 0, 0), (E.EVENT_L, 0.5, 1, 0),
          (E.EVENT_KMAG, 2.5, 0, 0), (E.EVENT_OMEGA, 3.9, 0, 0)]
    T = 6.0
    odefun = cs_odefun()
    st = solve(y0, ev, (0.0, T), odefun=odefun, rtol=1e-10, atol=1e-10)
    fns = []
    for kind, level, direction, _ in ev:
        def g(t, y, kind=kind, level=level):
            return E.event_g(kind, level, y, F0, CG * CG)
        g.direction = direction
        fns.append(g)
    sol = solve_ivp(lambda t, y: odefun(t, y), (0.0, T), y0, method="RK23", events=fns, rtol=1e-10, atol=1e-10)
    ref = sorted((float(t), j + 1) for j, ts in enumerate(sol.t_events) for t in ts)
    assert len(ref) >= 6 and len({j for _, j in ref}) >= 4
    assert np.array_equal(st["ie"], [j for _, j in ref])
    assert np.all(np.abs(st["te"] - [t for t, _ in ref]) <= 1e-6)
    for j, ye in zip(st["ie"], st["ye"]):
        kind, level, _, _ = ev[j - 1]
        assert abs(E.event_g(kind, level, ye, F0, CG * CG)) <= 1e-6

    # a terminal |k| level stops both at the same time
    st2 = solve(y0, [(E.EVENT_KMAG, 2.5, 0, 1)], (0.0, T), odefun=odefun, rtol=1e-10, atol=1e-10)
    fns[4].terminal = True
    sol2 = solve_ivp(lambda t, y: odefun(t, y), (0.0, T), y0, method="RK23", events=fns[4], rtol=1e-10, atol=1e-10)
    assert st2["status"] == 2 and sol2.status == 1 and abs(st2["t"] - sol2.t[-1]) <= 1e-6


@pytest.mark.parametrize("tspan", [(0.0, 3.0), tuple(np.linspace(0.0, 3.0, 13))])
@pytest.mark.parametrize("rtol,atol", [(1e-3, 1e-6), (1e-8, 1e-9)])
def test_controller_is_the_oracles_bit_for_bit(tspan, rtol, atol):
    y0 = np.array([0.3, 0.7, 4.0, -3.0])
    odefun = cs_odefun(U0=3.0)
    ref, sref = O.ode23(odefun, list(tspan), y0, rtol, atol)
    quiet = [(E.EVENT_X, 50.0, 0, 1), (E.EVENT_OMEGA, 1.0, 0, 0)]        # never reached: no record, no stop
    for events in ((), quiet):
        got, st = E.ode23(odefun, list(tspan), y0, rtol, atol, events=events, f=F0, gH=CG * CG)
        assert np.array_equal(got, ref) and st["te"].size == 0 and st["status"] == 0
        assert all(st[k] == sref[k] for k in ("nsteps", "nfailed", "nfevals", "t"))
    assert sref["nfailed"] > 0 or rtol < 1e-6
