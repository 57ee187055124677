"""ode23_events_tspans_oracle: events in either direction of integration, on the CPU.  Forward it is
ode23_events_oracle bit for bit, without events it is ode23_backward_oracle bit for bit in both directions, a backward
solve is the mirror image of a forward one bit for bit (events, records and terminal stops included), and on a zero flow
the backward crossings are the analytic ones."""
import math

import numpy as np
import pytest

import ode23_backward_oracle as B
import ode23_events_oracle as E
import ode23_events_tspans_oracle as ET
from test_oracle_backward import cs_odefun, mirror
from test_oracle_events import F0, CG, zero_flow

Y0 = np.array([1.3, 4.1, 2.4, -1.1])
# X, Y, |k| and omega keep their values under the mirror (x, y, k, l) -> (x, y, -k, -l); K and L flip sign, so their
# level and direction are negated with them
EVENTS = [(E.EVENT_X, 1.9, 0, 0), (E.EVENT_Y, 3.8, 1, 0), (E.EVENT_KMAG, 2.5, 0, 0), (E.EVENT_OMEGA, 3.9, -1, 0),
          (E.EVENT_K, 2.0, 1, 0), (E.EVENT_L, -1.0, 0, 0)]


def mirrored(events):
    return [(kind, -level, -d, term) if kind in (E.EVENT_K, E.EVENT_L) else (kind, level, d, term)
            for kind, level, d, term in events]


def solve(oracle, f, tspan, y0, events, rtol=1e-3, atol=1e-6):
    return oracle.ode23(f, np.asarray(tspan, dtype=np.float64), y0, rtol, atol, events=events, f=F0, gH=CG * CG)


def same_records(a, b):
    return (np.array_equal(a["te"], b["te"]) and np.array_equal(a["ye"], b["ye"]) and np.array_equal(a["ie"], b["ie"])
            and all(a[k] == b[k] for k in ("nsteps", "nfailed", "nfevals", "t", "status")))


@pytest.mark.parametrize("tspan", [[0.0, 3.0], np.linspace(0.0, 3.0, 31)])
@pytest.mark.parametrize("terminal", [False, True])
def test_forward_is_the_events_oracle_bit_for_bit(tspan, terminal):
    ev = EVENTS + ([(E.EVENT_X, 2.2, 0, 1)] if terminal else [])
    f = cs_odefun(1, 2.0)
    a, sa = solve(E, f, tspan, Y0, ev)
    b, sb = solve(ET, f, tspan, Y0, ev)
    assert sa["te"].size >= 3 and sa["status"] == (2 if terminal else 0)
    assert np.array_equal(a, b, equal_nan=True) and same_records(sa, sb)


@pytest.mark.parametrize("tspan", [[0.0, 3.0], np.linspace(0.0, 3.0, 31), [3.0, 0.0], np.linspace(3.0, 0.0, 31)])
@pytest.mark.parametrize("rtol", [1e-3, 1e-6])
def test_without_events_it_is_the_backward_oracle_bit_for_bit(tspan, rtol):
    f = cs_odefun(1, 2.0)
    a, sa = B.ode23(f, tspan, Y0, rtol, rtol * 1e-3)
    b, sb = ET.ode23(f, tspan, Y0, rtol, rtol * 1e-3)
    assert np.array_equal(a, b) and np.array_equal(sa["h"], sb["h"])
    assert all(sa[k] == sb[k] for k in ("nsteps", "nfailed", "nfevals", "t")) and sb["te"].size == 0


@pytest.mark.parametrize("dense", [False, True])
@pytest.mark.parametrize("terminal", [None, 2, 5])
def test_backward_is_the_mirror_of_forward_bit_for_bit(dense, terminal):
    """backward over [T .. 0] in the flow U0 == forward over [-T .. 0] in -U0 with (k, l) negated, rejections forced:
    te negated, ye mirrored, ie and the counts equal"""
    T = 3.0
    ts = np.linspace(T, 0.0, 31) if dense else np.array([T, 0.0])
    ev = [e[:3] + (int(j == terminal),) for j, e in enumerate(EVENTS)]
    for U0 in (3.0, 10.0, 30.0):
        Yb, sb = solve(ET, cs_odefun(1, U0), ts, Y0, ev)
        if sb["nfailed"] > 0 and sb["te"].size >= (2 if terminal else 3):
            break
    assert sb["nfailed"] > 0 and sb["te"].size >= (2 if terminal else 3) and np.all(np.diff(sb["te"]) <= 0)
    Yf, sf = solve(E, cs_odefun(1, -U0), -ts, mirror(Y0, 1), mirrored(ev))
    assert (sb["nsteps"], sb["nfailed"], sb["nfevals"], sb["status"]) == (sf["nsteps"], sf["nfailed"], sf["nfevals"], sf["status"])
    assert sb["status"] == (0 if terminal is None else 2)
    assert np.array_equal(sb["te"], -sf["te"]) and np.array_equal(sb["ie"], sf["ie"]) and sb["t"] == -sf["t"]
    assert np.array_equal(sb["ye"], mirror(sf["ye"], 1))
    assert np.array_equal(Yb, mirror(Yf, 1), equal_nan=True)
    # and the backward oracle's forward mirror is the same solve as this one's
    Yf2, sf2 = solve(ET, cs_odefun(1, -U0), -ts, mirror(Y0, 1), mirrored(ev))
    assert np.array_equal(Yf, Yf2, equal_nan=True) and same_records(sf, sf2)


def test_zero_flow_backward_x_crossings_are_analytic():
    y0 = [0.9, -0.4, 2.0, 1.0]                    # x' > 0: going back from T, x falls through the levels
    xdot = CG * y0[2] / math.sqrt(F0 ** 2 + CG ** 2 * (y0[2] ** 2 + y0[3] ** 2))
    T = 2.0
    ev = [(E.EVENT_X, c, 0, 0) for c in (0.2, 0.8, 0.55)] + [(E.EVENT_X, 0.7, 1, 0), (E.EVENT_X, 0.3, -1, 0)]
    _, st = solve(ET, zero_flow(), [T, 0.0], np.array(y0), ev)
    # every crossing falls in integration order (g decreases as t decreases): the rising-only event never fires
    assert np.array_equal(st["ie"], [2, 3, 5, 1]) and st["status"] == 0 and st["nsteps"] >= 10
    te = np.array([T + (c - y0[0]) / xdot for c in (0.8, 0.55, 0.3, 0.2)])
    assert np.all(np.abs(st["te"] - te) <= 1e-13 * T)
    assert np.all(np.abs(st["ye"][:, 0] - [0.8, 0.55, 0.3, 0.2]) <= 1e-13)
    assert np.array_equal(st["ye"][:, 2:], np.tile(y0[2:], (4, 1)))


def test_zero_flow_backward_terminal_stop():
    y0 = [0.9, -0.4, 2.0, 1.0]
    xdot = CG * y0[2] / math.sqrt(F0 ** 2 + CG ** 2 * (y0[2] ** 2 + y0[3] ** 2))
    T = 2.0
    ts = np.linspace(T, 0.0, 21)
    ev = [(E.EVENT_X, 0.2, 0, 0), (E.EVENT_X, 0.5, 0, 1), (E.EVENT_X, 0.6, 0, 1)]
    Y, st = solve(ET, zero_flow(), ts, np.array(y0), ev)
    tstar = T + (0.6 - y0[0]) / xdot                 # the first terminal crossing met going back
    assert st["status"] == 2 and np.array_equal(st["ie"], [3]) and st["t"] == st["te"][-1]
    assert abs(st["t"] - tstar) <= 1e-13 * T
    beyond = ts < st["t"]
    assert np.all(np.isnan(Y[beyond])) and np.all(np.isfinite(Y[~beyond]))
    Yn, _ = solve(ET, zero_flow(), ts, np.array(y0), [])
    assert np.array_equal(Y[~beyond], Yn[~beyond])


def test_zero_length_row_finds_nothing_and_keeps_its_state():
    y0 = np.array([0.9, -0.4, 2.0, 1.0])
    ev = [(E.EVENT_X, 0.9 + 1e-9, 0, 1), (E.EVENT_X, 0.0, 0, 0)]
    y, st = solve(ET, zero_flow(), [1.5, 1.5], y0, ev)
    assert np.array_equal(y, y0) and st["nsteps"] == 1 and st["te"].size == 0 and st["t"] == 1.5


def test_a_row_against_its_direction_is_refused():
    with pytest.raises(ValueError):
        solve(ET, zero_flow(), [2.0, 2.5, 0.0], np.array(Y0), EVENTS)
