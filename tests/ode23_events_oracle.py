"""The oracle of swrt_ode23_packets_events: MATLAB's ``ode23`` with ``odeset('Events', ...)`` for one packet, restated
operation for operation in the device's order (DESIGN.md section 11).

``ode23`` below is oracle.swrt_oracle.ode23's controller -- the same scalar operations in the same order, which
tests/test_oracle_events.py checks bit for bit against it -- with the event detection, location and terminal rule added
after each accepted step.  Event kinds are include/swrt.h's SWRT_EVENT_*."""
import math

import numpy as np

EVENT_X, EVENT_Y, EVENT_K, EVENT_L, EVENT_KMAG, EVENT_OMEGA = range(6)


def event_g(kind, level, v, f=0.0, gH=0.0):
    """g_j of an event at the state v = (x, y, k, l): a component, |k| or omega (load_data.m:33's expression), minus the
    level; every operation rounded on its own, as the device computes it."""
    kl = v[2] * v[2] + v[3] * v[3]
    g = v[kind] if kind <= EVENT_L else math.sqrt(kl) if kind == EVENT_KMAG else math.sqrt(f * f + gH * kl)
    return float(g) - level


def ntrp23_at(y, f1, f2, f3, f4, ynew, t, h, tnew, tau):
    """the accepted step's ntrp23 cubic at tau, formed as the device forms a dense row (s == 1 gives ynew itself)"""
    s = 1.0 if tau == tnew else (tau - t) / h
    if s == 1.0:
        return ynew.copy()
    s2 = s * s
    s3 = s2 * s
    w = (h * ((s - 4.0 / 3.0 * s2) + 5.0 / 9.0 * s3), h * (s2 - 2.0 / 3.0 * s3), h * (4.0 / 3.0 * s2 - 8.0 / 9.0 * s3), h * (-s2 + s3))
    return y + (((f1 * w[0] + f2 * w[1]) + f3 * w[2]) + f4 * w[3])


def event_locate(g, t, tnew, vL, vR):
    """te of a sign change of g(tau) (on the step's interpolant) between g(t) = vL and g(tnew) = vR: Illinois regula falsi,
    the operations of the device locator (ev_locate) in its order."""
    if vR == 0.0:
        return tnew
    tL, tR, gL, gR = t, tnew, vL, vR
    tol = 128.0 * max(float(np.spacing(abs(tL))), float(np.spacing(abs(tR))))
    half = 0.5 * tol
    moved, it = 0, 0                       # moved: the end that moved last, -1 left, +1 right
    while it < 64 and tR - tL > tol:
        tm = min(max(tR - gR * ((tR - tL) / (gR - gL)), tL + half), tR - half)
        gm = g(tm)
        if gm == 0.0:
            tR = tm
            break
        if (gm < 0.0) == (gL < 0.0):       # the sign changes across [tm, tR]
            tL, gL = tm, gm
            if moved < 0:
                gR = 0.5 * gR
            moved = -1
        else:
            tR, gR = tm, gm
            if moved > 0:
                gL = 0.5 * gL
            moved = 1
        it += 1
    return tR


def ode23(odefun, tspan, y0, rtol=1e-3, atol=1e-6, events=(), f=0.0, gH=0.0):
    """oracle.swrt_oracle.ode23 on one packet y0 = (x, y, k, l) with ``events``, a list of (kind, level, direction,
    terminal); ``f``, ``gH`` for EVENT_OMEGA.  After each accepted step event j fires when g_j at the previous accepted
    state is non-zero, neither value is NaN, the sign changes and the direction allows it (+1 rising, -1 falling, 0 both);
    it is located by ``event_locate`` on the step's cubic.  A step's records are kept in (te, j) order; a terminal one
    stops the solve at the earliest terminal te (later records dropped, the state that record's ye, dense rows after it
    NaN).  Returns (y_final or Y, stats) as oracle.swrt_oracle.ode23 does; stats also hold ``te``, ``ye`` (m, 4), ``ie``
    (1-based), ``status`` (2 after a terminal event, else 0) and ``t`` (where the solve ended).  Raises where the step
    size falls below hmin, as the oracle does."""
    tspan = np.asarray(tspan, dtype=np.float64)
    t0, tfinal = float(tspan[0]), float(tspan[-1])
    dense = tspan.size > 2
    y = np.array(y0, dtype=np.float64)
    if dense:
        Y = np.full((tspan.size, y.size), np.nan); Y[0] = y; nxt = 1
    vl = [event_g(kind, level, y, f, gH) for kind, level, _, _ in events]
    records = []
    tstop = None
    pw = 1.0 / 3.0
    threshold = atol / rtol
    hmax = min(abs(tfinal - t0), abs(0.1 * (tfinal - t0)))
    t = t0
    f1 = odefun(t, y)
    nfevals = 1
    hmin = 16 * np.spacing(abs(t))
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
            ynew = y + (f1 * (h * (2.0 / 9.0)) + f2 * (h * (1.0 / 3.0)) + f3 * (h * (4.0 / 9.0)))
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

        def at(tau):
            return ntrp23_at(y, f1, f2, f3, f4, ynew, t, h, tnew, tau)
        fired = []
        for j, (kind, level, direction, terminal) in enumerate(events):
            vL, vR = vl[j], event_g(kind, level, ynew, f, gH)
            vl[j] = vR
            if (vL < 0.0 and vR >= 0.0 and direction >= 0) or (vL > 0.0 and vR <= 0.0 and direction <= 0):
                te = event_locate(lambda tau: event_g(kind, level, at(tau), f, gH), t, tnew, vL, vR)
                fired.append((te, j))
                if terminal and (tstop is None or te < tstop):
                    tstop = te
        for te, j in sorted(fired):
            if tstop is None or te <= tstop:
                records.append((te, at(te), j + 1))
        ystop = None if tstop is None else at(tstop)
        if dense:
            while nxt < tspan.size and tnew - tspan[nxt] >= 0 and (tstop is None or tspan[nxt] <= tstop):
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
        if tstop is not None:
            t, y = tstop, ystop
            break
    stats = {"nsteps": nsteps, "nfailed": nfailed, "nfevals": nfevals, "t": t,
             "te": np.array([r[0] for r in records]), "ye": np.array([r[1] for r in records]).reshape(-1, y.size),
             "ie": np.array([r[2] for r in records], dtype=np.int64), "status": 2 if tstop is not None else 0}
    return (Y, stats) if dense else (y, stats)
