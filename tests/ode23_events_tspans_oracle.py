"""The oracle of swrt_ode23_packets_tspans_events: MATLAB's ``ode23`` with ``odeset('Events', ...)`` for one packet with
a tspan of either direction, restated operation for operation in the device's order (DESIGN.md section 11).

``ode23`` below is ode23_backward_oracle.ode23's controller (oracle.swrt_oracle.ode23 with ``tdir``) with
ode23_events_oracle.ode23's detection, and a locator, record order and terminal rule that follow the direction of
integration:
* detection is unchanged: vL is g_j at the previous accepted state, vR at ynew, and "rising" (vL < 0 <= vR) is rising
  along the integration, i.e. as t decreases backward;
* the crossing is located on [tL, tR] = [t, tnew] in integration order (tR < tL backward) by the Illinois regula falsi of
  ode23_events_oracle.event_locate applied to ``tdir*t``: the bracket test is ``tdir*(tR - tL) > tol`` and tm is clamped
  half inside both ends, so t -> -t gives te bit for bit up to sign;
* records come in order of encounter (ascending ``tdir*te``, then the event index);
* a terminal event stops the solve at the first terminal te* in integration order; records and dense rows beyond it
  (``tdir*(t - te*) > 0``) are dropped / stay NaN.
Forward (``tdir = +1``) every operation is ode23_events_oracle.ode23's; without events every operation is
ode23_backward_oracle.ode23's.  tests/test_oracle_events_tspans.py checks both bit for bit."""
import numpy as np

from ode23_events_oracle import event_g, ntrp23_at


def event_locate(g, t, tnew, vL, vR, tdir=1.0):
    """te of a sign change of g(tau) on the step's interpolant between g(t) = vL and g(tnew) = vR, t and tnew in
    integration order: ode23_events_oracle.event_locate on tdir*t (the device's ev_locate)"""
    if vR == 0.0:
        return tnew

    def key(v):                            # tdir*t, exact: the time in integration order and back
        return v if tdir > 0 else -v
    tL, tR, gL, gR = t, tnew, vL, vR
    tol = 128.0 * max(float(np.spacing(abs(tL))), float(np.spacing(abs(tR))))
    half = 0.5 * tol
    moved, it = 0, 0                       # moved: the end that moved last, -1 left, +1 right
    while it < 64 and key(tR) - key(tL) > tol:
        tm = tR - gR * ((tR - tL) / (gR - gL))
        tm = key(min(max(key(tm), key(tL) + half), key(tR) - half))
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
    """ode23 in either direction of time on one packet y0 = (x, y, k, l) with ``events``, a list of (kind, level,
    direction, terminal); ``f``, ``gH`` for EVENT_OMEGA.  Returns (y_final or Y, stats) as ode23_events_oracle.ode23 does
    (``te``, ``ye``, ``ie``, ``status``, ``t``), and ``h``, the accepted steps (signed), as ode23_backward_oracle.ode23
    does.  Raises ValueError on a tspan entry against the direction, RuntimeError where the step size falls below hmin."""
    tspan = np.asarray(tspan, dtype=np.float64)
    t0, tfinal = float(tspan[0]), float(tspan[-1])
    tdir = 1.0 if tfinal >= t0 else -1.0
    if np.any(tdir * np.diff(tspan) < 0):
        raise ValueError("ode23: tspan must be monotonic")
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
    hs = []
    done = False
    while not done:
        hmin = 16 * np.spacing(abs(t))
        absh = min(hmax, max(hmin, absh))
        h = tdir * absh
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
                h = tdir * absh; done = False
            else:
                break
        nsteps += 1
        hs.append(h)

        def at(tau):
            return ntrp23_at(y, f1, f2, f3, f4, ynew, t, h, tnew, tau)
        fired = []
        for j, (kind, level, direction, terminal) in enumerate(events):
            vL, vR = vl[j], event_g(kind, level, ynew, f, gH)
            vl[j] = vR
            if (vL < 0.0 and vR >= 0.0 and direction >= 0) or (vL > 0.0 and vR <= 0.0 and direction <= 0):
                te = event_locate(lambda tau: event_g(kind, level, at(tau), f, gH), t, tnew, vL, vR, tdir)
                fired.append((te, j))
                if terminal and (tstop is None or tdir * te < tdir * tstop):
                    tstop = te
        for te, j in sorted(fired, key=lambda r: (tdir * r[0], r[1])):
            if tstop is None or tdir * te <= tdir * tstop:
                records.append((te, at(te), j + 1))
        ystop = None if tstop is None else at(tstop)
        if dense:
            while nxt < tspan.size and tdir * (tnew - tspan[nxt]) >= 0 and (tstop is None or tdir * tspan[nxt] <= tdir * tstop):
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
    stats = {"nsteps": nsteps, "nfailed": nfailed, "nfevals": nfevals, "t": t, "h": np.array(hs),
             "te": np.array([r[0] for r in records]), "ye": np.array([r[1] for r in records]).reshape(-1, y.size),
             "ie": np.array([r[2] for r in records], dtype=np.int64), "status": 2 if tstop is not None else 0}
    return (Y, stats) if dense else (y, stats)
