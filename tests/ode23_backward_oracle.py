"""The oracle of ode23 with a decreasing tspan: MATLAB's direction rules (Shampine & Reichelt; ``odearguments`` / ``ode23``)
added to oracle.swrt_oracle.ode23's controller.

``ode23`` below is oracle.swrt_oracle.ode23 -- the same scalar operations in the same order, which
tests/test_oracle_backward.py checks bit for bit against it on forward solves -- with ``tdir``:
* ``tdir = +1`` when ``tfinal >= t0``, else ``-1``; every step is ``h = tdir*absh`` (the first attempt, the steps after an
  accept and the retries after a reject); the last step stays ``h = tfinal - t``;
* ``hmax``, ``htspan``, ``hmin``, the 1.1 stretch, the error norm and the rejection and growth rules act on ``absh`` and are
  unchanged;
* dense row j is written once ``tdir*(tnew - tspan[j]) >= 0``, with ``s = (tspan[j] - t)/h`` (positive for either sign);
* a ``tspan`` entry that steps against the direction raises ``ValueError`` (equal neighbours are allowed).
For ``tdir = +1`` every operation is oracle.swrt_oracle.ode23's (multiplying by 1.0 is exact)."""
import numpy as np


def ode23(odefun, tspan, y0, rtol=1e-3, atol=1e-6):
    """oracle.swrt_oracle.ode23 in either direction of time: returns (y_final or Y, stats); stats also hold ``h``, the
    accepted steps (signed)."""
    tspan = np.asarray(tspan, dtype=np.float64)
    t0, tfinal = float(tspan[0]), float(tspan[-1])
    tdir = 1.0 if tfinal >= t0 else -1.0
    if np.any(tdir * np.diff(tspan) < 0):
        raise ValueError("ode23: tspan must be monotonic")
    dense = tspan.size > 2
    y = np.array(y0, dtype=np.float64)
    if dense:
        Y = np.zeros((tspan.size, y.size)); Y[0] = y; nxt = 1
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
        if dense:
            while nxt < tspan.size and tdir * (tnew - tspan[nxt]) >= 0:
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
    stats = {"nsteps": nsteps, "nfailed": nfailed, "nfevals": nfevals, "t": t, "h": np.array(hs)}
    return (Y, stats) if dense else (y, stats)
