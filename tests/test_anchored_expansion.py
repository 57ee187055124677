"""CPU check of the anchored leapfrog's algebra with the kernels' arithmetic (DESIGN.md section 3e), in one dimension:
twiddles sincospi(kx * t_a) at the cell centre, weights (kx/kmax)^r by repeated products, the S/D swap for odd orders,
i^r / r! folded into H', z = pi * kmax * (t - t_a), G = sum_r z^r H'_r.  Against an extended-precision direct sum the
anchored route must be as accurate as the direct double-precision sum, and the anchor geometry must keep the truncation
bound below 2^-53."""
from math import factorial, pi

import numpy as np
import pytest

R = 8


def _cells(nx):
    kmax = nx // 2 - 1
    for m in range(8, 30):
        if (pi * kmax * 2.0 ** -m) ** R / factorial(R) <= 2.0 ** -53:
            return m


@pytest.mark.parametrize("nx,m", [(256, 14), (512, 15)])
def test_anchor_cells_meet_the_truncation_bound(nx, m):
    assert _cells(nx) == m


@pytest.mark.parametrize("nx", [256, 512])
def test_anchored_route_is_as_accurate_as_the_direct_sum(nx):
    rs = np.random.default_rng(1)
    kmax, ncol = nx // 2 - 1, 24
    kx = np.arange(0, kmax + 1)
    amp = 1.0 / np.maximum(kx, 1.0)[:, None] ** 2
    Cp = amp * (rs.standard_normal((kmax + 1, ncol)) + 1j * rs.standard_normal((kmax + 1, ncol)))
    Cm = amp * (rs.standard_normal((kmax + 1, ncol)) + 1j * rs.standard_normal((kmax + 1, ncol)))
    Cm[0] = 0.0
    S, D = Cp + Cm, Cp - Cm
    m = _cells(nx)
    h2 = 2.0 ** (1 - m)                              # cell width in the kernels' t in [0, 2) (theta = pi t)
    w = kx / float(kmax)
    wr = [np.ones_like(w)]
    for _ in range(1, R):
        wr.append(wr[-1] * w)
    scale = (np.abs(Cp) + np.abs(Cm)).sum(0)
    Cp_l, Cm_l, kx_l = Cp.astype(np.clongdouble), Cm.astype(np.clongdouble), kx.astype(np.longdouble)
    worst_a = worst_d = 0.0
    for t in rs.uniform(0.0, 2.0, 300):
        ia = np.floor(t / h2)
        ta = (ia + 0.5) * h2
        ca, sa = np.cos(np.pi * kx * ta)[:, None], np.sin(np.pi * kx * ta)[:, None]
        G = np.zeros(ncol, complex)
        z = pi * kmax * (t - ta)
        for r in range(R):
            P, Q = (S, D) if r % 2 == 0 else (D, S)
            Ht = (wr[r][:, None] * (P * ca + 1j * Q * sa)).sum(0)
            G += z ** r * ((1j) ** r / factorial(r) * Ht)
        tl = np.longdouble(t) * np.pi
        ref = (Cp_l * np.exp(1j * kx_l * tl)[:, None] + Cm_l * np.exp(-1j * kx_l * tl)[:, None]).sum(0)
        direct = (Cp * np.exp(1j * kx * np.pi * t)[:, None] + Cm * np.exp(-1j * kx * np.pi * t)[:, None]).sum(0)
        worst_a = max(worst_a, float((np.abs(G - ref) / scale).max()))
        worst_d = max(worst_d, float((np.abs(direct - ref) / scale).max()))
    assert worst_a < 2e-15 + 2 * worst_d, (worst_a, worst_d)
