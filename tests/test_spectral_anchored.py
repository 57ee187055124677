"""The anchored SPECTRAL leapfrog (psi-hat flows at nx = 256 and 512, DESIGN.md section 3e): the stack is contracted once
per occupied anchor cell (K1) and each packet gets its field from a degree-7 Taylor expansion around its anchor (K2).

* one step, and 16 two-frame sub-steps, against the C oracle's direct Fourier sums, including packets exactly on
  anchor-cell edges, at x = +-L/2, at t just below one period and all packets in one cell;
* per-packet determinism, which sharding and staging rely on: a shuffled ensemble, unequal shards and a padded
  ensemble give the same doubles as the full run, fused sub-steps equal single steps, step_host equals
  set + step + get.
"""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
from oracle import c_oracle as CO

pytestmark = pytest.mark.gpu

NX = [256, 512]


def _engine(w):
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL, device=0)
    eng.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
    if w.psik2 is not None:
        eng.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
    return eng


def _edge_packets(w, nx):
    """packets with k = l = 0 (no half drift, so they are keyed exactly where they are placed): on anchor-cell edges,
    at x = +-L/2, one ulp below a period, just below zero"""
    m = 15 if nx == 512 else 14
    cells = np.array([0, 1, 2, 777, 2 ** (m - 1), 2 ** m - 1])
    x = np.concatenate([cells * 2.0 ** -m * w.L, [w.L / 2, -w.L / 2, np.nextafter(w.L, 0.0), -5e-324, np.nextafter(0.0, 1.0)]])
    y = np.linspace(-w.L / 2, w.L / 2, x.size)
    return x, y, np.zeros_like(x), np.zeros_like(x)


def _sample(w, nx, nrand):
    xe, ye, ke, le = _edge_packets(w, nx)
    return (np.concatenate([w.x[:nrand], xe]), np.concatenate([w.y[:nrand], ye]),
            np.concatenate([w.k[:nrand], ke]), np.concatenate([w.l[:nrand], le]))


def _rel_increment_err(got, ref, start):
    d_got = np.stack(got) - np.stack(start)
    d_ref = np.stack(ref) - np.stack(start)
    scale = np.abs(d_ref).max(axis=1, keepdims=True)
    scale[scale == 0] = 1.0
    return float((np.abs(d_got - d_ref) / scale).max())


@pytest.mark.parametrize("nx", NX)
def test_one_step_against_oracle(nx):
    w = W.make_workload("C4", n_packets=4096, nx=nx)
    x, y, k, l = _sample(w, nx, 40)
    eng = _engine(w)
    eng.set_packets(x, y, k, l)
    eng.step(S.SCHEME_LEAPFROG, w.dt, 1)
    got = eng.get_packets()
    eng.close()
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean)
    ref = CO.leapfrog_spectral(x, y, k, l, planes, w.dx, w.nx, w.f, w.gH, w.dt, 1, precise=True)
    err = _rel_increment_err(got, ref, (x, y, k, l))
    assert err < 1e-12, f"one anchored step vs the oracle: {err:.3e}"


@pytest.mark.parametrize("nx", NX)
def test_two_frame_substeps_against_oracle(nx):
    w = W.make_workload("C4", n_packets=4096, nx=nx)
    x, y, k, l = _sample(w, nx, 16)
    m = 16
    a0, da = 0.5 / m, 1.0 / m
    eng = _engine(w)
    eng.set_packets(x, y, k, l)
    eng.step(S.SCHEME_LEAPFROG, w.dt / m, m, a0, da)
    got = eng.get_packets()
    eng.close()
    ref = (x, y, k, l)
    for j in range(m):
        al = a0 + j * da
        planes = W.planes_from_psik((1.0 - al) * w.psik + al * w.psik2, w.L, w.u_mean)
        ref = CO.leapfrog_spectral(*ref, planes, w.dx, w.nx, w.f, w.gH, w.dt / m, 1, precise=True)
    err = _rel_increment_err(got, ref, (x, y, k, l))
    assert err < 1e-9, f"16 anchored two-frame sub-steps vs the oracle: {err:.3e}"


def test_all_packets_in_one_anchor_and_a_single_packet():
    w = W.make_workload("C4", n_packets=64, nx=512)
    x = (12345.5 + np.linspace(-0.49, 0.49, 64)) * 2.0 ** -15 * w.L     # one cell of 2^-15 periods
    y = w.y[:64].copy()
    k = np.zeros(64); l = np.zeros(64)
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean)
    for sl in (slice(0, 64), slice(5, 6)):
        eng = _engine(w)
        eng.set_packets(x[sl], y[sl], k[sl], l[sl])
        eng.step(S.SCHEME_LEAPFROG, w.dt, 1)
        got = eng.get_packets()
        eng.close()
        ref = CO.leapfrog_spectral(x[sl], y[sl], k[sl], l[sl], planes, w.dx, w.nx, w.f, w.gH, w.dt, 1, precise=True)
        assert _rel_increment_err(got, ref, (x[sl], y[sl], k[sl], l[sl])) < 1e-12


def _run(w, x, y, k, l, m, single=False):
    eng = _engine(w)
    eng.set_packets(x, y, k, l)
    a0, da = 0.5 / m, 1.0 / m
    if single:
        for j in range(m):
            eng.step(S.SCHEME_LEAPFROG, w.dt / m, 1, a0 + j * da, 0.0)
    else:
        eng.step(S.SCHEME_LEAPFROG, w.dt / m, m, a0, da)
    out = np.stack(eng.get_packets())
    eng.close()
    return out


@pytest.mark.parametrize("nx", NX)
def test_shuffle_shards_and_padding_are_bit_identical(nx):
    w = W.make_workload("C4", n_packets=70001, nx=nx)
    m = 2
    full = _run(w, w.x, w.y, w.k, w.l, m)
    assert np.isfinite(full).all()
    perm = np.random.default_rng(7).permutation(w.n_packets)
    shuf = _run(w, w.x[perm], w.y[perm], w.k[perm], w.l[perm], m)
    assert np.array_equal(shuf, full[:, perm])
    cut = 23456
    a = _run(w, w.x[:cut], w.y[:cut], w.k[:cut], w.l[:cut], m)
    b = _run(w, w.x[cut:], w.y[cut:], w.k[cut:], w.l[cut:], m)
    assert np.array_equal(np.concatenate([a, b], axis=1), full)
    z = np.zeros(37)
    pad = _run(w, np.concatenate([z, w.x]), np.concatenate([z, w.y]), np.concatenate([z + 1.0, w.k]), np.concatenate([z, w.l]), m)
    assert np.array_equal(pad[:, 37:], full)


def test_fused_substeps_equal_single_steps():
    w = W.make_workload("C4", n_packets=20000, nx=512)
    assert np.array_equal(_run(w, w.x, w.y, w.k, w.l, 3), _run(w, w.x, w.y, w.k, w.l, 3, single=True))


@pytest.mark.parametrize("n", [1, 300007, 800003])
def test_step_host_equals_set_step_get(n):
    w = W.make_workload("C3", n_packets=n, nx=256)
    m = 2
    a0, da = 0.5 / m, 1.0 / m
    eng = _engine(w)
    eng.set_packets(w.x, w.y, w.k, w.l)
    eng.step(S.SCHEME_LEAPFROG, w.dt / m, m, a0, da)
    ref = np.stack(eng.get_packets())
    got = np.stack(eng.step_host(S.SCHEME_LEAPFROG, w.dt / m, m, w.x, w.y, w.k, w.l, alpha0=a0, dalpha=da))
    eng.close()
    assert np.array_equal(got, ref)
