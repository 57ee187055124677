"""ode23 backward in time (a decreasing tspan, MATLAB's ``ode23(odefun, [T 0], y0)``) on the CPU: the backward oracle
(ode23_backward_oracle.ode23) against analytic solutions and its own mirror image, and the host controller
(reference_api.ode23, which also serves ShardedEnsemble.ode23) against the oracle on a numpy stand-in for the device."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

import ode23_backward_oracle as B
from oracle import swrt_oracle as O
from oracle import c_oracle as CO
from swraytracing_b200 import reference_api as R
from swraytracing_b200 import workloads as W
from swraytracing_b200.distributed import ShardedEnsemble

ROOT = Path(__file__).resolve().parent.parent
F0, CG = 3.0, 1.0


def cs_odefun(n, U0, km=1.0, a=0.3):
    """the ray RHS on y = [x; y; k; l] of n packets in the closed-form Childress-Soward flow of amplitude U0: every term is
    a product with U0 or with (k, l), so negating U0 and (k, l) negates the x-part and keeps the k-part, bit for bit"""
    def f(t, y):
        x, yy, k, l = y[:n], y[n:2 * n], y[2 * n:3 * n], y[3 * n:]
        return np.concatenate(O.rhs_from_eval(O.childress_soward_point(x, yy, U0, km, a), k, l, F0, CG))
    return f


def packets(n, seed=4):
    rs = np.random.RandomState(seed)
    i = np.arange(n)
    return np.concatenate([rs.uniform(0, 2 * np.pi, n), rs.uniform(0, 2 * np.pi, n), 3 * np.cos(0.7 * i), 3 * np.sin(0.7 * i)])


def mirror(y, n):
    """(x, y, k, l) -> (x, y, -k, -l)"""
    z = y.copy()
    z[..., 2 * n:] = -z[..., 2 * n:]
    return z


@pytest.mark.parametrize("tspan", [[0.0, 2.0], np.linspace(0.0, 3.0, 31)])
@pytest.mark.parametrize("rtol", [1e-3, 1e-6])
def test_forward_is_the_oracle_bit_for_bit(tspan, rtol):
    n = 8
    f = cs_odefun(n, 2.0)
    a, sa = O.ode23(f, tspan, packets(n), rtol, rtol * 1e-3)
    b, sb = B.ode23(f, tspan, packets(n), rtol, rtol * 1e-3)
    assert np.array_equal(a, b)
    assert all(sa[k] == sb[k] for k in ("nsteps", "nfailed", "nfevals", "t")) and np.all(sb["h"] > 0)


@pytest.mark.parametrize("rtol", [1e-3, 1e-6])
def test_exponential_decay_backward(rtol):
    # y' = -y from y(T) = 1: y(t) = exp(T - t).  ode23's global error is a small multiple of rtol per unit of growth
    T = 2.0
    y, st = B.ode23(lambda t, y: -y, [T, 0.0], np.array([1.0]), rtol, rtol * 1e-3)
    assert st["t"] == 0.0 and np.all(st["h"] < 0) and st["h"].sum() == pytest.approx(-T, abs=1e-13)
    assert abs(y[0] - np.exp(T)) <= 10 * rtol * np.exp(T)
    ts = np.linspace(T, 0.0, 41)
    Y, sd = B.ode23(lambda t, y: -y, ts, np.array([1.0]), rtol, rtol * 1e-3)
    assert Y[0, 0] == 1.0 and np.all(np.abs(Y[:, 0] - np.exp(T - ts)) <= 10 * rtol * np.exp(T - ts))


@pytest.mark.parametrize("rtol", [1e-3, 1e-6])
def test_harmonic_oscillator_backward(rtol):
    # y = (cos t, -sin t) solves y1' = y2, y2' = -y1; start from its value at T and integrate to 0
    T = 3.0
    f = lambda t, y: np.array([y[1], -y[0]])
    y0 = np.array([np.cos(T), -np.sin(T)])
    y, st = B.ode23(f, [T, 0.0], y0, rtol, rtol * 1e-3)
    assert st["t"] == 0.0 and st["nsteps"] >= 10
    assert np.abs(y - [1.0, 0.0]).max() <= 10 * rtol
    ts = np.linspace(T, 0.0, 61)
    Y, _ = B.ode23(f, ts, y0, rtol, rtol * 1e-3)
    assert np.abs(Y - np.stack([np.cos(ts), -np.sin(ts)], axis=1)).max() <= 10 * rtol


def test_oracle_mirror_identity_with_rejections():
    """backward over [T .. 0] in the flow U0 == forward over [-T .. 0] in the flow -U0 with (k, l) negated, bit for bit:
    t - absh = -(-t + absh), the RHS is odd in (U, k) for x and even for k, |.| and eps(|t|) are unchanged"""
    n, T = 6, 2.0
    ts = np.linspace(T, 0.0, 21)
    for U0 in (3.0, 10.0, 30.0):
        Yb, sb = B.ode23(cs_odefun(n, U0), ts, packets(n), 1e-3, 1e-6)
        if sb["nfailed"] > 0:
            break
    assert sb["nfailed"] > 0
    Yf, sf = B.ode23(cs_odefun(n, -U0), -ts, mirror(packets(n), n), 1e-3, 1e-6)
    assert (sb["nsteps"], sb["nfailed"], sb["nfevals"]) == (sf["nsteps"], sf["nfailed"], sf["nfevals"])
    assert np.array_equal(sb["h"], -sf["h"]) and sb["t"] == -sf["t"] == 0.0
    assert np.array_equal(Yb, mirror(Yf, n))


class OracleEngine:
    """oracle-backed stand-in with the Engine interface (tests/test_host_logic.py's), its ode23 building blocks in
    oracle.ode23's operation order, with the dense output (bs23_interp) added"""

    def __init__(self, grids, dx, f, gH):
        self.grids, self.dx, self.f, self.gH = grids, dx, f, gH
        self.attempts = 0

    @property
    def n(self):
        return self.s[0].size

    def set_packets(self, x, y, k, l, a=None):
        self.s = [np.array(v, dtype=np.float64) for v in (x, y, k, l)]

    def get_packets(self, with_a=False):
        return tuple(self.s)

    def _F(self, alpha, st):
        e6 = CO.interpolate6(st[0], st[1], self.grids, self.dx)
        return list(O.rhs_from_eval(e6, st[2], st[3], self.f, np.sqrt(self.gH)))

    def odefun(self, t, y):
        """the same RHS on the oracle's flat state"""
        return np.concatenate(self._F(0.0, np.split(y, 4)))

    def bs23_begin(self, alpha, thr):
        self.f1 = self._F(alpha, self.s)
        return max(np.max(np.abs(f) / np.maximum(np.abs(y), thr)) for f, y in zip(self.f1, self.s))

    def bs23_attempt(self, h, alphas, thr):
        self.attempts += 1
        assert self.attempts < 10000, "runaway solve"
        y = self.s
        self.f2 = self._F(alphas[0], [a + b * (h * 0.5) for a, b in zip(y, self.f1)])
        self.f3 = self._F(alphas[1], [a + b * (h * 0.75) for a, b in zip(y, self.f2)])
        self.yn = [a + (b * (h * (2.0 / 9.0)) + c * (h * (1.0 / 3.0)) + d * (h * (4.0 / 9.0)))
                   for a, b, c, d in zip(y, self.f1, self.f2, self.f3)]
        self.f4 = self._F(alphas[2], self.yn)
        fE = [b * (-5 / 72) + c * (1 / 12) + d * (1 / 9) + e * (-1 / 8) for b, c, d, e in zip(self.f1, self.f2, self.f3, self.f4)]
        return max(np.max(np.abs(g) / np.maximum(np.maximum(np.abs(a), np.abs(b)), thr)) for g, a, b in zip(fE, y, self.yn))

    def bs23_interp(self, h, s):
        if s == 1.0:
            return tuple(self.yn)
        s2, s3 = s * s, s * s * s
        w = (h * (s - 4.0 / 3.0 * s2 + 5.0 / 9.0 * s3), h * (s2 - 2.0 / 3.0 * s3), h * (4.0 / 3.0 * s2 - 8.0 / 9.0 * s3), h * (-s2 + s3))
        return tuple(a + (b * w[0] + c * w[1] + d * w[2] + e * w[3]) for a, b, c, d, e in zip(self.s, self.f1, self.f2, self.f3, self.f4))

    def bs23_accept(self):
        self.s, self.f1 = self.yn, self.f4


def c2_engine(n, psik_sign=1.0):
    w = W.make_workload("C2", n_packets=n, nx=32)
    kx_, ky_ = O.wavenumbers(32)
    grids = [O.k2g(p) for p in O.velocity_planes_k(psik_sign * w.psik, kx_, ky_)]
    return w, OracleEngine(grids, w.dx, w.f, w.gH)


@pytest.mark.parametrize("dense", [False, True])
def test_host_controller_backward_equals_oracle(dense):
    n = 64
    w, e = c2_engine(n)
    T = 20 * w.dt
    tspan = np.linspace(T, 0.0, 17) if dense else [T, 0.0]
    e.set_packets(w.x, w.y, w.k, w.l)
    st = R.ode23(e, tspan, None)
    got = np.concatenate(e.get_packets())
    ref, so = B.ode23(e.odefun, tspan, np.concatenate([w.x, w.y, w.k, w.l]))
    assert (st["nsteps"], st["nfailed"], st["nfevals"], st["t"]) == (so["nsteps"], so["nfailed"], so["nfevals"], 0.0)
    assert st["nsteps"] >= 10
    if dense:
        assert np.array_equal(st["Y"].reshape(len(tspan), 4 * n), ref) and np.array_equal(got, ref[-1])
    else:
        assert np.array_equal(got, ref)


def test_host_controller_mirror_takes_the_mirror_steps():
    """backward over [T .. 0] finishes (no runaway) in exactly the steps of its forward mirror over [-T .. 0] in the
    flow -psi, and its packets are the mirror's with k, l negated, bit for bit"""
    n = 64
    w, e = c2_engine(n)
    _, em = c2_engine(n, -1.0)
    T = 20 * w.dt
    ts = np.linspace(T, 0.0, 9)
    e.set_packets(w.x, w.y, w.k, w.l)
    em.set_packets(w.x, w.y, -w.k, -w.l)
    a, b = R.ode23(e, ts, None), R.ode23(em, -ts, None)
    assert (a["nsteps"], a["nfailed"], a["nfevals"]) == (b["nsteps"], b["nfailed"], b["nfevals"]) and a["nsteps"] >= 10
    assert e.attempts == em.attempts == a["nsteps"] + a["nfailed"]
    assert np.array_equal(a["Y"], b["Y"] * np.array([1, 1, -1, -1.0])[None, :, None])


@pytest.mark.parametrize("tspan", [[0.0, 1.0, 0.5, 2.0], [2.0, 1.0, 1.5, 0.0], [1.0, 2.0, 0.0]])
def test_tspan_against_its_direction_is_refused(tspan):
    w, e = c2_engine(16)
    e.set_packets(w.x, w.y, w.k, w.l)
    with pytest.raises(ValueError, match="monotonic"):
        R.ode23(e, tspan, None)
    with pytest.raises(ValueError, match="monotonic"):
        B.ode23(e.odefun, tspan, np.concatenate([w.x, w.y, w.k, w.l]))
    assert e.attempts == 0


def test_equal_neighbours_stay_accepted():
    w, e = c2_engine(16)
    T = 4 * w.dt
    ts = [T, T / 2, T / 2, 0.0]
    e.set_packets(w.x, w.y, w.k, w.l)
    st = R.ode23(e, ts, None)
    ref, _ = B.ode23(e.odefun, ts, np.concatenate([w.x, w.y, w.k, w.l]))
    assert np.array_equal(st["Y"].reshape(4, -1), ref) and np.array_equal(ref[1], ref[2])


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, str(ROOT))
    w, e = c2_engine(1001)
    ens = ShardedEnsemble(e, w.n_packets, rank, world, dist)
    ens.set_packets_global(w.x, w.y, w.k, w.l)
    st = ens.ode23([20 * w.dt, 0.0], np.inf)        # global error norm: MAX all-reduce per attempted step
    allq = ens.gather_packets()
    if rank == 0:
        np.savez(tmp, nsteps=st["nsteps"], nfailed=st["nfailed"], x=allq[0], y=allq[1], k=allq[2], l=allq[3])
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_two_ranks_backward_match_single_rank(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "r.npz")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = np.load(out)
    w, e = c2_engine(1001)
    ens = ShardedEnsemble(e, w.n_packets)
    ens.set_packets_global(w.x, w.y, w.k, w.l)
    st = ens.ode23([20 * w.dt, 0.0], np.inf)
    assert (int(got["nsteps"]), int(got["nfailed"])) == (st["nsteps"], st["nfailed"]) and st["nsteps"] >= 10
    for a, b in zip("xykl", ens.gather_packets()):
        assert np.array_equal(got[a], b), a
