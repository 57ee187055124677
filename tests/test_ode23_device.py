"""swrt_ode23 / Engine.ode23: a whole ode23 solve with the step-size controller on the device, checked against the host
controller (reference_api.ode23) driving the same device building blocks."""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from oracle import swrt_oracle as O

pytestmark = pytest.mark.gpu

L = 2 * np.pi
F0, GH0 = 3.0, 1.0
MODES = [(S.MODE_SPECTRAL, 32), (S.MODE_SPECTRAL, 64), (S.MODE_LAGRANGE6, 32), (S.MODE_NUFFT, 32)]


def make_psik(nx, seed, amp=0.3):
    rs = np.random.RandomState(seed)
    kx_, ky_ = O.wavenumbers(nx)
    return (rs.randn(nx - 1, nx // 2) + 1j * rs.randn(nx - 1, nx // 2)) / (1 + kx_ ** 2 + ky_ ** 2) ** 1.5 * amp


def make_packets(n, seed=5):
    rs = np.random.RandomState(seed)
    i = np.arange(n)
    return rs.uniform(-L, L, n), rs.uniform(-L, L, n), 3 * np.cos(0.37 * i), 3 * np.sin(0.37 * i)


def engine(mode, nx, two, ngpu=1, amp=0.3):
    e = S.Engine(nx, L, F0, GH0, mode, ngpu=ngpu)
    e.set_flow_spectral(make_psik(nx, 7, amp), slot=0)
    if two:
        e.set_flow_spectral(make_psik(nx, 8, amp), slot=1)
    return e


class Recorder:
    """the host controller's target, recording the step size of every accepted attempt"""
    def __init__(self, eng):
        self.eng, self.h, self._last = eng, [], None

    def __getattr__(self, name):
        return getattr(self.eng, name)

    def bs23_attempt(self, hstep, alphas, threshold):
        self._last = hstep
        return self.eng.bs23_attempt(hstep, alphas, threshold)

    def bs23_accept(self):
        self.h.append(self._last)
        return self.eng.bs23_accept()


def host_and_device(e, packets, tspan, tmax, rtol, atol):
    e.set_packets(*packets)
    rec = Recorder(e)
    sh = R.ode23(rec, tspan, tmax, rtol, atol)
    ph = np.stack(e.get_packets())
    e.set_packets(*packets)
    sd = e.ode23(tspan, tmax, rtol, atol, trace=100000)
    pd = np.stack(e.get_packets())
    return sh, np.array(rec.h), ph, sd, pd


def assert_same_solve(sh, hh, ph, sd, pd, tfinal, exact_if_same_steps=False):
    assert (sd["nsteps"], sd["nfailed"], sd["nfevals"]) == (sh["nsteps"], sh["nfailed"], sh["nfevals"])
    assert sh["t"] == tfinal and sd["t"] == tfinal
    hd = sd["h"]
    assert hd.shape == hh.shape
    # the device power is correctly rounded; glibc's pow (the host controller's) is off by one ulp on rare arguments
    assert np.all(np.abs(hd - hh) <= 2 * np.spacing(np.abs(hh)))
    assert abs(hd.sum() - (tfinal - 0.0)) < 1e-12 * max(1.0, abs(tfinal))
    scale = np.abs(ph).max(axis=1, keepdims=True)
    assert np.all(np.abs(pd - ph) <= 1e-12 * scale)
    if exact_if_same_steps and np.array_equal(hd, hh):
        assert np.array_equal(pd, ph)


@pytest.mark.parametrize("mode,nx", MODES)
@pytest.mark.parametrize("two", [False, True])
@pytest.mark.parametrize("tol", [(1e-3, 1e-6), (1e-6, 1e-7)])
def test_same_solve_as_host_controller(mode, nx, two, tol):
    tmax = 0.4
    with engine(mode, nx, two) as e:
        sh, hh, ph, sd, pd = host_and_device(e, make_packets(300), [0.0, tmax], tmax if two else None, *tol)
        assert sh["nsteps"] >= 10                    # MaxStep = 0.1*(tf - t0)
        assert_same_solve(sh, hh, ph, sd, pd, tmax, exact_if_same_steps=mode == S.MODE_LAGRANGE6)


@pytest.mark.parametrize("mode,nx", MODES)
def test_rejections_match(mode, nx):
    # a strong flow: the controller's first guesses are rejected.  The solve is kept to a few hundred steps because the
    # flow is chaotic: over thousands of steps a one-ulp step-size difference (glibc's pow, DESIGN.md section 11) grows
    # beyond the tolerances below
    for amp in (3.0, 10.0, 30.0):
        with engine(mode, nx, True, amp=amp) as e:
            sh, hh, ph, sd, pd = host_and_device(e, make_packets(200, seed=9), [0.0, 0.2], 0.2, 1e-3, 1e-6)
        if sh["nfailed"] > 0:
            break
    assert sh["nfailed"] > 0 and sh["nsteps"] <= 400
    assert_same_solve(sh, hh, ph, sd, pd, 0.2, exact_if_same_steps=mode == S.MODE_LAGRANGE6)


@pytest.mark.parametrize("mode", [S.MODE_SPECTRAL, S.MODE_LAGRANGE6])
def test_dense_output_c1_shape(mode):
    # SW_zero_background_raytracing.m:70-78: 1,000 packets, RelTol 1e-6, AbsTol 1e-7, output at dt*(0:N)
    dt, N = 0.05, 40
    tspan = dt * np.arange(N + 1)
    with engine(mode, 32, False) as e:
        pk = make_packets(1000, seed=3)
        e.set_packets(*pk)
        sh = R.ode23(e, tspan, None, 1e-6, 1e-7)
        e.set_packets(*pk)
        sd = e.ode23(tspan, None, 1e-6, 1e-7)
        assert (sd["nsteps"], sd["nfailed"], sd["nfevals"]) == (sh["nsteps"], sh["nfailed"], sh["nfevals"])
        assert sd["Y"].shape == sh["Y"].shape == (N + 1, 4, 1000)
        assert np.array_equal(sd["Y"][0], np.stack(pk))
        scale = np.abs(sh["Y"]).max(axis=(0, 2))[None, :, None]
        assert np.all(np.abs(sd["Y"] - sh["Y"]) <= 1e-12 * scale)
        assert np.array_equal(sd["Y"][-1], np.stack(e.get_packets()))     # the last row is ynew of the final step


def test_shuffled_ensemble_is_permuted_bit_for_bit():
    pk = np.stack(make_packets(5000, seed=11))
    perm = np.random.RandomState(1).permutation(pk.shape[1])
    with engine(S.MODE_SPECTRAL, 64, True) as e:
        e.set_packets(*pk)
        a = e.ode23([0.0, 0.4], 0.4, 1e-6, 1e-7, trace=1000)
        ya = np.stack(e.get_packets())
        e.set_packets(*pk[:, perm])
        b = e.ode23([0.0, 0.4], 0.4, 1e-6, 1e-7, trace=1000)
        yb = np.stack(e.get_packets())
    assert (a["nsteps"], a["nfailed"]) == (b["nsteps"], b["nfailed"]) and np.array_equal(a["h"], b["h"])
    assert np.array_equal(yb, ya[:, perm])


def test_two_devices_equal_one_bit_for_bit():
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two GPUs")
    pk = make_packets(3001, seed=12)
    tspan = 0.04 * np.arange(11)
    res = []
    for ngpu in (1, 2):
        with engine(S.MODE_SPECTRAL, 32, True, ngpu=ngpu) as e:
            e.set_packets(*pk)
            st = e.ode23(tspan, 0.4, 1e-6, 1e-7, trace=1000)
            res.append((st, np.stack(e.get_packets())))
    (a, ya), (b, yb) = res
    assert (a["nsteps"], a["nfailed"], a["nfevals"]) == (b["nsteps"], b["nfailed"], b["nfevals"])
    assert np.array_equal(a["h"], b["h"]) and np.array_equal(ya, yb) and np.array_equal(a["Y"], b["Y"])


def test_few_host_waits_and_launches_per_batch():
    # the reference's unit of work at 50 packets: one solve over a QG step [0, dt] between two frames (C3 flow, 256^2).
    # LAGRANGE6 attempt: 3 x (stage, evaluation, RHS) + norm + controller + accept
    from swraytracing_b200 import workloads as W
    w = W.make_workload("C3", n_packets=50)
    per_attempt = 12
    with S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6) as e:
        e.set_flow_spectral(w.psik, 0, u_mean=w.u_mean); e.set_flow_spectral(w.psik2, 1, u_mean=w.u_mean)
        e.set_packets(w.x, w.y, w.k, w.l)
        e.launch_count(reset=True)
        st = e.ode23([0.0, w.dt], w.dt)
        launches = e.launch_count()
    assert st["nsteps"] == 12
    assert st["host_waits"] <= 3
    # begin (evaluation, RHS, norm) + the controller's set-up, then whole attempts only, at least one per decision
    queued, rest = divmod(launches - 4, per_attempt)
    assert rest == 0 and queued >= st["nsteps"] + st["nfailed"]


@pytest.mark.parametrize("mode", [S.MODE_SPECTRAL, S.MODE_LAGRANGE6, S.MODE_NUFFT])
def test_blown_up_packet_fails_like_host_and_handle_survives(mode):
    pk = [a.copy() for a in make_packets(100)]
    pk[2][17] = np.inf
    with engine(mode, 32, True) as e:
        e.set_packets(*pk)
        with pytest.raises(RuntimeError, match="hmin at t"):
            R.ode23(e, [0.0, 0.4], 0.4)
        e.set_packets(*pk)
        with pytest.raises(S.SwrtError, match="hmin at t = ") as ex:
            e.ode23([0.0, 0.4], 0.4)
        assert ex.value.code == -2                   # SWRT_ERR_STATE
        # the same handle solves the next (finite) ensemble exactly as the host controller does
        good = make_packets(100)
        sh, hh, ph, sd, pd = host_and_device(e, good, [0.0, 0.4], 0.4, 1e-3, 1e-6)
        assert_same_solve(sh, hh, ph, sd, pd, 0.4)


def test_qgsw_driver_ode23_device(tmp_path):
    from swraytracing_b200 import drivers, fieldio
    nx, Np, nif, U_g, f, Cg = 64, 20, 2.0, 0.5, 3.0, 1.0
    out = {}
    for integ in ("ode23", "ode23_device"):
        d = tmp_path / integ
        out[integ] = drivers.qgsw_raytrace(nx, Np, nif, 6000, 0, U_g, f, Cg, outdir=str(d), max_steps=6, r_drag=0.01,
                                           integrator=integ, log=lambda s: None)
    a, b = out["ode23"], out["ode23_device"]
    assert (a["ode23_steps"], a["ode23_failed"]) == (b["ode23_steps"], b["ode23_failed"]) and a["ode23_steps"] >= 60
    assert np.abs(np.concatenate(a["packets"]) - np.concatenate(b["packets"])).max() < 1e-9
    ta, xa, ka = fieldio.load_packet_frames(tmp_path / "ode23", Np)
    tb, xb, kb = fieldio.load_packet_frames(tmp_path / "ode23_device", Np)
    assert np.array_equal(ta, tb) and np.abs(xa - xb).max() < 1e-9 and np.abs(ka - kb).max() < 1e-9
