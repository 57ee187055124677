"""swrt_packet_quantity / swrt_hist2 on the device: every quantity against a numpy restatement of the same operations,
every histogram against the host histcounts2 (tests/test_hist2_contract.py) of the device's own packet_quantity arrays,
both kernel paths (per-CTA shared-memory counters, global counters), agreement with swrt_hist_omega, accumulation, the
refusals, a two-GPU handle and the MEX gateway."""
import ctypes as C

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
from test_hist2_contract import histcounts2
from test_mex_gateway import Mex

pytestmark = pytest.mark.gpu

MODES = {"spectral": S.MODE_SPECTRAL, "lagrange6": S.MODE_LAGRANGE6, "nufft": S.MODE_NUFFT}
PI = np.pi
THETA_EDGES = np.linspace(-PI, PI, 37)


def _engine(w, mode=S.MODE_SPECTRAL, ngpu=1, flow=True):
    eng = S.Engine(w.nx, w.L, w.f, w.gH, mode, device=0, ngpu=ngpu)
    if flow:
        eng.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
        eng.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
    return eng


def _workload(n=4099):
    return W.make_workload("C4", n_packets=n, nx=32)          # L = 20, two frames, mean shear, k on a ring


def _wrap(x, L):
    r = x - L * np.floor(x / L)
    r = np.where(r < 0, r + L, r)
    return np.where(r >= L, 0.0, r)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _edge_packets(L):
    """x on multiples of L, within an ulp of them and many periods away, plus signed zeros"""
    m = np.array([0.0, 1.0, -1.0, 2.0, -3.0, 7.0, 1e3, -1e6, 2.0 ** 40])
    on = m * L
    xs = np.concatenate([on, np.nextafter(on, np.inf), np.nextafter(on, -np.inf), [-0.0, 0.0, 0.5 * L, L - 1e-300],
                         1e7 * L + np.array([0.3, -0.3, 1e-9]), np.linspace(-50 * L, 50 * L, 1001)])
    return xs


def test_positional_and_wavevector_quantities_are_the_numpy_expressions():
    w = _workload()
    x = _edge_packets(w.L)
    n = x.size
    rs = np.random.RandomState(1)
    y = np.roll(x, 7)
    k, l = rs.randn(n) * 3, rs.randn(n) * 3
    k[:4], l[:4] = [0.0, -0.0, 1e-160, 3e200], [0.0, 2.0, 1e-160, 1e-300]
    eng = _engine(w, flow=False)
    eng.set_packets(x, y, k, l)
    with np.errstate(over="ignore"):
        kmag = np.sqrt(k * k + l * l)                       # 3e200 squared overflows to inf, on the device too
    for q, ref in ((S.Q_XMOD, _wrap(x, w.L)), (S.Q_YMOD, _wrap(y, w.L)), (S.Q_K, k), (S.Q_L, l), (S.Q_KMAG, kmag)):
        got = eng.packet_quantity(q)
        assert np.array_equal(_bits(got), _bits(ref)), (q, np.flatnonzero(_bits(got) != _bits(ref))[:5])
    xm = eng.packet_quantity(S.Q_XMOD)
    assert xm.min() >= 0.0 and xm.max() < w.L
    eng.close()


def test_theta_is_atan2_within_two_ulp_and_exact_at_the_axes():
    w = _workload()
    rs = np.random.RandomState(2)
    k, l = rs.randn(20000), rs.randn(20000)
    k[:1000] *= 1e-8; l[1000:2000] *= 1e8                      # near the axes
    sk = np.array([0.0, 0.0, -0.0, -0.0, 1.0, -1.0, -1.0, 0.0, 0.0, -0.0, -0.0, 3.5, -2.0, -2.0])
    sl = np.array([0.0, -0.0, 0.0, -0.0, 0.0, 0.0, -0.0, 1.0, -1.0, 2.0, -5.0, -0.0, 0.0, -0.0])
    want = np.array([0.0, -0.0, PI, -PI, 0.0, PI, -PI, PI / 2, -PI / 2, PI / 2, -PI / 2, -0.0, PI, -PI])
    assert np.array_equal(_bits(np.arctan2(sl, sk)), _bits(want))
    k, l = np.concatenate([sk, k]), np.concatenate([sl, l])
    eng = _engine(w, flow=False)
    eng.set_packets(np.zeros_like(k), np.zeros_like(k), k, l)
    th = eng.packet_quantity(S.Q_THETA)
    eng.close()
    assert np.array_equal(_bits(th[:sk.size]), _bits(want))                   # +-0, +-pi/2, +-pi with both signed zeros
    ref = np.arctan2(l, k)
    assert np.all(np.abs(th - ref) <= 2 * np.spacing(np.abs(ref))) and th.min() >= -PI and th.max() <= PI


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("alpha", [0.0, 0.37])
def test_frequencies_equal_swrt_omega_bit_for_bit(mode, alpha):
    w = _workload()
    eng = _engine(w, MODES[mode])
    eng.set_packets(w.x, w.y, w.k * (1 + 0.1 * np.sin(np.arange(w.n_packets))), w.l)
    om, Om = eng.omega(alpha)
    assert np.array_equal(_bits(eng.packet_quantity(S.Q_OMEGA, alpha)), _bits(om))
    assert np.array_equal(_bits(eng.packet_quantity(S.Q_OMEGA_ABS, alpha)), _bits(Om))
    eng.close()


def _spread_packets(w, n, seed=4):
    """packets with |k| and omega spread off the ring, a few blown up and a few far out of range"""
    rs = np.random.RandomState(seed)
    th = rs.uniform(-PI, PI, n)
    kmag = np.abs(3.0 + 0.5 * rs.randn(n))
    k, l = kmag * np.cos(th), kmag * np.sin(th)
    x, y = rs.uniform(-2 * w.L, 2 * w.L, n), rs.uniform(-2 * w.L, 2 * w.L, n)
    k[5::211] = np.nan                                          # blown-up packets
    x[7::307] = np.inf
    k[9::401] = 1e6                                             # far out of range
    return x, y, k, l


EDGES = {
    "uniform": lambda lo, hi: np.linspace(lo, hi, 41),
    "nonuniform": lambda lo, hi: lo + (hi - lo) * np.linspace(0.0, 1.0, 29) ** 2,
    "repeated": lambda lo, hi: np.sort(np.concatenate([np.linspace(lo, hi, 21), np.linspace(lo, hi, 21)[5:9], [hi, hi]])),
}
PAIRS = {"kmag_theta": (S.Q_KMAG, (1.0, 5.0), S.Q_THETA, (-PI, PI)),
         "omegaabs_theta": (S.Q_OMEGA_ABS, None, S.Q_THETA, (-PI, PI)),
         "xmod_ymod": (S.Q_XMOD, (0.0, 20.0), S.Q_YMOD, (2.0, 17.0))}


@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("edges", list(EDGES))
def test_hist2_equals_host_histcounts2_of_the_device_quantities(pair, edges):
    w = _workload()
    qx, xr, qy, yr = PAIRS[pair]
    eng = _engine(w)
    eng.set_packets(*_spread_packets(w, 30011))
    alpha = 0.25
    vx, vy = eng.packet_quantity(qx, alpha), eng.packet_quantity(qy, alpha)
    if xr is None:
        f = vx[np.isfinite(vx)]
        xr = (np.quantile(f, 0.02), np.quantile(f, 0.98))
    xe, ye = EDGES[edges](*xr), EDGES[edges](*yr)
    got = eng.hist2(qx, xe, qy, ye, alpha)
    ref = histcounts2(vx, vy, xe, ye)
    assert got.shape == (xe.size - 1, ye.size - 1) and got.dtype == np.uint64
    assert np.array_equal(got, ref) and 0 < int(ref.sum()) < w.n_packets * 10
    eng.close()


def test_packets_on_edges_and_dropped_packets():
    """k on inner and outer |k| edges (|k| = sqrt(k*k) is exact), theta exactly -pi, 0, pi/2, pi; x on the x edges,
    including the closed last bin of each axis; NaN and out-of-range packets are not counted"""
    w = _workload()
    ke = np.array([1.0, 1.5, 2.0, 2.5, 3.0, 4.0])
    te = np.array([-PI, -PI / 2, 0.0, PI / 2, PI])
    k = np.concatenate([ke, -ke, -ke, [0.0, 0.0, np.nan, 4.5, 0.5, np.inf]])
    l = np.concatenate([0.0 * ke, 0.0 * ke, -0.0 * ke, [1.5, -4.0, 1.0, 0.0, 0.0, 0.0]])
    n = k.size
    xe = np.array([0.0, 2.5, 5.0, 10.0])
    x = np.resize(np.array([0.0, 2.5, 5.0, 10.0, 20.0, 7.0]), n)      # 20 wraps to 0; 10 is the closed last x edge
    y = np.resize(np.array([10.0, 0.0, 2.5, 11.0]), n)
    eng = _engine(w, flow=False)
    eng.set_packets(x, y, k, l)
    km, th = eng.packet_quantity(S.Q_KMAG), eng.packet_quantity(S.Q_THETA)
    assert set(km[:18]) <= set(ke) and set(th[:18]) <= {0.0, PI, -PI}
    got = eng.hist2(S.Q_KMAG, ke, S.Q_THETA, te)
    assert np.array_equal(got, histcounts2(km, th, ke, te))
    # the closed last bins: |k| in [3, 4] holds k = -3 and k = -4 (on the outer edge), theta = pi and -pi (both outer edges)
    assert got[-1, -1] == 2 and got[-1, 0] == 2 and got[0, -1] == 1 and got[0, 0] == 1
    assert int(got.sum()) == 18 + 2                                    # NaN, 4.5 (out of range), 0.5 and inf dropped
    gx = eng.hist2(S.Q_XMOD, xe, S.Q_YMOD, xe)
    assert np.array_equal(gx, histcounts2(eng.packet_quantity(S.Q_XMOD), eng.packet_quantity(S.Q_YMOD), xe, xe))
    assert gx[-1, :].sum() > 0 and gx[:, -1].sum() > 0
    eng.close()


@pytest.mark.parametrize("bins", [(65, 65), (4096, 65), (4096, 4096)], ids=["64x64-shared", "4095x64-global", "4095x4095-global"])
def test_both_kernel_paths_equal_host_histcounts2(bins):
    w = _workload()
    eng = _engine(w, flow=False)
    n = 1_000_003
    rs = np.random.RandomState(7)
    th = rs.uniform(-PI, PI, n)
    kmag = rs.uniform(0.5, 5.5, n)
    eng.set_packets(rs.uniform(0, w.L, n), rs.uniform(0, w.L, n), kmag * np.cos(th), kmag * np.sin(th))
    xe, ye = np.linspace(1.0, 5.0, bins[0]), np.linspace(-PI, PI, bins[1])
    got = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)
    assert np.array_equal(got, histcounts2(eng.packet_quantity(S.Q_KMAG), eng.packet_quantity(S.Q_THETA), xe, ye))
    eng.close()


@pytest.mark.parametrize("bins", [(65, 65), (4096, 65)], ids=["shared", "global"])
def test_every_packet_in_one_bin_counts_n(bins):
    """the ring initial condition with narrow |k| bins: every packet in one bin, on both paths"""
    w = _workload()
    eng = _engine(w, flow=False)
    n = 2_000_001
    eng.set_packets(np.zeros(n), np.zeros(n), np.full(n, 3.0), np.full(n, 1e-3))
    xe, ye = np.linspace(2.0, 4.0, bins[0]), np.linspace(0.0, 0.5, bins[1])
    got = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)
    assert int(got.sum()) == n and int(got.max()) == n
    eng.close()


@pytest.mark.parametrize("kind,q", [(S.HIST_INTRINSIC, S.Q_OMEGA), (S.HIST_ABSOLUTE, S.Q_OMEGA_ABS)])
def test_summed_over_theta_equals_hist_omega(kind, q):
    w = _workload()
    eng = _engine(w)
    eng.set_packets(*_spread_packets(w, 50021))
    alpha = 0.6
    vals = eng.packet_quantity(q, alpha)
    f = vals[np.isfinite(vals)]
    edges = np.linspace(f.min() * 0.99, np.quantile(f, 0.9), 301)
    h1 = eng.hist_omega(edges, kind, alpha)
    h2 = eng.hist2(q, edges, S.Q_THETA, np.array([-PI, PI]), alpha)
    assert h2.shape == (300, 1) and np.array_equal(h2[:, 0], h1) and int(h1.sum()) > 0
    eng.close()


def test_accumulate_adds_to_the_given_counts():
    w = _workload()
    eng = _engine(w)
    eng.set_packets(*_spread_packets(w, 10007))
    xe, ye = np.linspace(1.0, 5.0, 33), THETA_EDGES
    a = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)
    c = a + np.uint64(5)
    out = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye, counts=c)
    assert out is c and np.array_equal(c, 2 * a + np.uint64(5))
    eng.close()


def test_refusals_leave_the_handle_usable():
    w = _workload()
    eng = _engine(w)
    eng.set_packets(*_spread_packets(w, 5003))
    lib, h = eng.lib, eng._h
    xe, ye = np.linspace(1.0, 5.0, 33), THETA_EDGES
    before = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)
    u64 = C.POINTER(C.c_uint64)
    out = np.zeros(32 * 36, dtype=np.uint64)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))                  # noqa: E731
    cp = out.ctypes.data_as(u64)
    dec = xe.copy(); dec[5] = dec[4] - 1e-12
    nan, inf = xe.copy(), xe.copy()
    nan[3] = np.nan; inf[-1] = np.inf
    big = np.linspace(0.0, 1.0, 4097)
    calls = [(8, dp(xe), 33, S.Q_THETA, dp(ye), 37, cp), (-1, dp(xe), 33, S.Q_THETA, dp(ye), 37, cp),
             (S.Q_KMAG, dp(xe), 33, 99, dp(ye), 37, cp),
             (S.Q_KMAG, dp(xe), 1, S.Q_THETA, dp(ye), 37, cp), (S.Q_KMAG, dp(xe), 33, S.Q_THETA, dp(ye), 1, cp),
             (S.Q_KMAG, dp(big), 4097, S.Q_THETA, dp(ye), 37, cp), (S.Q_KMAG, dp(xe), 33, S.Q_THETA, dp(big), 4097, cp),
             (S.Q_KMAG, dp(dec), 33, S.Q_THETA, dp(ye), 37, cp), (S.Q_KMAG, dp(xe), 33, S.Q_THETA, dp(dec), 33, cp),
             (S.Q_KMAG, dp(nan), 33, S.Q_THETA, dp(ye), 37, cp), (S.Q_KMAG, dp(inf), 33, S.Q_THETA, dp(ye), 37, cp),
             (S.Q_KMAG, None, 33, S.Q_THETA, dp(ye), 37, cp), (S.Q_KMAG, dp(xe), 33, S.Q_THETA, None, 37, cp),
             (S.Q_KMAG, dp(xe), 33, S.Q_THETA, dp(ye), 37, None)]
    for qx, xp, nx_, qy, yp, ny_, c in calls:
        assert lib.swrt_hist2(h, qx, xp, nx_, qy, yp, ny_, 0.0, c, 0) == -1
        assert np.array_equal(eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye), before)
    qo = np.empty(eng.n)
    assert lib.swrt_packet_quantity(h, 8, 0.0, dp(qo)) == -1 and lib.swrt_packet_quantity(h, S.Q_K, 0.0, None) == -1
    assert np.array_equal(eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye), before)
    eng.close()


def test_state_refusals():
    """OMEGA_ABS needs flow slot 0; a two-frame alpha needs slot 1 (as swrt_omega refuses it)"""
    w = _workload()
    x, y, k, l = _spread_packets(w, 1001)
    bare = _engine(w, flow=False)
    bare.set_packets(x, y, k, l)
    for call in (lambda: bare.hist2(S.Q_OMEGA_ABS, np.linspace(0, 9, 5), S.Q_THETA, THETA_EDGES),
                 lambda: bare.packet_quantity(S.Q_OMEGA_ABS)):
        with pytest.raises(S.SwrtError) as ei:
            call()
        assert ei.value.code == -2
    assert bare.hist2(S.Q_OMEGA, np.linspace(0, 9, 5), S.Q_THETA, THETA_EDGES).sum() > 0     # omega needs no flow
    bare.close()
    one = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL)
    one.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
    one.set_packets(x, y, k, l)
    with pytest.raises(S.SwrtError) as ei:
        one.hist2(S.Q_OMEGA_ABS, np.linspace(0, 9, 5), S.Q_THETA, THETA_EDGES, alpha=0.5)
    assert ei.value.code == -2
    with pytest.raises(S.SwrtError) as ei2:
        one.omega(0.5)
    assert ei2.value.code == -2
    assert one.hist2(S.Q_OMEGA_ABS, np.linspace(0, 9, 5), S.Q_THETA, THETA_EDGES).sum() > 0
    one.close()


def test_two_gpu_handle_equals_one_gpu():
    if S.load_library().swrt_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    w = _workload(20011)
    pk = _spread_packets(w, 20011)
    res = []
    for ngpu in (1, 2):
        eng = _engine(w, ngpu=ngpu)
        eng.set_packets(*pk)
        res.append((eng.hist2(S.Q_OMEGA_ABS, np.linspace(2.0, 9.0, 129), S.Q_THETA, THETA_EDGES, 0.3),
                    eng.hist2(S.Q_XMOD, np.linspace(0, 20, 4001), S.Q_YMOD, np.linspace(0, 20, 201)),
                    eng.packet_quantity(S.Q_OMEGA_ABS, 0.3)))
        eng.close()
    for a, b in zip(*res):
        assert np.array_equal(a, b)


@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    return Mex(request.param)


def test_mex_hist2_and_packet_quantity_equal_the_engine(mex):
    w = _workload(3001)
    pk = _spread_packets(w, 3001)
    xe, ye = np.linspace(1.0, 5.0, 17), THETA_EDGES
    h = mex("create", float(w.nx), w.L, w.f, w.gH, 0.0)
    mex("set_flow_spectral", h, 0.0, w.psik, w.u_mean, nlhs=0)
    mex("set_flow_spectral", h, 1.0, w.psik2, w.u_mean, nlhs=0)
    mex("set_packets", h, *pk, nlhs=0)
    N = mex("hist2", h, float(S.Q_KMAG), xe, float(S.Q_THETA), ye)
    Na = mex("hist2", h, float(S.Q_OMEGA_ABS), np.linspace(2.0, 9.0, 33), float(S.Q_THETA), ye, 0.4)
    qs = {q: mex("packet_quantity", h, float(q), 0.4) for q in range(8)}
    mex("destroy", h, nlhs=0)
    eng = _engine(w)
    eng.set_packets(*pk)
    assert N.dtype == np.float64 and N.shape == (16, 36)
    assert np.array_equal(N, eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye).astype(np.float64))
    assert np.array_equal(Na, eng.hist2(S.Q_OMEGA_ABS, np.linspace(2.0, 9.0, 33), S.Q_THETA, ye, 0.4).astype(np.float64))
    for q, v in qs.items():
        assert v.shape == (3001,) and np.array_equal(_bits(v), _bits(eng.packet_quantity(q, 0.4))), q
    eng.close()
