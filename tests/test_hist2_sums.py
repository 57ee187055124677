"""swrt_weight_scale / swrt_hist2_sums on the device.  The weights are recomputed in numpy from get_packets and the
device's omega (one rounded product each, as on the device) and binned with the host bin rule (tests/test_hist2_contract.py);
every bin is held to the correctly rounded exact sum (Fraction) where the contract makes it exact, and to the fixed-point
mirror of tests/test_hist2_sums_contract.py bit for bit everywhere.  Also: counts, invariance under packet order, halves
and two GPUs, the edge cases, the refusals and the MEX gateway."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

import swraytracing_b200 as S
from test_hist2 import _engine, _workload, THETA_EDGES
from test_hist2_contract import bin_of
from test_hist2_sums_contract import exact_double, mirror_acc, scale_exp_of
from test_mex_gateway import Mex

pytestmark = pytest.mark.gpu

PI = np.pi
ALL_W = [S.W_ACTION, S.W_ENERGY, S.W_PSEUDO_K, S.W_PSEUDO_L]
PAIRS = {"kmag_theta": (S.Q_KMAG, np.linspace(2.0, 4.0, 17), S.Q_THETA, THETA_EDGES),
         "xmod_ymod": (S.Q_XMOD, np.linspace(0.0, 20.0, 11), S.Q_YMOD, np.linspace(0.0, 20.0, 9))}


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _packets(n, wavevectors, seed=3, L=20.0):
    rs = np.random.RandomState(seed)
    th = rs.uniform(-PI, PI, n)
    kmag = np.full(n, 3.0) if wavevectors == "ring" else rs.uniform(1.8, 4.2, n)
    return rs.uniform(-L, 2 * L, n), rs.uniform(-L, 2 * L, n), kmag * np.cos(th), kmag * np.sin(th)


def _host(eng, qx, xe, qy, ye, kinds, alpha):
    """the flat bin of every packet (-1: not counted) and the weights of each kind, from the device's own packets"""
    _, _, k, l, a = eng.get_packets(with_a=True)
    om = eng.packet_quantity(S.Q_OMEGA, alpha)
    bx, by = bin_of(eng.packet_quantity(qx, alpha), xe), bin_of(eng.packet_quantity(qy, alpha), ye)
    bins = np.where((bx >= 0) & (by >= 0), bx + by * (len(xe) - 1), -1)
    w = {S.W_ACTION: a, S.W_ENERGY: om * a, S.W_PSEUDO_K: k * a, S.W_PSEUDO_L: l * a}
    return bins, [w[v] for v in kinds]


def _mirror(bins, ws, exps, nbx, nby):
    acc = np.stack([mirror_acc(bins, w, int(E), nbx * nby) for w, E in zip(ws, exps)])
    return acc.reshape(len(ws), nby, nbx, 4).transpose(0, 2, 1, 3)


def _check_against_mirror(eng, qx, xe, qy, ye, kinds, alpha=0.0):
    nbx, nby = len(xe) - 1, len(ye) - 1
    sums, counts, acc = eng.hist2_sums(qx, xe, qy, ye, kinds, alpha, return_acc=True)
    bins, ws = _host(eng, qx, xe, qy, ye, kinds, alpha)
    exps = eng.weight_scale(kinds, alpha)
    assert exps.tolist() == [scale_exp_of(w) for w in ws]
    ref_acc = _mirror(bins, ws, exps, nbx, nby)
    assert np.array_equal(acc, ref_acc)
    assert np.array_equal(_bits(sums), _bits(S.fixed_sums_to_double(ref_acc, exps)))
    assert np.array_equal(counts, eng.hist2(qx, xe, qy, ye, alpha))
    return sums, counts, bins, ws


@pytest.mark.parametrize("wavevectors", ["ring", "random"])
@pytest.mark.parametrize("pair", list(PAIRS))
def test_sums_are_the_correctly_rounded_exact_sums(pair, wavevectors):
    """a in [0.5, 2]: every weight within 2^42 of the largest, so each bin is the exact sum rounded once"""
    w = _workload()
    qx, xe, qy, ye = PAIRS[pair]
    eng = _engine(w)
    n = 20011
    rs = np.random.RandomState(1)
    eng.set_packets(*_packets(n, wavevectors), a=rs.uniform(0.5, 2.0, n))
    alpha = 0.3
    sums, counts, bins, ws = _check_against_mirror(eng, qx, xe, qy, ye, ALL_W, alpha)
    nbx = len(xe) - 1
    for v, wv in enumerate(ws):
        E = scale_exp_of(wv)
        assert np.all(np.abs(wv[bins >= 0]) >= np.ldexp(1.0, E - 43))
        exact = {}
        for b, x in zip(bins, wv):
            if b >= 0:
                exact[b] = exact.get(b, 0) + Fraction(float(x))
        for b, f in exact.items():
            want = exact_double(int(f * 2 ** (95 - E)), E)
            assert f * 2 ** (95 - E) == int(f * 2 ** (95 - E))
            assert _bits([sums[v, b % nbx, b // nbx]])[0] == _bits([want])[0], (v, b)
    assert int(counts.sum()) > n // 4 and np.all(sums[0][counts == 0] == 0.0)
    eng.close()


@pytest.mark.parametrize("wavevectors", ["ring", "random"])
def test_spread_actions_equal_the_fixed_point_mirror(wavevectors):
    """a over 2^-60..1: small weights are rounded to 2^(E-95), exactly as the mirror rounds them"""
    w = _workload()
    eng = _engine(w)
    n = 100003
    rs = np.random.RandomState(2)
    eng.set_packets(*_packets(n, wavevectors, seed=5), a=np.exp2(rs.uniform(-60.0, 0.0, n)))
    _check_against_mirror(eng, S.Q_KMAG, np.linspace(2.0, 4.0, 65), S.Q_THETA, THETA_EDGES, ALL_W, 0.7)
    _check_against_mirror(eng, S.Q_XMOD, np.linspace(0.0, 20.0, 129), S.Q_YMOD, np.linspace(0.0, 20.0, 257), [S.W_PSEUDO_L])
    eng.close()


def test_large_grid_and_every_packet_in_one_bin():
    w = _workload()
    eng = _engine(w, flow=False)
    n = 1_000_003
    rs = np.random.RandomState(7)
    eng.set_packets(*_packets(n, "random", seed=7), a=np.exp2(rs.uniform(-20.0, 0.0, n)))
    _check_against_mirror(eng, S.Q_KMAG, np.linspace(1.5, 4.5, 513), S.Q_THETA, np.linspace(-PI, PI, 513), ALL_W)
    m = 2_000_001
    eng.set_packets(np.zeros(m), np.zeros(m), np.full(m, 3.0), np.full(m, 1e-3), a=rs.uniform(0.5, 2.0, m))
    sums, counts, _, ws = _check_against_mirror(eng, S.Q_KMAG, np.linspace(2.0, 4.0, 65), S.Q_THETA, np.linspace(0.0, 0.5, 65), ALL_W)
    assert int(counts.max()) == m and np.count_nonzero(sums[0]) == 1
    eng.close()


def test_unit_action_sums_are_the_counts():
    w = _workload()
    eng = _engine(w)
    eng.set_packets(*_packets(50021, "random"))                                  # a = NULL: every action is 1
    xe, ye = np.linspace(2.0, 4.0, 33), THETA_EDGES
    sums, counts = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, S.W_ACTION)
    h = eng.hist2(S.Q_KMAG, xe, S.Q_THETA, ye)
    assert np.array_equal(counts, h) and np.array_equal(sums[0], h.astype(np.float64)) and int(h.sum()) > 0
    assert eng.weight_scale(S.W_ACTION).tolist() == [1]
    eng.close()


def test_invariant_under_packet_order_halves_and_devices():
    w = _workload()
    n = 40009
    rs = np.random.RandomState(4)
    x, y, k, l = _packets(n, "random", seed=9)
    a = np.exp2(rs.uniform(-50.0, 0.0, n))
    a[: n // 2] *= 2.0 ** -20                                                     # the halves' own scales differ
    xe, ye, alpha = np.linspace(2.0, 4.0, 41), THETA_EDGES, 0.45
    eng = _engine(w)
    eng.set_packets(x, y, k, l, a)
    whole = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, alpha, return_acc=True)
    exps = eng.weight_scale(ALL_W, alpha)
    p = rs.permutation(n)
    eng.set_packets(x[p], y[p], k[p], l[p], a[p])
    shuffled = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, alpha, return_acc=True)
    for u, v in zip(whole, shuffled):
        assert np.array_equal(u.view(np.int64) if u.dtype == np.float64 else u, v.view(np.int64) if v.dtype == np.float64 else v)
    parts = []
    for sl in (slice(0, n // 2), slice(n // 2, n)):
        eng.set_packets(x[sl], y[sl], k[sl], l[sl], a[sl])
        assert np.all(eng.weight_scale(ALL_W, alpha) <= exps)
        parts.append(eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, alpha, scale_exp=exps, return_acc=True))
    acc = parts[0][2] + parts[1][2]
    assert np.array_equal(acc, whole[2]) and np.array_equal(parts[0][1] + parts[1][1], whole[1])
    assert np.array_equal(_bits(S.fixed_sums_to_double(acc, exps)), _bits(whole[0]))
    eng.close()
    if S.load_library().swrt_device_count() >= 2:
        two = _engine(w, ngpu=2)
        two.set_packets(x, y, k, l, a)
        got = two.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, alpha, return_acc=True)
        assert np.array_equal(two.weight_scale(ALL_W, alpha), exps)
        assert np.array_equal(_bits(got[0]), _bits(whole[0])) and np.array_equal(got[1], whole[1]) and np.array_equal(got[2], whole[2])
        two.close()


def test_edge_cases():
    w = _workload()
    eng = _engine(w, flow=False)
    n = 5003
    x, y, k, l = _packets(n, "random", seed=6)
    a = np.random.RandomState(6).uniform(0.5, 2.0, n)
    xe, ye = np.linspace(2.0, 4.0, 9), np.linspace(-PI, PI, 9)
    # NaN weights: NaN in their own bins only; a packet with NaN or out-of-range coordinates is not counted even when its
    # weight is NaN (k = NaN makes both its |k| and its weights NaN)
    a[10] = np.nan
    a[20] = np.inf
    k[30] = np.nan
    k[40] = 1e6
    a[40] = np.nan
    eng.set_packets(x, y, k, l, a)
    sums, counts, bins, ws = _check_against_mirror(eng, S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W)
    nan_bins = {int(bins[10]), int(bins[20])}
    assert bins[30] == -1 and bins[40] == -1 and bins[10] >= 0 and bins[20] >= 0
    for v in range(4):
        flat = sums[v].ravel(order="F")
        assert set(np.flatnonzero(np.isnan(flat)).tolist()) == nan_bins, v
    assert np.any(sums[2] < 0) and np.any(sums[3] < 0)                            # negative pseudomomentum
    # all-zero weights
    eng.set_packets(x, y, np.where(np.isfinite(k), k, 3.0), l, np.zeros(n))
    s0, c0 = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W)
    assert np.array_equal(_bits(s0), _bits(np.zeros_like(s0))) and int(c0.sum()) > 0
    assert eng.weight_scale(ALL_W).tolist() == [0, 0, 0, 0]
    # a caller's exponent too small for some weights: those are out of range, their bins NaN
    eng.set_packets(x, y, np.where(np.isfinite(k), k, 3.0), l, np.full(n, 0.75))
    s1, _ = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, [S.W_ACTION], scale_exp=[0])
    s2, c2 = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, [S.W_ACTION], scale_exp=[-1])
    assert np.array_equal(s1[0], 0.75 * c2.astype(np.float64)) and np.all(np.isnan(s2[0][c2 > 0])) and np.all(s2[0][c2 == 0] == 0)
    eng.close()


def test_refusals_leave_the_handle_usable():
    w = _workload()
    eng = _engine(w)
    eng.set_packets(*_packets(5003, "random"), a=np.full(5003, 0.5))
    lib, h = eng.lib, eng._h
    xe, ye = np.linspace(2.0, 4.0, 33), THETA_EDGES
    before = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, 0.2, return_acc=True)
    dp = lambda v: v.ctypes.data_as(C.POINTER(C.c_double))                        # noqa: E731
    ip = lambda v: v.ctypes.data_as(C.POINTER(C.c_int32))                         # noqa: E731
    sums = np.zeros(4 * 32 * 36)
    wk = np.array(ALL_W + [0], dtype=np.int32)
    bad_kind = np.array([0, 4], dtype=np.int32)
    neg_kind = np.array([-1], dtype=np.int32)
    e_lo, e_hi = np.array([-1074], dtype=np.int32), np.array([1025], dtype=np.int32)
    dec = xe.copy(); dec[5] = dec[4] - 1e-12
    calls = [(S.Q_KMAG, dp(xe), 33, ip(wk), 0, None), (S.Q_KMAG, dp(xe), 33, ip(wk), 5, None),
             (S.Q_KMAG, dp(xe), 33, ip(bad_kind), 2, None), (S.Q_KMAG, dp(xe), 33, ip(neg_kind), 1, None),
             (S.Q_KMAG, dp(xe), 33, None, 1, None), (S.Q_KMAG, dp(xe), 33, ip(wk), 1, ip(e_lo)),
             (S.Q_KMAG, dp(xe), 33, ip(wk), 1, ip(e_hi)), (8, dp(xe), 33, ip(wk), 1, None),
             (S.Q_KMAG, dp(dec), 33, ip(wk), 1, None), (S.Q_KMAG, dp(xe), 1, ip(wk), 1, None), (S.Q_KMAG, None, 33, ip(wk), 1, None)]
    for qx, xp, nxe, wp, nw, ep in calls:
        assert lib.swrt_hist2_sums(h, qx, xp, nxe, S.Q_THETA, dp(ye), 37, 0.2, wp, nw, ep, dp(sums), None, None) == -1
    out = np.zeros(4, dtype=np.int32)
    assert lib.swrt_weight_scale(h, ip(wk), 0, 0.0, ip(out)) == -1 and lib.swrt_weight_scale(h, ip(bad_kind), 2, 0.0, ip(out)) == -1
    assert lib.swrt_weight_scale(h, ip(wk), 1, 0.0, None) == -1
    after = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, 0.2, return_acc=True)
    for u, v in zip(before, after):
        assert np.array_equal(u, v)
    eng.close()


def test_state_refusals():
    """OMEGA_ABS needs a flow; the energy weight needs omega but no flow"""
    w = _workload()
    bare = _engine(w, flow=False)
    bare.set_packets(*_packets(1001, "random"))
    with pytest.raises(S.SwrtError) as ei:
        bare.hist2_sums(S.Q_OMEGA_ABS, np.linspace(0, 9, 5), S.Q_THETA, THETA_EDGES, S.W_ACTION)
    assert ei.value.code == -2
    s, c = bare.hist2_sums(S.Q_KMAG, np.linspace(2.0, 4.0, 5), S.Q_THETA, THETA_EDGES, S.W_ENERGY)
    assert int(c.sum()) > 0 and np.all(s[0][c > 0] > 0)
    assert bare.weight_scale(S.W_ENERGY)[0] > 0
    bare.close()


@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    return Mex(request.param)


def test_mex_hist2_sums_equals_the_engine(mex):
    w = _workload(3001)
    pk = _packets(3001, "random", seed=12)
    a = np.random.RandomState(12).uniform(0.5, 2.0, 3001)
    xe, ye = np.linspace(2.0, 4.0, 17), THETA_EDGES
    h = mex("create", float(w.nx), w.L, w.f, w.gH, 0.0)
    mex("set_flow_spectral", h, 0.0, w.psik, w.u_mean, nlhs=0)
    mex("set_flow_spectral", h, 1.0, w.psik2, w.u_mean, nlhs=0)
    mex("set_packets", h, *pk, a, nlhs=0)
    Sm, N = mex("hist2_sums", h, float(S.Q_KMAG), xe, float(S.Q_THETA), ye, np.array(ALL_W, dtype=np.float64), 0.4, nlhs=2)
    S1 = mex("hist2_sums", h, float(S.Q_OMEGA_ABS), np.linspace(2.0, 9.0, 9), float(S.Q_THETA), ye, np.array([1.0]), 0.4)
    mex("destroy", h, nlhs=0)
    eng = _engine(w)
    eng.set_packets(*pk, a)
    sums, counts = eng.hist2_sums(S.Q_KMAG, xe, S.Q_THETA, ye, ALL_W, 0.4)
    assert Sm.shape == (16, 36 * 4) and N.shape == (16, 36)
    assert np.array_equal(_bits(Sm.reshape((16, 36, 4), order="F")), _bits(sums.transpose(1, 2, 0)))
    assert np.array_equal(N, counts.astype(np.float64))
    s1, _ = eng.hist2_sums(S.Q_OMEGA_ABS, np.linspace(2.0, 9.0, 9), S.Q_THETA, ye, S.W_ENERGY, 0.4)
    assert S1.shape == (8, 36) and np.array_equal(_bits(S1), _bits(s1[0]))
    eng.close()
