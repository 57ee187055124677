"""Per-bin weighted sums on the CPU: the fixed-point contract of swrt_weight_scale / swrt_hist2_sums without a device.
swrt_fixed_sums_to_double (host only) against Python's exact Fraction arithmetic; a numpy mirror of the device's
quantization and digit split (``quantize``, ``mirror_acc``: what tests/test_hist2_sums.py holds the device to); the Python
layer's layout and refusals on a stand-in library; and ShardedEnsemble.hist2_sums on a gloo 2-rank world."""
import ctypes as C
import os
import socket
from fractions import Fraction
from types import SimpleNamespace

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200.distributed import ShardedEnsemble, shard_range
from test_hist2_contract import bin_of

TWO95 = 2.0 ** 95


def scale_exp_of(w):
    """the least E with |w| < 2^E over the finite weights (0 when none is finite and non-zero)"""
    a = np.abs(np.asarray(w, dtype=np.float64))
    a = a[np.isfinite(a)]
    m = a.max() if a.size else 0.0
    return int(np.frexp(m)[1]) if m > 0 else 0


def quantize(w, E):
    """the device's steps: |q| = rint(|w| 2^s1 2^s2) (s1 + s2 = 95 - E), digits of |q| by exact fp64 operations, signed
    like w -> (int64 digits (n, 3), bad (n,)): bad = not finite or |w| >= 2^E"""
    w = np.asarray(w, dtype=np.float64)
    s = 95 - E
    s1 = s >> 1
    with np.errstate(invalid="ignore", over="ignore"):
        qd = (np.abs(w) * np.ldexp(1.0, s1)) * np.ldexp(1.0, s - s1)
        bad = ~(qd < TWO95)
        q = np.rint(np.where(bad, 0.0, qd))
    h2 = np.floor(q * 2.0 ** -64)
    r = q - h2 * 2.0 ** 64
    h1 = np.floor(r * 2.0 ** -32)
    h0 = r - h1 * 2.0 ** 32
    d = np.stack([h0, h1, h2], axis=1).astype(np.int64)
    return np.where((w < 0)[:, None], -d, d), bad


def mirror_acc(bins, w, E, nb):
    """the accumulators (nb, 4) of one weight kind: digits and bad counts added per bin (bin -1: not counted)"""
    d, bad = quantize(w, E)
    keep = np.asarray(bins) >= 0
    acc = np.zeros((nb, 4), dtype=np.int64)
    for c in range(3):
        np.add.at(acc[:, c], bins[keep], d[keep, c])
    np.add.at(acc[:, 3], bins[keep], bad[keep].astype(np.int64))
    return acc


def exact_double(S_int, E):
    """float(Fraction(S) 2^(E-95)), correctly rounded; +-inf past the largest double"""
    f = Fraction(S_int) * Fraction(2) ** (E - 95)
    try:
        return float(f)
    except OverflowError:
        return float("inf") if f > 0 else float("-inf")


def _finish(acc, E):
    """swrt_fixed_sums_to_double through ctypes on (m, 4) accumulators of one kind"""
    acc = np.ascontiguousarray(acc, dtype=np.int64)
    out = np.full(acc.shape[0], 12345.0)
    e = np.array([E], dtype=np.int32)
    rc = S.load_library().swrt_fixed_sums_to_double(acc.ctypes.data_as(C.POINTER(C.c_int64)), acc.shape[0], 1,
                                                    e.ctypes.data_as(C.POINTER(C.c_int32)), out.ctypes.data_as(C.POINTER(C.c_double)))
    assert rc == 0
    return out


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _check_finish(acc, E):
    got = _finish(acc, E)
    for row, g in zip(acc, got):
        if row[3]:
            assert np.isnan(g), row
            continue
        want = exact_double(int(row[0]) + (int(row[1]) << 32) + (int(row[2]) << 64), E)
        assert _bits([g])[0] == _bits([want])[0], (list(row), E, g, want)


I64 = np.iinfo(np.int64)


def test_fixed_sums_to_double_equals_the_correctly_rounded_fraction_on_random_accumulators():
    rs = np.random.RandomState(11)
    for E in (0, 1, -7, 52, 95, 96, 200, -300, -1000, -1073, 1024, 900):
        acc = np.zeros((400, 4), dtype=np.int64)
        acc[:, :3] = rs.randint(I64.min, I64.max, size=(400, 3), dtype=np.int64)
        acc[100:200, :3] >>= rs.randint(0, 63, size=(100, 3))                      # every magnitude
        acc[200:300, 2] = 0
        acc[250:300, 1] = 0
        acc[300:310, 3] = 1                                                        # non-finite weights: NaN
        _check_finish(acc, E)


def test_fixed_sums_to_double_adversarial_cases():
    two32 = 1 << 32
    rows, exps = [], []

    def add(c0, c1, c2, E):
        rows.append([c0, c1, c2, 0]); exps.append(E)

    for E in (95, 0, -1000, -1073, 1024):
        add(0, 0, 0, E)
        add(-1, 0, 0, E); add(1, 0, 0, E)
        add(two32 - 1, two32 - 1, 0, E); add(two32, -1, 0, E)                     # carries between digits
        add(-two32, 1, 0, E); add(0, -two32, 1, E)                                 # exactly zero through carries
        add(I64.max, I64.max, I64.max, E); add(I64.min, I64.min, I64.min, E)       # the extremes
        add(I64.min, 0, 0, E); add(0, 0, I64.min, E); add(I64.max, I64.min, I64.max, E)
    # exact halfway cases at 53 bits: 2^53 + 1 (tie, even down), 2^53 + 3 (tie, even up), and the values beside them
    for base in ((1 << 53) + 1, (1 << 53) + 3, (1 << 54) + 2, (1 << 54) + 6):
        for sgn in (1, -1):
            for eps in (0, 1, -1):
                v = sgn * ((base << 20) + eps)
                add(v & (two32 - 1), (v >> 32) & (two32 - 1), v >> 64, 95)
    # subnormal results: E = -1033 puts bit 0 at 2^-1128; the quantum there is 2^-1074 = 2^54 units, 2^-1022 is 2^106
    for v in (1 << 54, (1 << 54) - 1, 1 << 53, (1 << 53) + 1, 3 << 53, 5 << 52, (1 << 106) + (1 << 53), (1 << 106) - 1, 7):
        for sgn in (1, -1):
            add(sgn * v & (two32 - 1), (sgn * v >> 32) & (two32 - 1), sgn * v >> 64, -1033)
    # overflow: E = 1024 puts bit 0 at 2^929; DBL_MAX = (2^53 - 1) 2^971, half an ulp above it is a tie that goes to inf
    mx = ((1 << 53) - 1) << 42
    for v in (mx, mx + (1 << 41) - 1, mx + (1 << 41), 1 << 95, (1 << 96) + 5):
        for sgn in (1, -1):
            add(sgn * v & (two32 - 1), (sgn * v >> 32) & (two32 - 1), sgn * v >> 64, 1024)
    for row, E in zip(rows, exps):
        _check_finish(np.array([row], dtype=np.int64), E)
    mxrow = np.array([[mx & (two32 - 1), (mx >> 32) & (two32 - 1), mx >> 64, 0]], dtype=np.int64)
    assert _finish(mxrow, 1024)[0] == np.finfo(np.float64).max
    tie = mx + (1 << 41)
    assert _finish(np.array([[tie & (two32 - 1), (tie >> 32) & (two32 - 1), tie >> 64, 0]], dtype=np.int64), 1024)[0] == np.inf
    tiny = _finish(np.array([[0, 0, 0, 0], [1, 0, 0, 0], [-1, 0, 0, 0]], dtype=np.int64), -1073)
    assert _bits(tiny).tolist() == _bits([0.0, 0.0, -0.0]).tolist()                # +0 for an exact zero, signed underflow


def test_fixed_sums_to_double_layout_and_refusals():
    lib = S.load_library()
    acc = np.zeros((2, 3, 4), dtype=np.int64)
    acc[0, :, 0] = [1, 2, 3]
    acc[1, :, 0] = [4, 5, 6]
    e = np.array([95, 96], dtype=np.int32)
    out = np.empty(6)
    i64p, i32p, dp = C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_double)
    assert lib.swrt_fixed_sums_to_double(acc.ctypes.data_as(i64p), 3, 2, e.ctypes.data_as(i32p), out.ctypes.data_as(dp)) == 0
    assert out.tolist() == [1.0, 2.0, 3.0, 8.0, 10.0, 12.0]                         # sums[v*nbins + b], kind v at 2^(E_v-95)
    assert lib.swrt_fixed_sums_to_double(None, 3, 2, e.ctypes.data_as(i32p), out.ctypes.data_as(dp)) == -1
    assert lib.swrt_fixed_sums_to_double(acc.ctypes.data_as(i64p), -1, 2, e.ctypes.data_as(i32p), out.ctypes.data_as(dp)) == -1
    # the Python wrapper takes Engine.hist2_sums' (nw, nbx, nby, 4) accumulators
    a4 = np.zeros((2, 3, 2, 4), dtype=np.int64)
    a4[..., 0] = np.arange(12).reshape(2, 3, 2)
    s = S.fixed_sums_to_double(a4, [95, 94])
    assert s.shape == (2, 3, 2) and np.array_equal(s[0], a4[0, ..., 0]) and np.array_equal(s[1], a4[1, ..., 0] / 2.0)
    for bad, e in ((a4.astype(np.int32), [95, 95]), (a4[..., :3], [95, 95]), (a4, [95])):
        with pytest.raises(ValueError):
            S.fixed_sums_to_double(bad, e)


def test_mirror_quantizes_weights_near_the_scale_exactly_and_reproduces_the_integer_sum():
    rs = np.random.RandomState(5)
    for E in (1, 0, -20, 30, 700, -1000):
        top = np.ldexp(1.0, E)
        w = rs.uniform(-1.0, 1.0, 5000) * top
        w[:500] = np.ldexp(rs.uniform(1.0, 2.0, 500), E - 44 + rs.randint(0, 44, 500)) * np.sign(rs.randn(500))  # >= 2^(E-43)
        w[500:510] = [top * (1 - 2.0 ** -53), -top * (1 - 2.0 ** -53), 0.0, -0.0, np.ldexp(1.0, E - 43), np.ldexp(1.0, E - 44),
                      np.ldexp(3.0, E - 97), np.ldexp(1.0, E - 96), np.ldexp(1.0, E - 97), np.ldexp(5.0, E - 98)]
        assert scale_exp_of(w) <= E
        d, bad = quantize(w, E)
        assert not bad.any() and np.all(np.abs(d) < 2 ** 32) and np.all(np.abs(d[:, 2]) <= 2 ** 31)
        q = [int(a) + (int(b) << 32) + (int(c) << 64) for a, b, c in d]
        exact = [Fraction(float(x)) * Fraction(2) ** (95 - E) for x in w]
        for qi, xi, wi in zip(q, exact, w):
            assert qi == round(xi)                                                   # Python's round: half to even
            if abs(wi) >= np.ldexp(1.0, E - 43):
                assert qi == xi                                                      # no rounding at all
            assert abs(qi - xi) <= Fraction(1, 2)
        bins = rs.randint(-1, 7, w.size)
        acc = mirror_acc(bins, w, E, 7)
        for b in range(7):
            assert int(acc[b, 0]) + (int(acc[b, 1]) << 32) + (int(acc[b, 2]) << 64) == sum(qi for qi, bi in zip(q, bins) if bi == b)
    d, bad = quantize(np.array([np.nan, np.inf, -np.inf, 2.0, 1.0, 0.999]), 1)
    assert bad.tolist() == [True, True, True, True, False, False]                    # not finite, or |w| >= 2^E


def test_scale_exp_of_is_the_least_power_of_two_above_every_finite_weight():
    assert scale_exp_of([0.5, -0.25]) == 0 and scale_exp_of([1.0]) == 1 and scale_exp_of([-3.0, np.nan, np.inf]) == 2
    assert scale_exp_of([0.0, np.nan]) == 0 and scale_exp_of([5e-324]) == -1073 and scale_exp_of([1.7e308]) == 1024


# ---- the Python layer on a stand-in library ----------------------------------------------------------------------------
class SumsLib:
    """swrt_hist2_sums / swrt_weight_scale as the C side sees them: sums[(v*nby + j)*nbx + i] = v + 10 i + 1000 j,
    counts[j*nbx + i] = i + 1000 j, acc[4 b + c] = 4 b + c; scale_exp[v] = kind + 7"""

    def __init__(self):
        self.calls = []

    def swrt_hist2_sums(self, h, qx, xe, nxe, qy, ye, nye, alpha, w, nw, e, sums, counts, acc):
        kinds = np.ctypeslib.as_array(w, shape=(nw,)).copy()
        self.calls.append((qx, qy, alpha, kinds, None if not e else np.ctypeslib.as_array(e, shape=(nw,)).copy(), bool(acc)))
        nbx, nby = nxe - 1, nye - 1
        s = np.ctypeslib.as_array(sums, shape=(nw * nbx * nby,))
        c = np.ctypeslib.as_array(counts, shape=(nbx * nby,))
        for v in range(nw):
            for j in range(nby):
                for i in range(nbx):
                    s[(v * nby + j) * nbx + i] = v + 10 * i + 1000 * j
                    c[j * nbx + i] = i + 1000 * j
        if acc:
            a = np.ctypeslib.as_array(acc, shape=(4 * nw * nbx * nby,))
            a[:] = np.arange(a.size)
        return 0

    def swrt_weight_scale(self, h, w, nw, alpha, e):
        kinds = np.ctypeslib.as_array(w, shape=(nw,))
        self.calls.append(("scale", kinds.copy(), alpha))
        np.ctypeslib.as_array(e, shape=(nw,))[:] = kinds + 7
        return 0

    def swrt_last_error(self, h):
        return b"stand-in"


def fake_engine():
    eng = SimpleNamespace(n=5, _h=None, lib=SumsLib())
    eng._check = lambda rc: S.Engine._check(eng, rc)
    return eng


def test_hist2_sums_layout():
    e = fake_engine()
    sums, counts, acc = S.Engine.hist2_sums(e, S.Q_KMAG, [0, 1, 2, 3], S.Q_THETA, np.linspace(-1, 1, 5),
                                            [S.W_ENERGY, S.W_PSEUDO_K], alpha=0.5, return_acc=True)
    assert sums.shape == (2, 3, 4) and counts.shape == (3, 4) and acc.shape == (2, 3, 4, 4)
    assert sums.dtype == np.float64 and counts.dtype == np.uint64 and acc.dtype == np.int64
    assert all(sums[v, i, j] == v + 10 * i + 1000 * j for v in range(2) for i in range(3) for j in range(4))
    assert all(counts[i, j] == i + 1000 * j for i in range(3) for j in range(4))
    assert all(acc[v, i, j, c] == 4 * ((v * 4 + j) * 3 + i) + c for v in range(2) for i in range(3) for j in range(4) for c in range(4))
    (qx, qy, alpha, kinds, exps, want_acc), = e.lib.calls
    assert (qx, qy, alpha, exps, want_acc) == (S.Q_KMAG, S.Q_THETA, 0.5, None, True) and kinds.tolist() == [1, 2]
    s1, c1 = S.Engine.hist2_sums(e, S.Q_XMOD, [0, 1], S.Q_YMOD, [0, 1], S.W_ACTION, scale_exp=[-3])
    assert s1.shape == (1, 1, 1) and c1.shape == (1, 1)
    assert e.lib.calls[-1][4].tolist() == [-3] and e.lib.calls[-1][5] is False
    assert S.Engine.weight_scale(e, (S.W_PSEUDO_L, S.W_ACTION), 0.25).tolist() == [10, 7]


@pytest.mark.parametrize("weights,scale_exp", [([], None), ([0, 1, 2, 3, 0], None), ([4], None), ([-1], None), ([0.5], None),
                                               ([[0, 1]], None), ([0, 1], [3]), ([0], [1, 2])])
def test_hist2_sums_refuses_bad_weights_before_any_call(weights, scale_exp):
    e = fake_engine()
    with pytest.raises(ValueError):
        S.Engine.hist2_sums(e, S.Q_XMOD, [0, 1, 2], S.Q_YMOD, [0, 1], weights, scale_exp=scale_exp)
    if scale_exp is None:
        with pytest.raises(ValueError):
            S.Engine.weight_scale(e, weights)
    assert e.lib.calls == []


def test_weight_constants_match_the_header():
    import re
    from pathlib import Path
    text = (Path(__file__).resolve().parent.parent / "include" / "swrt.h").read_text()
    defs = dict((m.group(1), int(m.group(2))) for m in re.finditer(r"#define SWRT_(W_\w+|MAX_WEIGHTS)\s+(\d+)", text))
    assert defs == {"W_ACTION": 0, "W_ENERGY": 1, "W_PSEUDO_K": 2, "W_PSEUDO_L": 3, "MAX_WEIGHTS": 4}
    for name, val in defs.items():
        assert getattr(S, name) == val and name in S.__all__


# ---- ShardedEnsemble.hist2_sums on gloo ---------------------------------------------------------------------------------
class WeightEngine:
    """an Engine stand-in: its shard's |k| x theta bins and weights through the numpy mirror"""

    def set_packets(self, x, y, k, l, a=None):
        self.k, self.l = np.asarray(k, dtype=np.float64), np.asarray(l, dtype=np.float64)
        self.a = np.ones_like(self.k) if a is None else np.asarray(a, dtype=np.float64)

    def _w(self, kind):
        return {S.W_ACTION: self.a, S.W_PSEUDO_K: self.k * self.a, S.W_PSEUDO_L: self.l * self.a}[kind]

    def weight_scale(self, weights, alpha=0.0):
        return np.array([scale_exp_of(self._w(v)) for v in np.atleast_1d(weights)], dtype=np.int32)

    def hist2_sums(self, qx, xedges, qy, yedges, weights, alpha=0.0, scale_exp=None, return_acc=False):
        assert (qx, qy, return_acc) == (S.Q_KMAG, S.Q_THETA, True) and scale_exp is not None
        nbx, nby = len(xedges) - 1, len(yedges) - 1
        bx = bin_of(np.sqrt(self.k * self.k + self.l * self.l), xedges)
        by = bin_of(np.arctan2(self.l, self.k), yedges)
        bins = np.where((bx >= 0) & (by >= 0), bx + by * nbx, -1)
        kinds = np.atleast_1d(weights)
        acc = np.stack([mirror_acc(bins, self._w(v), int(E), nbx * nby) for v, E in zip(kinds, scale_exp)])
        acc = acc.reshape(len(kinds), nby, nbx, 4).transpose(0, 2, 1, 3)
        counts = np.bincount(bins[bins >= 0], minlength=nbx * nby).reshape((nbx, nby), order="F").astype(np.uint64)
        return S.fixed_sums_to_double(acc, scale_exp), counts, acc


def _packets(n=1003):
    rs = np.random.RandomState(8)
    th = rs.uniform(-np.pi, np.pi, n)
    kmag = 3.0 + 0.2 * rs.randn(n)
    k, l = kmag * np.cos(th), kmag * np.sin(th)
    a = np.exp2(rs.uniform(-30, 0, n))
    a[: n // 2] *= 1e-6                                                 # the two halves' largest weights differ
    k[::97] = np.nan
    return rs.uniform(0, 1, n), rs.uniform(0, 1, n), k, l, a


XE, YE = np.linspace(2.0, 4.0, 9), np.linspace(-np.pi, np.pi, 17)
WK = [S.W_ACTION, S.W_PSEUDO_K, S.W_PSEUDO_L]


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    x, y, k, l, a = _packets()
    ens = ShardedEnsemble(WeightEngine(), x.size, rank, world, dist)
    ens.set_packets_global(x, y, k, l, a)
    s, c = ens.hist2_sums(S.Q_KMAG, XE, S.Q_THETA, YE, WK)
    np.save(f"{out}.{rank}.npy", np.concatenate([s.ravel(), c.astype(np.float64).ravel()]))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_hist2_sums_two_gloo_ranks_equal_one_rank(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "h2s")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    x, y, k, l, a = _packets()
    one = ShardedEnsemble(WeightEngine(), x.size)
    one.set_packets_global(x, y, k, l, a)
    s, c = one.hist2_sums(S.Q_KMAG, XE, S.Q_THETA, YE, WK)
    assert s.shape == (3, 8, 16) and int(c.sum()) > 0 and np.all(s[0][c > 0] > 0) and np.any(s[1] < 0)
    ref = np.concatenate([s.ravel(), c.astype(np.float64).ravel()])
    lo = shard_range(x.size, 1, 2)[0]
    assert np.max(np.abs(a[:lo])) < np.max(np.abs(a[lo:])) * 1e-5                  # the halves' own scales differ
    for r in range(2):
        assert np.array_equal(_bits(np.load(f"{out}.{r}.npy")), _bits(ref))
