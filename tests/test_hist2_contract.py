"""Two-dimensional packet histograms on the CPU: the Python side of swrt_packet_quantity / swrt_hist2 without a device.
Engine.hist2 and Engine.packet_quantity run on a stand-in handle whose library plays the C side, so the memory layout
handed to C (counts[i + j*(nxe-1)] = N(i, j)), accumulation and the refusals raised before any device call are checked
here; ShardedEnsemble.hist2 on a gloo 2-rank world must equal one rank.  ``histcounts2`` below is the host restatement of
the bin rule that the GPU tests (tests/test_hist2.py) hold the device to."""
import os
import re
import socket
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200.distributed import ShardedEnsemble, shard_range

ROOT = Path(__file__).resolve().parent.parent


def bin_of(v, edges):
    """the bin of every v on one axis (-1: NaN or out of range): the last a with e[a] <= v, v == e[-1] in the last bin"""
    v = np.asarray(v, dtype=np.float64)
    e = np.asarray(edges, dtype=np.float64)
    nb = e.size - 1
    ok = (v >= e[0]) & (v <= e[-1])
    a = np.minimum(np.searchsorted(e, np.where(ok, v, e[0]), side="right") - 1, nb - 1)
    return np.where(ok, a, -1)


def histcounts2(qx, qy, xedges, yedges):
    """MATLAB's histcounts2(Qx, Qy, xedges, yedges) -> (nxe-1, nye-1) uint64"""
    bx, by = bin_of(qx, xedges), bin_of(qy, yedges)
    keep = (bx >= 0) & (by >= 0)
    nbx, nby = len(xedges) - 1, len(yedges) - 1
    flat = np.bincount(bx[keep] + by[keep] * nbx, minlength=nbx * nby)
    return flat.reshape((nbx, nby), order="F").astype(np.uint64)


def test_histcounts2_restatement_bin_rule():
    e = [0.0, 1.0, 1.0, 2.0, 3.0]                   # a repeated edge: [1, 1) is empty, 1 goes to [1, 2)
    assert list(bin_of([0.0, 0.5, 1.0, 2.0, 2.5, 3.0, 3.5, -0.1, np.nan], e)) == [0, 0, 2, 3, 3, 3, -1, -1, -1]
    N = histcounts2([0.0, 3.0, 3.0, np.nan, 1.0], [0.0, 1.0, 0.5, 0.0, 9.0], e, [0.0, 0.5, 1.0])
    assert N.shape == (4, 2) and N.dtype == np.uint64
    assert N[0, 0] == 1 and N[3, 1] == 2 and N.sum() == 3


def test_quantity_constants_match_the_header():
    text = (ROOT / "include" / "swrt.h").read_text()
    defs = dict((m.group(1), int(m.group(2))) for m in re.finditer(r"#define SWRT_(Q_\w+)\s+(\d+)", text))
    assert len(defs) == 8
    for name, val in defs.items():
        assert getattr(S, name) == val, name
        assert name in S.__all__


class Hist2Lib:
    """swrt_hist2 / swrt_packet_quantity as the C side sees them: counts[i + j*(nxe-1)] gets i + 1000*j (+ the old value
    when accumulating), out[i] gets q + i"""

    def __init__(self):
        self.calls = []

    def swrt_hist2(self, h, qx, xe, nxe, qy, ye, nye, alpha, counts, acc):
        self.calls.append((qx, np.ctypeslib.as_array(xe, shape=(nxe,)).copy(), qy, np.ctypeslib.as_array(ye, shape=(nye,)).copy(),
                           alpha, acc))
        if nxe < 2 or nye < 2:
            return -1
        c = np.ctypeslib.as_array(counts, shape=((nxe - 1) * (nye - 1),))
        for j in range(nye - 1):
            for i in range(nxe - 1):
                c[i + j * (nxe - 1)] = (c[i + j * (nxe - 1)] if acc else 0) + i + 1000 * j
        return 0

    def swrt_packet_quantity(self, h, q, alpha, out):
        self.calls.append((q, alpha))
        o = np.ctypeslib.as_array(out, shape=(5,))
        o[:] = q + np.arange(5)
        return 0

    def swrt_last_error(self, h):
        return b"stand-in"


def fake_engine(n=5):
    lib = Hist2Lib()
    eng = SimpleNamespace(n=n, _h=None, lib=lib)
    eng._check = lambda rc: S.Engine._check(eng, rc)
    return eng


def test_hist2_layout_is_column_major_n_of_i_j():
    e = fake_engine()
    xe, ye = [0, 1, 2, 3], np.linspace(-1.0, 1.0, 11)[::2]           # ints, and a strided view
    N = S.Engine.hist2(e, S.Q_KMAG, xe, S.Q_THETA, ye, alpha=0.25)
    assert N.shape == (3, 5) and N.dtype == np.uint64
    assert all(N[i, j] == i + 1000 * j for i in range(3) for j in range(5))
    (qx, sx, qy, sy, alpha, acc), = e.lib.calls
    assert (qx, qy, alpha, acc) == (S.Q_KMAG, S.Q_THETA, 0.25, 0)
    assert np.array_equal(sx, [0.0, 1.0, 2.0, 3.0]) and np.array_equal(sy, np.linspace(-1.0, 1.0, 6))


@pytest.mark.parametrize("order", ["C", "F"])
def test_hist2_accumulates_into_the_given_counts(order):
    e = fake_engine()
    counts = np.full((2, 3), 7, dtype=np.uint64, order=order)
    out = S.Engine.hist2(e, S.Q_XMOD, [0, 1, 2], S.Q_YMOD, [0, 1, 2, 3], counts=counts)
    assert out is counts and e.lib.calls[0][-1] == 1
    assert all(counts[i, j] == 7 + i + 1000 * j for i in range(2) for j in range(3))


@pytest.mark.parametrize("bad", [np.zeros((3, 2), dtype=np.uint64), np.zeros((2, 3), dtype=np.int64), [[0, 0, 0], [0, 0, 0]]])
def test_hist2_refuses_counts_of_the_wrong_shape_or_type_before_any_call(bad):
    e = fake_engine()
    with pytest.raises(ValueError):
        S.Engine.hist2(e, S.Q_XMOD, [0, 1, 2], S.Q_YMOD, [0, 1, 2, 3], counts=bad)
    assert e.lib.calls == []


def test_hist2_library_refusal_raises():
    e = fake_engine()
    with pytest.raises(S.SwrtError) as ei:
        S.Engine.hist2(e, S.Q_XMOD, [0.0], S.Q_YMOD, [0, 1])
    assert ei.value.code == -1


def test_packet_quantity_returns_one_value_per_packet():
    e = fake_engine(5)
    q = S.Engine.packet_quantity(e, S.Q_OMEGA_ABS, alpha=0.5)
    assert e.lib.calls == [(S.Q_OMEGA_ABS, 0.5)] and np.array_equal(q, S.Q_OMEGA_ABS + np.arange(5.0))


class QuantityEngine:
    """an Engine stand-in that bins its shard's packets with the host restatement"""

    def set_packets(self, x, y, k, l, a=None):
        self.s = [np.asarray(v, dtype=np.float64) for v in (x, y, k, l)]

    def hist2(self, qx, xedges, qy, yedges, alpha=0.0):
        q = {S.Q_K: self.s[2], S.Q_L: self.s[3], S.Q_KMAG: np.sqrt(self.s[2] * self.s[2] + self.s[3] * self.s[3]),
             S.Q_THETA: np.arctan2(self.s[3], self.s[2])}
        return histcounts2(q[qx], q[qy], xedges, yedges)


def _packets(n=1001):
    rs = np.random.RandomState(3)
    th = rs.uniform(-np.pi, np.pi, n)
    kmag = 3.0 + 0.2 * rs.randn(n)
    k, l = kmag * np.cos(th), kmag * np.sin(th)
    k[::97] = np.nan                                 # blown-up packets are dropped on every rank
    return rs.uniform(0, 1, n), rs.uniform(0, 1, n), k, l


XE, YE = np.linspace(2.0, 4.0, 17), np.linspace(-np.pi, np.pi, 33)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    x, y, k, l = _packets()
    ens = ShardedEnsemble(QuantityEngine(), x.size, rank, world, dist)
    ens.set_packets_global(x, y, k, l)
    N = ens.hist2(S.Q_KMAG, XE, S.Q_THETA, YE)
    local = ens.engine.hist2(S.Q_KMAG, XE, S.Q_THETA, YE)
    np.save(f"{out}.{rank}.npy", np.stack([N, local]))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_hist2_two_gloo_ranks_equal_one_rank(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "h2")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    x, y, k, l = _packets()
    one = ShardedEnsemble(QuantityEngine(), x.size)
    one.set_packets_global(x, y, k, l)
    ref = one.hist2(S.Q_KMAG, XE, S.Q_THETA, YE)
    assert ref.dtype == np.uint64 and ref.shape == (16, 32) and 0 < int(ref.sum()) < x.size
    parts = [np.load(f"{out}.{r}.npy") for r in range(2)]
    for r in range(2):
        assert np.array_equal(parts[r][0], ref)                        # every rank holds the global counts, bit-exact
    assert np.array_equal(parts[0][1] + parts[1][1], ref)              # and they are the sum of the two shards' own
    assert shard_range(x.size, 1, 2)[0] > 0 and parts[0][1].sum() > 0 and parts[1][1].sum() > 0
