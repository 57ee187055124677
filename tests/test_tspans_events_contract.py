"""Events with a tspan per packet, on the CPU: the Python side of swrt_ode23_packets_tspans_events without a device.
Engine.ode23_packets_tspans_events runs on a stand-in handle whose library records the C call, so the 1-D broadcast, the
n x ntspan layout handed to C, the refusals (raised before any call) and the event tuples are checked here;
ShardedEnsemble.ode23_packets_tspans_events must hand each rank its own columns."""
from types import SimpleNamespace

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200.distributed import ShardedEnsemble, shard_range

EVENTS = [(S.EVENT_X, 0.5), (S.EVENT_OMEGA, 4.3, -1), (S.EVENT_KMAG, 3.0, 1, True)]


class RecordingLib:
    """the C functions the per-packet solves call, recording their tspan as the C side reads it and their events"""

    def __init__(self, n):
        self.n, self.calls = n, []

    def __getattr__(self, name):
        if not name.startswith("swrt_ode23_packets"):
            raise AttributeError(name)

        def call(h, ts, nt, tmax, rtol, atol, ev, nev, cap, *rest):
            size = nt * (self.n if "tspans" in name else 1)
            evs = [(ev[j].kind, ev[j].level, ev[j].direction, ev[j].terminal, ev[j].reserved) for j in range(nev)]
            self.calls.append((name, np.ctypeslib.as_array(ts, shape=(size,)).copy(), nt, evs, cap))
            return 0
        return call


def fake_engine(n):
    e = SimpleNamespace(n=n, _h=None, lib=RecordingLib(n), _check=lambda rc: None)
    e._ode23_events = lambda *a: S.Engine._ode23_events(e, *a)
    return e


def test_two_dimensional_tspan_is_handed_to_c_column_major():
    n, nt = 5, 4
    ts = np.arange(nt * n, dtype=np.float64).reshape(nt, n) * 0.1
    ts[:, 1::2] = ts[::-1, 1::2]                       # every other packet backward
    e = fake_engine(n)
    out = S.Engine.ode23_packets_tspans_events(e, ts, 0.4, EVENTS, ev_cap=3)
    (name, seen, ntspan, _, cap), = e.lib.calls
    assert name == "swrt_ode23_packets_tspans_events" and ntspan == nt and cap == 3
    assert all(seen[j * n + i] == ts[j, i] for j in range(nt) for i in range(n))     # entry j of packet i at j*n + i
    assert out["Y"].shape == (nt, 4, n) and np.array_equal(out["t"], ts[-1])
    assert out["te"].shape == (3, n) and out["ye"].shape == (3, 4, n) and out["ie"].shape == (3, n) and out["ne"].shape == (n,)


def test_fortran_ordered_tspan_is_laid_out_for_c():
    ts = np.asfortranarray(np.array([[0.0, 0.1, 0.2], [1.0, 0.5, 0.2]]))
    e = fake_engine(3)
    S.Engine.ode23_packets_tspans_events(e, ts, None, EVENTS)
    (_, seen, _, _, _), = e.lib.calls
    assert np.array_equal(seen, ts.ravel(order="C"))


@pytest.mark.parametrize("row", [[0.0, 0.4], [0.4, 0.1, 0.0], [0.2, 0.2, 0.2]])
def test_one_dimensional_tspan_is_broadcast_to_every_packet(row):
    n = 6
    e = fake_engine(n)
    out = S.Engine.ode23_packets_tspans_events(e, row, 0.4, EVENTS)
    (name, seen, nt, _, _), = e.lib.calls
    assert name == "swrt_ode23_packets_tspans_events" and nt == len(row)
    assert np.array_equal(seen, np.repeat(row, n)) and np.array_equal(out["t"], np.full(n, row[-1]))


def test_event_tuples_are_packed_as_ode23_packets_packs_them():
    n = 4
    a, b = fake_engine(n), fake_engine(n)
    S.Engine.ode23_packets(a, [0.0, 0.4], 0.4, events=EVENTS, ev_cap=2)
    S.Engine.ode23_packets_tspans_events(b, [0.0, 0.4], 0.4, EVENTS, ev_cap=2)
    (na, _, _, ea, ca), = a.lib.calls
    (nb, _, _, eb, cb), = b.lib.calls
    assert na == "swrt_ode23_packets_events" and nb == "swrt_ode23_packets_tspans_events"
    assert ea == eb == [(S.EVENT_X, 0.5, 0, 0, 0), (S.EVENT_OMEGA, 4.3, -1, 0, 0), (S.EVENT_KMAG, 3.0, 1, 1, 0)] and ca == cb == 2


@pytest.mark.parametrize("shape", [(1,), (2, 4), (2, 6), (1, 5), (2, 5, 1), ()])
def test_wrong_shapes_are_refused_before_any_call(shape):
    e = fake_engine(5)
    with pytest.raises(ValueError):
        S.Engine.ode23_packets_tspans_events(e, np.zeros(shape), 0.4, EVENTS)
    assert e.lib.calls == []


class RecordingTarget:
    """an Engine stand-in that records what ShardedEnsemble asks of it"""

    def __init__(self):
        self.seen = []

    def ode23_packets_tspans_events(self, tspan, tmax, events, rtol=1e-3, atol=1e-6, ev_cap=4):
        self.seen.append((np.array(tspan), events, ev_cap))
        return {}


@pytest.mark.parametrize("world", [1, 2, 3])
def test_sharded_ensemble_hands_each_rank_its_columns(world):
    n_total = 11
    ts = np.stack([np.arange(n_total) * 0.01, 1.0 - np.arange(n_total) * 0.1])
    for rank in range(world):
        t = RecordingTarget()
        ShardedEnsemble(t, n_total, rank, world).ode23_packets_tspans_events(ts, 1.0, EVENTS, ev_cap=5)
        lo, hi = shard_range(n_total, rank, world)
        (seen, evs, cap), = t.seen
        assert np.array_equal(seen, ts[:, lo:hi]) and evs == EVENTS and cap == 5
    t = RecordingTarget()
    ShardedEnsemble(t, n_total, 1, 2).ode23_packets_tspans_events([1.0, 0.0], 1.0, EVENTS)
    assert np.array_equal(t.seen[0][0], [1.0, 0.0])                  # a shared row goes as it is


def test_sharded_ensemble_refuses_a_tspan_of_the_wrong_width():
    t = RecordingTarget()
    with pytest.raises(ValueError):
        ShardedEnsemble(t, 10, 0, 2).ode23_packets_tspans_events(np.zeros((2, 9)), 1.0, EVENTS)
    assert t.seen == []
