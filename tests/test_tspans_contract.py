"""Per-packet time spans on the CPU: the Python side of swrt_ode23_packets_tspans without a device.  Engine.ode23_packets
runs on a stand-in handle whose library records the C call, so the shape rules, the refusals (raised before any device
call) and the memory layout handed to C are checked here; ShardedEnsemble.ode23 must hand each rank its own columns."""
from types import SimpleNamespace

import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from swraytracing_b200.distributed import ShardedEnsemble, shard_range


class RecordingLib:
    """the C functions Engine.ode23_packets calls, recording their tspan as the C side would read it"""

    def __init__(self, n):
        self.n, self.calls = n, []

    def _call(self, name, tspan_ptr, nt, *rest):
        self.calls.append((name, np.ctypeslib.as_array(tspan_ptr, shape=(nt * (self.n if name.endswith("tspans") else 1),)).copy(), nt))
        return 0

    def __getattr__(self, name):
        if not name.startswith("swrt_ode23_packets"):
            raise AttributeError(name)
        return lambda h, ts, nt, *rest: self._call(name, ts, nt, *rest)


def fake_engine(n):
    return SimpleNamespace(n=n, _h=None, lib=RecordingLib(n), _check=lambda rc: None)


def test_two_dimensional_tspan_selects_the_per_packet_entry_point():
    n, nt = 5, 4
    ts = np.arange(nt * n, dtype=np.float64).reshape(nt, n) * 0.1           # [j, i] = time j of packet i
    e = fake_engine(n)
    out = S.Engine.ode23_packets(e, ts, 0.4)
    (name, seen, ntspan), = e.lib.calls
    assert name == "swrt_ode23_packets_tspans" and ntspan == nt
    # C reads entry j of packet i at tspan[j*n + i]
    assert all(seen[j * n + i] == ts[j, i] for j in range(nt) for i in range(n))
    assert out["Y"].shape == (nt, 4, n) and np.array_equal(out["t"], ts[-1])


def test_fortran_ordered_tspan_is_laid_out_for_c():
    n, nt = 3, 2
    ts = np.asfortranarray(np.array([[0.0, 0.1, 0.2], [1.0, 0.5, 0.2]]))
    e = fake_engine(n)
    S.Engine.ode23_packets(e, ts, None)
    (_, seen, _), = e.lib.calls
    assert np.array_equal(seen, ts.ravel(order="C"))


def test_one_dimensional_tspan_keeps_the_shared_path():
    e = fake_engine(5)
    out = S.Engine.ode23_packets(e, [0.0, 0.4], 0.4)
    (name, seen, nt), = e.lib.calls
    assert name == "swrt_ode23_packets" and nt == 2 and np.array_equal(seen, [0.0, 0.4]) and out["t"] == 0.4


@pytest.mark.parametrize("shape", [(2, 4), (2, 6), (1, 5), (2, 5, 1)])
def test_wrong_shapes_are_refused_before_any_device_call(shape):
    e = fake_engine(5)
    with pytest.raises(ValueError):
        S.Engine.ode23_packets(e, np.zeros(shape), 0.4)
    assert e.lib.calls == []


def test_per_packet_tspan_with_events_is_refused():
    e = fake_engine(5)
    with pytest.raises(ValueError, match="events"):
        S.Engine.ode23_packets(e, np.zeros((3, 5)), 0.4, events=[(S.EVENT_X, 0.0)])
    assert e.lib.calls == []


class RecordingTarget:
    """an Engine stand-in that records what reference_api.ode23 asks of it"""

    def __init__(self, n):
        self.n, self.seen = n, []

    def ode23_packets(self, tspan, tmax, rtol=1e-3, atol=1e-6, events=None, ev_cap=4):
        self.seen.append(np.array(tspan))
        return {"steps": np.zeros(self.n, dtype=np.int32)}

    def __getattr__(self, name):            # anything else (ode23, bs23_*, get_packets) is a device call
        raise AssertionError(f"device call {name}")


@pytest.mark.parametrize("on_device", [False, True])
def test_coupled_solve_refuses_a_per_packet_tspan(on_device):
    t = RecordingTarget(4)
    with pytest.raises(ValueError, match="per_packet"):
        R.ode23(t, np.zeros((2, 4)), 0.4, on_device=on_device)
    with pytest.raises(ValueError, match="per_packet"):
        R.ode23(t, np.zeros((2, 4)), 0.4, reduce_max=lambda v: v)
    assert t.seen == []


def test_reference_api_passes_a_per_packet_tspan_through():
    t = RecordingTarget(4)
    ts = np.array([[0.0, 0.1, 0.2, 0.3], [0.4, 0.0, 0.2, 0.5]])
    R.ode23(t, ts, 0.4, per_packet=True)
    assert len(t.seen) == 1 and np.array_equal(t.seen[0], ts)


@pytest.mark.parametrize("world", [1, 2, 3])
def test_sharded_ensemble_hands_each_rank_its_columns(world):
    n_total = 11
    ts = np.stack([np.arange(n_total) * 0.01, 1.0 + np.arange(n_total) * 0.1])
    for rank in range(world):
        t = RecordingTarget(0)
        ens = ShardedEnsemble(t, n_total, rank, world)
        ens.ode23(ts, 1.0, per_packet=True)
        lo, hi = shard_range(n_total, rank, world)
        assert len(t.seen) == 1 and np.array_equal(t.seen[0], ts[:, lo:hi])


def test_sharded_ensemble_refuses_a_tspan_of_the_wrong_width():
    t = RecordingTarget(0)
    ens = ShardedEnsemble(t, 10, 0, 2)
    with pytest.raises(ValueError):
        ens.ode23(np.zeros((2, 9)), 1.0, per_packet=True)
    with pytest.raises(ValueError, match="per_packet"):
        ens.ode23(np.zeros((2, 10)), 1.0)
    assert t.seen == []
