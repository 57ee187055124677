"""The gateway's whole-solve commands, executed through tests/mex_harness: swrt_mex('ode23', ...) and
swrt_mex('ode23_packets', ...) against the ctypes path (engine.py), bit for bit, in both complex-storage layouts."""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
from test_mex_gateway import Mex

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=[False, True], ids=["separate-complex", "interleaved-complex"])
def mex(request):
    return Mex(request.param)


def _setup(mex, n, blow_up=False):
    w = W.make_workload("C3", n_packets=n, nx=32)
    k = w.k.copy()
    if blow_up:
        k[3] = np.inf
    h = mex("create", float(w.nx), w.L, w.f, w.gH, float(S.MODE_LAGRANGE6))
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6)
    for slot, psik in ((0.0, w.psik), (1.0, w.psik2)):
        mex("set_flow_spectral", h, slot, psik, nlhs=0)
        eng.set_flow_spectral(psik, int(slot))
    mex("set_packets", h, w.x, w.y, k, w.l, nlhs=0)
    eng.set_packets(w.x, w.y, k, w.l)
    return w, h, eng


def test_gateway_ode23(mex):
    w, h, eng = _setup(mex, 301)
    tspan = w.dt * np.linspace(0.0, 1.0, 6)
    st, Y = mex("ode23", h, tspan, w.dt, 1e-6, 1e-7, nlhs=2)
    ref = eng.ode23(tspan, w.dt, 1e-6, 1e-7)
    assert np.array_equal(np.ravel(st)[:3], [ref["nsteps"], ref["nfailed"], ref["nfevals"]])
    # n x 4*numel(tspan): reshape(Y, n, 4, []) is the state at every tspan entry
    assert np.array_equal(Y.reshape(301, 4, tspan.size, order="F"), ref["Y"].transpose(2, 1, 0))
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()))
    mex("destroy", h, nlhs=0); eng.close()


def test_gateway_ode23_packets(mex):
    w, h, eng = _setup(mex, 301, blow_up=True)
    tspan = w.dt * np.linspace(0.0, 1.0, 6)
    st, Y, pstat, t_end = mex("ode23_packets", h, tspan, w.dt, 1e-6, 1e-7, nlhs=4)
    ref = eng.ode23_packets(tspan, w.dt, 1e-6, 1e-7)
    assert np.array_equal(np.ravel(st)[:4], [ref["nsteps"], ref["nfailed"], ref["nfevals"], ref["stopped"]]) and ref["stopped"] == 1
    assert np.array_equal(pstat, np.stack([ref["steps"], ref["rejected"], ref["status"]], axis=1))
    assert np.array_equal(t_end, ref["t_end"])
    assert np.array_equal(Y.reshape(301, 4, tspan.size, order="F"), ref["Y"].transpose(2, 1, 0), equal_nan=True)
    assert np.all(np.isnan(ref["Y"][1:, :, 3])) and np.isfinite(ref["Y"][1:, :, 4:]).all()   # the stopped packet's rows
    assert np.array_equal(np.stack(mex("get_packets", h, nlhs=5))[:4], np.stack(eng.get_packets()), equal_nan=True)
    st1 = mex("ode23_packets", h, [0.0, w.dt], w.dt, 1e-3, 1e-6)         # stats only
    assert np.ravel(st1).shape == (5,) and np.ravel(st1)[3] == 1
    mex("destroy", h, nlhs=0); eng.close()
