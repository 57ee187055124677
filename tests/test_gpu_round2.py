"""GPU tests of the round-2 library features, all through the C ABI (ctypes):

* fused runs on a time-dependent flow (one multi-blend launch + ONE packet kernel for m sub-steps) are the same doubles
  as m single-step calls, in all three modes and for the RK4 steppers;
* ``swrt_step_host`` (host arrays in, steps, host arrays out, pipelined over packet chunks through the pinned ring) is the
  same doubles as ``swrt_set_packets`` + ``swrt_step`` + ``swrt_get_packets``, for ragged sizes that straddle chunks;
* ``swrt_set_packets`` / ``swrt_get_packets`` round-trip pageable buffers bit for bit through the staging ring;
* a multi-device handle (``swrt_params.ngpu = 2``, in-library NCCL) gives bit-identical packets, histograms and ode23
  decisions to the one-device handle (skipped when the box has one GPU).
"""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import reference_api as R
from swraytracing_b200 import workloads as W

pytestmark = pytest.mark.gpu

MODES = {"spectral": S.MODE_SPECTRAL, "lagrange6": S.MODE_LAGRANGE6, "nufft": S.MODE_NUFFT}


def _ndev():
    return int(S.load_library().swrt_device_count())


def _engine(w, mode, ngpu=1, with_h=False):
    eng = S.Engine(w.nx, w.L, w.f, w.gH, mode, device=0, ngpu=ngpu)
    if with_h:
        sc = 0.3 / np.abs(W._fulspec_ifft(w.psik)).max()            # |eta| <= 0.3, so that H = 1 + eta stays positive
        eng.set_flow_planes_spectral(W.planes_from_psik(w.psik, w.L, w.u_mean, etak=sc * w.psik), slot=0)
        if w.psik2 is not None:
            eng.set_flow_planes_spectral(W.planes_from_psik(w.psik2, w.L, w.u_mean, etak=sc * w.psik2), slot=1)
    else:
        eng.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
        if w.psik2 is not None:
            eng.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
    return eng


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("scheme", ["leapfrog", "rk4_packet", "rk4_xka"])
def test_fused_time_dependent_run_equals_single_steps(mode, scheme):
    """m sub-steps of a two-frame flow in one call (pre-blended operands, one packet kernel) == m calls of one step with
    alpha_j = alpha0 + j*dalpha, bit for bit.  C4-like inputs: L = 20, mean shear, ragged packet count."""
    w = W.make_workload("C4", n_packets=1537, nx=32)
    sch = {"leapfrog": S.SCHEME_LEAPFROG, "rk4_packet": S.SCHEME_RK4_PACKET, "rk4_xka": S.SCHEME_RK4_XKA}[scheme]
    m = 5
    a0, da = 0.5 / m, 1.0 / m
    res = []
    for fused in (True, False):
        eng = _engine(w, MODES[mode], with_h=(scheme == "rk4_xka"))
        eng.set_packets(w.x, w.y, w.k, w.l)
        if fused:
            eng.step(sch, w.dt / m, m, a0, da)
        else:
            for j in range(m):
                eng.step(sch, w.dt / m, 1, a0 + j * da, 0.0)
        res.append(np.stack(eng.get_packets(with_a=True)))
        eng.close()
    assert np.isfinite(res[0]).all()
    assert np.array_equal(res[0], res[1])
    assert np.abs(res[0][:4] - np.stack([w.x, w.y, w.k, w.l])).max() > 1e-6      # the packets did move


def test_fused_run_longer_than_the_blend_arena():
    """more sub-steps than one pre-blended run holds (32): several runs, same doubles as single steps"""
    w = W.make_workload("C3", n_packets=700, nx=32)
    m = 70
    res = []
    for fused in (True, False):
        eng = _engine(w, S.MODE_SPECTRAL)
        eng.set_packets(w.x, w.y, w.k, w.l)
        if fused:
            eng.step(S.SCHEME_LEAPFROG, w.dt / m, m, 0.5 / m, 1.0 / m)
        else:
            for j in range(m):
                eng.step(S.SCHEME_LEAPFROG, w.dt / m, 1, 0.5 / m + j * (1.0 / m), 0.0)
        res.append(np.stack(eng.get_packets()))
        eng.close()
    assert np.array_equal(res[0], res[1])


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("n", [1, 1000, 16384, 70001, 300007, 800003])
def test_step_host_equals_set_step_get(mode, n):
    """swrt_step_host == swrt_set_packets + swrt_step + swrt_get_packets bit for bit; sizes straddle the staging chunks
    (one chunk, exact chunk, ragged tails, more chunks than ring slots; 800,003 packets also puts the dense kernel on its
    chunked path: whole waves of 64-packet tiles per chunk); pageable numpy buffers"""
    w = W.make_workload("C3", n_packets=n, nx=32)
    eng = _engine(w, MODES[mode])
    m = 3
    a0, da = 0.5 / m, 1.0 / m
    eng.set_packets(w.x, w.y, w.k, w.l)
    eng.step(S.SCHEME_LEAPFROG, w.dt / m, m, a0, da)
    ref = np.stack(eng.get_packets())
    got = np.stack(eng.step_host(S.SCHEME_LEAPFROG, w.dt / m, m, w.x, w.y, w.k, w.l, alpha0=a0, dalpha=da))
    assert np.array_equal(got, ref)
    # the device keeps the final packets, and in-place output (aliasing the inputs) works
    assert np.array_equal(np.stack(eng.get_packets()), ref)
    bufs = [a.copy() for a in (w.x, w.y, w.k, w.l)]
    eng.step_host(S.SCHEME_LEAPFROG, w.dt / m, m, *bufs, alpha0=a0, dalpha=da, out=bufs)
    assert np.array_equal(np.stack(bufs), ref)
    eng.close()


@pytest.mark.parametrize("mode", ["lagrange6", "nufft", "spectral"])
def test_step_host_rk4_xka_with_wave_action(mode):
    w = W.make_workload("C5", n_packets=40001, nx=32)
    eng = _engine(w, MODES[mode], with_h=True)
    a = np.linspace(0.5, 2.0, w.n_packets)
    eng.set_packets(w.x, w.y, w.k, w.l, a)
    eng.step(S.SCHEME_RK4_XKA, w.dt, 2)
    ref = np.stack(eng.get_packets(with_a=True))
    got = np.stack(eng.step_host(S.SCHEME_RK4_XKA, w.dt, 2, w.x, w.y, w.k, w.l, a))
    assert np.array_equal(got, ref)
    assert np.abs(ref[4] - a).max() > 0          # wave action was transported
    eng.close()


def test_set_get_packets_round_trip_through_the_staging_ring():
    w = W.make_workload("C2", n_packets=3, nx=16)
    eng = _engine(w, S.MODE_LAGRANGE6)
    rs = np.random.RandomState(3)
    for n in (0, 1, 5, 16384, 16385, 100000, 1 << 20):
        arrs = [rs.standard_normal(n) for _ in range(5)]
        eng.set_packets(*arrs)
        back = eng.get_packets(with_a=True)
        for a, b in zip(arrs, back):
            assert np.array_equal(a, b)
        eng.set_packets(*arrs[:4])                      # a = NULL -> ones
        assert np.array_equal(eng.get_packets(with_a=True)[4], np.ones(n))
    eng.close()


def test_step_host_argument_errors():
    w = W.make_workload("C2", n_packets=10, nx=16)
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_LAGRANGE6)
    with pytest.raises(S.SwrtError) as ei:                   # no flow yet
        eng.step_host(S.SCHEME_LEAPFROG, w.dt, 1, w.x, w.y, w.k, w.l)
    assert ei.value.code == -2
    eng.set_flow_spectral(w.psik)
    with pytest.raises(S.SwrtError) as ei:
        eng.step_host(7, w.dt, 1, w.x, w.y, w.k, w.l)
    assert ei.value.code == -1
    with pytest.raises(S.SwrtError):                         # dalpha without a second frame
        eng.step_host(S.SCHEME_LEAPFROG, w.dt, 2, w.x, w.y, w.k, w.l, alpha0=0.25, dalpha=0.5)
    eng.close()


# ------------------------------------------------------------------------------------------------
# multi-device handle (in-library sharding + NCCL)
# ------------------------------------------------------------------------------------------------
def test_multi_device_handle_argument_errors():
    lib = S.load_library()
    nd = _ndev()
    with pytest.raises(S.SwrtError) as ei:
        S.Engine(32, 6.28, 3.0, 1.0, ngpu=nd + 1)
    assert ei.value.code == -1 and "devices" in str(ei.value)
    e = S.Engine(32, 6.28, 3.0, 1.0, ngpu=1)
    assert lib.swrt_num_devices(e._h) == 1 and e.shard_info(0) == (0, 0, 0)
    e.close()


needs2 = pytest.mark.skipif(_ndev() < 2, reason="needs >= 2 CUDA devices (the in-library multi-device handle)")


@needs2
@pytest.mark.parametrize("mode", list(MODES))
def test_multi_device_handle_is_bit_identical_to_one_device(mode):
    """ngpu = 2 through the SAME C-ABI calls: packets after leapfrog / RK4 steps, step_host, histograms (blocking and
    launch/wait), ode23 decisions and the per-packet inspection calls all equal the one-device handle's, bit for bit"""
    w = W.make_workload("C3", n_packets=20011, nx=32)
    edges = np.linspace(0.0, 8.0, 300)
    out = []
    for ngpu in (1, 2):
        eng = _engine(w, MODES[mode], ngpu=ngpu)
        eng.set_packets(w.x, w.y, w.k, w.l)
        assert int(eng.lib.swrt_num_packets(eng._h)) == w.n_packets
        eng.step(S.SCHEME_LEAPFROG, w.dt / 4, 4, 0.125, 0.25)
        st1 = np.stack(eng.get_packets())
        ev = eng.eval(0.5)
        rhs = np.stack(eng.rhs(0.5))
        om, Om = eng.omega(0.5)
        h_int = eng.hist_omega(edges)
        h_abs = eng.hist_omega(edges, S.HIST_ABSOLUTE, 0.5)
        ptr, nb = eng.hist_omega_launch(edges)
        eng.hist_omega_wait()
        d = eng.diag(0.5)
        sol = R.ode23(eng, [0.0, w.dt], w.dt)
        st2 = np.stack(eng.get_packets())
        eng.step(S.SCHEME_RK4_PACKET, w.dt, 2)
        st3 = np.stack(eng.get_packets())
        st4 = np.stack(eng.step_host(S.SCHEME_LEAPFROG, w.dt / 2, 2, w.x, w.y, w.k, w.l, alpha0=0.25, dalpha=0.5))
        gx, gy = np.meshgrid(np.linspace(0, w.L, 24), np.linspace(0, w.L, 24))
        th = np.linspace(0, 2 * np.pi, 50)
        ideal = eng.ideal_omega_hist(gx.ravel(), gy.ravel(), 5 * np.cos(th), 5 * np.sin(th), np.sqrt(9 + 25.0), np.linspace(3.0, 9.0, 100))
        if ngpu == 2:
            infos = [eng.shard_info(i) for i in range(2)]
            assert infos[0] == (0, 0, w.n_packets // 2) and infos[1] == (1, w.n_packets // 2, w.n_packets - w.n_packets // 2)
        out.append(dict(st1=st1, ev=ev, rhs=rhs, om=om, Om=Om, h_int=h_int, h_abs=h_abs, d=d, nsteps=sol["nsteps"], nfailed=sol["nfailed"],
                        st2=st2, st3=st3, st4=st4, ideal=ideal))
        eng.close()
    a, b = out
    for key in ("st1", "ev", "rhs", "om", "Om", "h_int", "h_abs", "st2", "st3", "st4", "ideal"):
        assert np.array_equal(a[key], b[key]), key
    assert a["nsteps"] == b["nsteps"] and a["nfailed"] == b["nfailed"]
    assert int(a["h_int"].sum()) == w.n_packets
    # sums are re-associated across devices: equal to round-off; extrema, counts exact
    assert np.allclose(a["d"], b["d"], rtol=1e-13, atol=0) and a["d"][2] == b["d"][2] and a["d"][3] == b["d"][3] and a["d"][6] == b["d"][6]


@needs2
def test_multi_device_handle_fewer_packets_than_devices():
    w = W.make_workload("C2", n_packets=1, nx=16)
    eng = _engine(w, S.MODE_SPECTRAL, ngpu=2)
    one = _engine(w, S.MODE_SPECTRAL, ngpu=1)
    for e in (eng, one):
        e.set_packets(w.x, w.y, w.k, w.l)
        e.step(S.SCHEME_LEAPFROG, w.dt, 3)
    assert np.array_equal(np.stack(eng.get_packets()), np.stack(one.get_packets()))
    assert np.array_equal(eng.hist_omega(np.linspace(0, 8, 30)), one.hist_omega(np.linspace(0, 8, 30)))
    eng.close(); one.close()


@needs2
def test_multi_device_handle_qg_frame_producer():
    """swrt_set_flow_from_qg on a multi-device handle: the frame is built on the first device and peer-copied"""
    nx, L, f, Cg = 32, 2 * np.pi, 3.0, 1.0
    w0 = W.make_workload("C2", n_packets=4, nx=nx)
    kx, ky = W.wavenumbers(nx)
    qk = -(f / Cg + kx ** 2 + ky ** 2) * w0.psik            # q-hat of the synthetic streamfunction (grid_U.m:2 inverted)
    res = []
    for ngpu in (1, 2):
        qg = S.QGFlow(nx, L, qk, f / Cg, 1e-3, f, Cg, r_drag=0.01, device=0)
        qg.step(3)
        eng = S.Engine(nx, L, f, Cg ** 2, S.MODE_SPECTRAL, ngpu=ngpu)
        qg.to_flow(eng, 0)
        w = W.make_workload("C2", n_packets=501, nx=nx)
        eng.set_packets(w.x, w.y, w.k, w.l)
        res.append(eng.eval())
        eng.close(); qg.close()
    assert np.array_equal(res[0], res[1])


# ------------------------------------------------------------------------------------------------
# fused SPECTRAL RK4 steppers (one launch per run of steps) against the composed route
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nx", [32, 64, 128, 130, 256, 512])
@pytest.mark.parametrize("scheme", ["rk4_packet", "rk4_xka"])
@pytest.mark.parametrize("flow", ["psi", "planes", "two-frame"])
def test_spectral_fused_rk4_equals_the_composed_launches(nx, scheme, flow):
    """step_packet / step_packet_xka in SPECTRAL mode: the fused kernel (five contractions + the RK4 update with the packet
    in registers, ONE launch) against the composed route of round 1 (five EVAL launches + five glue kernels per step,
    swrt_set_tuning flag 4).  Same contraction order, so the evaluations agree to the last bits; the stage arithmetic is
    compiled in two places, hence 1e-13 rather than bit equality."""
    xka = scheme == "rk4_xka"
    if xka and flow == "psi":
        pytest.skip("step_packet_xka needs the H plane (planes upload)")
    w = W.make_workload("C4" if flow == "two-frame" else "C5", n_packets=1203, nx=nx)
    sch = S.SCHEME_RK4_XKA if xka else S.SCHEME_RK4_PACKET
    m = 3
    a0, da = (0.5 / m, 1.0 / m) if flow == "two-frame" else (0.0, 0.0)
    res, launches = [], []
    for fused in (True, False):
        eng = _engine(w, S.MODE_SPECTRAL, with_h=(xka or flow == "planes"))
        eng.set_tuning(unfused_rk4=not fused)
        eng.set_packets(w.x, w.y, w.k, w.l, np.linspace(0.5, 2.0, w.n_packets))
        eng.step(sch, w.dt, 1, a0, 0.0)                       # warm: stacks packed
        n0 = eng.launch_count(reset=True)
        eng.step(sch, w.dt, m, a0, da)
        launches.append(eng.launch_count())
        res.append(np.stack(eng.get_packets(with_a=True)))
        eng.close()
    assert np.isfinite(res[0]).all()
    scale = np.abs(res[1]).max(axis=1, keepdims=True)
    assert (np.abs(res[0] - res[1]) / scale).max() < 1e-13
    assert launches[0] == (3 if flow == "two-frame" else 1)     # one packet kernel (+ the two multi-blends of a two-frame run)
    assert launches[1] >= 9 * m                                  # 4-5 evaluations + 4 stage kernels + the final update, per step
    if xka:
        assert np.abs(res[0][4] - np.linspace(0.5, 2.0, w.n_packets)).max() > 0


# ------------------------------------------------------------------------------------------------
# where the x twiddles live: rotation in registers / shared-memory table / global (L2) table
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nx", [64, 128, 256, 512])
def test_twiddle_homes_agree_and_match_the_exact_sum(nx):
    """swrt_set_tuning bits 3-4 pick where the dense kernel keeps a step's x twiddles.  The three homes run the SAME
    recurrences (the table forms tabulate them), so the evaluations agree to the last bits (<= 1e-14 of max|plane|), and each
    is within 1e-12 of the long-double exact-sum oracle; 20 leapfrog steps agree to 1e-12.  256^2 and 512^2 exercise the L2
    table that is the default above 128^2.  The leapfrog contracts the six planes: a psi-hat leapfrog at 256^2 and 512^2
    runs anchored, which has no twiddle home."""
    from oracle import c_oracle as CO
    w = W.make_workload("C3", n_packets=389, nx=nx)
    planes = W.planes_from_psik(w.psik, w.L, w.u_mean)
    ref = CO.spectral_eval(w.x, w.y, planes, w.dx, nx, precise=True)
    scale = np.abs(ref).max(axis=1, keepdims=True)
    evs, trajs, homes = [], [], []
    for tw in (0, 1, 2, 3):
        eng = S.Engine(nx, w.L, w.f, w.gH, S.MODE_SPECTRAL)
        eng.set_tuning(twiddles=tw)
        eng.set_flow_spectral(w.psik, 0, w.u_mean)
        eng.set_packets(w.x, w.y, w.k, w.l)
        ev = eng.eval()
        assert (np.abs(ev - ref) / scale).max() < 1e-12, (nx, tw)
        eng.set_tuning(twiddles=tw, use_psi_moments=False)
        eng.step(S.SCHEME_LEAPFROG, w.dt, 20)
        evs.append(ev); trajs.append(np.stack(eng.get_packets()))
        eng.close()
    for ev, tr in zip(evs[1:], trajs[1:]):
        assert (np.abs(ev - evs[0]) / scale).max() < 1e-14
        assert np.abs(tr - trajs[0]).max() < 1e-12
    geo = S.engine.spectral_geometry(nx, 3, 1)
    assert geo["twiddle_table"] == (1 if nx <= 128 else 2)


def test_a_blown_up_packet_does_not_poison_its_neighbours():
    """non-finite packets travel through swrt_step_host (chunked, staged) without touching the others; swrt_diag counts them"""
    w = W.make_workload("C2", n_packets=40000, nx=32)
    x = w.x.copy(); k = w.k.copy()
    bad = [0, 17, 16384, 39999]
    x[bad[:2]] = np.nan; k[bad[2:]] = np.inf
    for mode in MODES.values():
        eng = _engine(w, mode)
        got = np.stack(eng.step_host(S.SCHEME_LEAPFROG, w.dt, 3, x, w.y, k, w.l))
        clean = _engine(w, mode)
        ref = np.stack(clean.step_host(S.SCHEME_LEAPFROG, w.dt, 3, w.x, w.y, w.k, w.l))
        good = np.ones(w.n_packets, dtype=bool); good[bad] = False
        assert np.array_equal(got[:, good], ref[:, good])
        assert not np.isfinite(got[:, bad]).all(axis=0).any()
        assert eng.diag()[4] == len(bad)
        eng.close(); clean.close()


def test_interpolate_rejects_what_matlab_would_reject():
    """interpolate.m:45-46 wraps BOTH stencil indices with nx, so an nx x ny array with ny < nx makes MATLAB raise
    "index exceeds array bounds"; swrt_interpolate returns SWRT_ERR_ARG instead of reading out of bounds, and the Python
    mirror refuses x / y of different lengths"""
    F = np.arange(8.0 * 6).reshape(8, 6)
    with pytest.raises(S.SwrtError) as ei:
        S.interpolate_dev(np.array([1.0]), np.array([1.0]), F, 1.0, 1.0)
    assert ei.value.code == -1 and "ny >= nx" in str(ei.value)
    with pytest.raises(ValueError):
        S.interpolate_dev(np.zeros(3), np.zeros(4), np.zeros((8, 8)), 1.0, 1.0)
    # ny > nx is legal in the reference (only the first nx columns are ever read) and matches the restatement bit for bit
    from oracle import swrt_oracle as O
    G = np.random.RandomState(1).standard_normal((8, 11))
    x, y = np.random.RandomState(2).uniform(-20, 20, (2, 50))
    assert np.array_equal(S.interpolate_dev(x, y, G, 0.7, 0.7), O.interpolate(x, y, G, 0.7, 0.7))
