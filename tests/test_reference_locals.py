"""The reference's file-local / nested functions, executed unmodified, against the oracle and the product.

``tests/golden/reference_locals_nx32.npz`` (made by ``tests/golden/run_reference_locals.py`` with ``oracle/minimat``) holds the
outputs of functions no MATLAB session can call from outside their file: ``odefun`` -- the ``ode23`` right-hand side nested
in ``generate_raytracing_ode`` (qgsw_raytrace.m:258-268, qg2layersw_raytrace.m:297-307) -- ``ode_xk2y`` / ``ode_y2xk``, the QG
frame producers ``initial_q`` / ``inertial_ring`` / ``filter`` / ``update`` (one layer) and ``update`` / ``mmult3`` / ``diag_exp``
(two layers); plus the top-level ``interpolate_par.m`` (nested ``compute_FI`` through ``arrayfun``), the six-argument
``grid_U.m`` with a mean shear, the complex / multi-frame branches of ``write_field.m`` / ``read_field.m``, and one driver
script run as a whole: ``ray_trace_sw/raytrace.m`` (its first packet over 300 ``step_packet`` calls).

CPU tests: the oracle's restatements equal them (bit for bit where no FFT is involved, 1e-15 of the plane otherwise);
``-m gpu`` tests: the product (``swrt_rhs``, ``swrt_interpolate`` with bump 1e-10, the device ``grid_U``, the on-device QG
solver) is held to the same files.
"""
import json
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import swrt_oracle as O          # noqa: E402

GOLD = ROOT / "tests" / "golden"
R = np.load(GOLD / "reference_locals_nx32.npz")
H = np.load(GOLD / "hotpath_nx32.npz")
NAMES = ("u", "v", "ux", "uy", "vx", "vy")
NX, L, F0 = int(H["nx"]), float(H["L"]), float(H["f"])
DX = L / NX
KX, KY = O.wavenumbers(NX)
K2 = KX ** 2 + KY ** 2
TMAX = float(R["tmax"])
# a checkout of the original MATLAB project (ndefilippis/SWRaytracing), which this repository does not carry
REF = Path(os.environ.get("SWRT_REFERENCE_DIR", "")).absolute()
HAVE_REF = bool(os.environ.get("SWRT_REFERENCE_DIR")) and (REF / "ode_symplectic.m").exists()


def frames():
    g1 = list(H["grids"])
    g2 = [O.k2g(p) for p in O.velocity_planes_k(H["psik2"], KX, KY)]
    return dict(zip(NAMES, g1)), dict(zip(NAMES, g2))


def rel(got, ref):
    ref = np.asarray(ref)
    return float(np.abs(np.asarray(got) - ref).max() / max(np.abs(ref).max(), 1e-300))


def test_provenance_lists_the_driver_files():
    prov = json.loads(str(R["provenance"]))
    ex = set(prov["reference_files_executed"])
    assert {"qg_flow_ray_trace/qgsw_raytrace.m", "qg_flow_ray_trace/qg2layersw_raytrace.m", "interpolate_par.m", "qg_flow_ray_trace/grid_U.m",
            "qg_flow_ray_trace/interpolate_U.m", "qg_flow_ray_trace/interpolate.m", "qg_flow_ray_trace/write_field.m",
            "qg_flow_ray_trace/read_field.m"} <= ex
    if HAVE_REF:
        import hashlib
        for relp, sha in prov["reference_files_executed"].items():
            assert hashlib.sha256((REF / relp).read_bytes()).hexdigest() == sha, relp


@pytest.mark.skipif(not HAVE_REF, reason="set SWRT_REFERENCE_DIR to a checkout of the original MATLAB project")
def test_rerunning_the_generator_reproduces_the_committed_file(tmp_path):
    """tests/golden/run_reference_locals.py --quick, executed again here from the unmodified reference: every array equals the
    committed one bit for bit (the two script trajectories are compared on the steps the quick run makes)"""
    sys.path.insert(0, str(GOLD))
    import run_reference_locals as G
    out = tmp_path / "locals.npz"
    G.main(["--ref", str(REF), "--quick", "--out", str(out)])
    N = np.load(out)
    assert set(N.files) == set(R.files)
    for key in R.files:
        if key == "provenance":
            assert json.loads(str(N[key]))["reference_files_executed"] == json.loads(str(R[key]))["reference_files_executed"]
        elif key in ("raytrace_p1", "rsw_p1"):
            assert np.array_equal(N[key], R[key][: N[key].shape[0]]), key
        elif key.startswith("odefun_") or key in ("ode_xk2y", "qg2_odefun_tmid"):            # [x; y; k; l] blocks of the first 24 packets
            assert np.array_equal(N[key].reshape(4, 24), R[key].reshape(4, -1)[:, :24]), key
        elif key in ("ode_y2xk_x", "ode_y2xk_k"):
            assert np.array_equal(N[key], R[key][:24]), key
        elif key == "interpolate_par":
            assert np.array_equal(N[key], R[key][:, :24]), key
        elif key == "qgsw_packets_y":
            assert np.array_equal(N[key], R[key][: N[key].shape[0]]), key
        elif key.startswith("qgsw_file_"):
            assert np.array_equal(N[key], R[key][: N[key].size]), key
        elif key == "swz_odefun":
            assert np.array_equal(N[key].reshape(4, 24), R[key].reshape(4, -1)[:, :24]), key
        elif key in ("swz_omega", "swz_grad_omega"):
            assert np.array_equal(N[key], R[key][:24]), key
        elif key in ("c1_x", "c1_y", "c1_k", "c1_l"):
            assert np.array_equal(N[key], R[key][:40]), key
        elif key == "c1_final":
            assert np.array_equal(N[key], R[key][:, :40]), key
        else:
            assert np.array_equal(N[key], R[key]), key


def test_oracle_odefun_and_state_packing_equal_the_nested_reference_function():
    """qgsw_raytrace.m:232-268: y = [x; y; k; l]; dydt bit for bit at alpha = 0, 1/4, 1 (pure Lagrange arithmetic + blend)"""
    x, y, k, l = (H[n] for n in ("x", "y", "k", "l"))
    n = x.size
    yv = np.concatenate([x, y, k, l])
    assert np.array_equal(R["ode_xk2y"], yv)
    assert np.array_equal(R["ode_y2xk_x"], np.stack([x, y], 1)) and np.array_equal(R["ode_y2xk_k"], np.stack([k, l], 1))
    bf1, bf2 = frames()
    ode = O.generate_raytracing_ode(bf1, bf2, n, F0, 1.0, TMAX, DX)
    for tag, t in (("t0", 0.0), ("tmid", 0.25 * TMAX), ("tend", TMAX)):
        assert np.array_equal(ode(t, yv), R["odefun_" + tag]), tag
    assert np.array_equal(R["qg2_odefun_tmid"], R["odefun_tmid"])          # the two drivers carry the same text


def test_oracle_interpolate_par_equals_the_reference():
    x, y = H["x"], H["y"]
    for j, g in enumerate(H["grids"]):
        assert np.array_equal(O.interpolate_par(x, y, g, DX, DX), R["interpolate_par"][j])
    # and it is NOT the live interpolate (bump 1e-13): the two differ at the 1e-10 level
    d = np.abs(O.interpolate(x, y, H["grids"][0], DX, DX) - R["interpolate_par"][0]).max()
    assert 1e-13 < d < 1e-8


def test_oracle_interpolate_at_the_awkward_places_equals_both_reference_copies():
    """on nodes, one ulp either side, at the bump's own scale, at the domain ends, mod(-tiny, nx) = nx, a million periods away"""
    ex, ey = R["edge_x"], R["edge_y"]
    assert ex.size >= 60 and (ex == 0).any() and (ex < 0).any() and (np.abs(ex) > 1e6).any()
    for j in range(2):
        g = H["grids"][j]
        assert np.array_equal(O.interpolate(ex, ey, g, DX, DX), R["edge_interpolate_live"][j])
        assert np.array_equal(O.interpolate(ex, ey, g, DX, DX, O.BUMP_QG), R["edge_interpolate_qg"][j])
        on = np.abs(ex / DX - np.round(ex / DX)) < 1e-9
        assert on.sum() > 20 and np.abs(R["edge_interpolate_live"][j] - R["edge_interpolate_qg"][j])[~on].max() > 1e-12


def _g24():
    names = ("u", "v", "ux", "uy", "vx", "vy")
    bf1 = dict(zip(names, R["g24_planes1"])); bf2 = dict(zip(names, R["g24_planes2"]))
    return bf1, bf2, float(R["g24_L"]) / 24, tuple(R["g24_" + c] for c in "xykl")


def test_oracle_on_a_24x24_grid_with_L_20_equals_the_reference():
    """a grid that is not a power of two, a domain that is not 2*pi: odefun (bump 1e-10) and two RK4 steps of step_packet /
    step_packet_xka (bump 1e-13) per packet, bit for bit"""
    bf1, bf2, h, (x, y, k, l) = _g24()
    ode = O.generate_raytracing_ode(bf1, bf2, x.size, float(R["g24_f"]), float(R["g24_C0"]), 0.2, h)
    assert np.array_equal(ode(0.06, np.concatenate([x, y, k, l])), R["g24_odefun"])
    fields = dict(zip(("u", "v", "u_x", "u_y", "v_x", "v_y"), R["g24_planes1"]))
    fields["H"] = R["g24_H"]
    for xka, key in ((True, "g24_rk4x2_xka"), (False, "g24_rk4x2_packet")):
        st = (x, y, k, l, np.ones(x.size))
        for _ in range(2):
            st = O.rk4_step_batch(*st, float(R["g24_dt"]), float(R["g24_C0"]), float(R["g24_f"]), fields, h, xka)
        assert np.array_equal(np.stack(st)[: R[key].shape[0]], R[key]), key


def test_oracle_qg_producers_equal_the_reference_locals():
    xs = O.matlab_linspace(-L / 2, L / 2, NX)
    X, Y = np.meshgrid(xs, xs)
    q0 = O.initial_q(X, Y, 0.5, 3.0, O.matlab_rand_stream(146))
    assert np.array_equal(q0, R["initial_q"])
    ring = O.qg_inertial_ring(0.1, K2, 3.0, 0.25)
    assert ring.any() and np.array_equal(ring, R["inertial_ring"])
    assert np.array_equal(O.qg_filter(KX, KY, DX), R["filter"])
    assert np.array_equal(O.g2k(q0), R["update_qk_in"])
    got = O.qg_update(R["update_qk_in"], K2, 3.0, 0.3, 0.1, R["inertial_ring"], KX, KY)
    assert np.array_equal(got, R["update"])


def test_oracle_two_layer_operators_equal_the_reference_locals():
    B, q2 = R["qg2_B"], R["qg2_qk_in"]
    assert np.array_equal(O.mmult3(B, q2), R["qg2_mmult3"])
    assert np.array_equal(O.qg2_update(q2, B, KX, KY), R["qg2_update"])
    A = B.astype(complex) * (1 + 0.5j)
    E = R["qg2_diag_exp"]
    assert E.shape[:2] == (2, 2) and np.array_equal(E[0, 0], np.exp(0.3 * A[0, 0])) and np.array_equal(E[1, 1], np.exp(0.3 * A[1, 1]))
    assert not E[0, 1].any() and not E[1, 0].any()


def test_oracle_grid_U_with_shear_equals_the_reference():
    flow = O.grid_U(R["update_qk_in"], 3.0, K2, KX, KY, float(R["grid_U_shear_value"]))
    for j, nm in enumerate(NAMES):
        assert np.array_equal(flow[nm], R["grid_U_shear"][j]), nm
    assert abs(R["grid_U_shear"][0].mean() - float(R["grid_U_shear_value"])) < 1e-14


def test_product_field_files_equal_the_reference_writer_and_reader(tmp_path):
    """swraytracing_b200.fieldio (host-side, no device): the bytes write_field.m appends for a complex two-frame file and what
    read_field.m returns for frame lists"""
    from swraytracing_b200 import fieldio
    qk = R["update_qk_in"]
    fieldio.write_field(qk, tmp_path / "spec", 1)
    fieldio.write_field(2 * qk, tmp_path / "spec", 2)
    assert np.array_equal(np.fromfile(tmp_path / "spec.bin"), R["write_field_complex_bytes"])
    back = fieldio.read_field(tmp_path / "spec", qk.shape[0], qk.shape[1], 1, [2])
    assert np.array_equal(back, R["read_field_complex_frame2"]) and np.array_equal(back, 2 * qk)
    for fr, g in enumerate(H["grids"][:3], 1):
        fieldio.write_field(g, tmp_path / "grid", fr)
    got = fieldio.read_field(tmp_path / "grid", NX, NX, 1, [3, 1], True)
    assert np.array_equal(got, R["read_field_frames_3_1"])
    assert np.array_equal(got[:, :, 0], H["grids"][2]) and np.array_equal(got[:, :, 1], H["grids"][0])


def test_oracle_two_layer_driver_equals_the_executed_driver():
    """qg2layersw_raytrace(32, 0, 2, 600, 100, 0.3, 3, 1) executed as the reference wrote it (rng(5), B / factor_L, pageeig,
    integrating-factor AB3, CFL logic): the restated driver has the same PV spectra at the start of steps 1, 2, 4, 7 --
    bit-identical before the first step, to round-off after (V exp(D t) V^-1 is evaluated by einsum here, pagemtimes there) --
    and prints the same header"""
    log = str(R["qg2_driver_log"])
    for steps, ref in zip((0, 1, 3, 6), R["qg2_driver_states"]):
        r = O.qg2layersw_driver(32, 0, 2, 600, 100, 0.3, 3.0, 1.0, max_steps=steps)
        err = np.abs(r["qk"] - ref).max() / np.abs(ref).max()
        assert (err == 0.0) if steps == 0 else (err < 1e-13), (steps, err)
    assert "Initial time step: %f" % r["dt"] in log and "Froude Number: %f" % r["Fr"] in log
    assert "Background velocity (parameter,computed): (0.300000,%f)" % (r["Fr"] * 1.0) in log and "Simulation time: %f" % r["T"] in log


def test_theoretical_omega_pdf_of_the_executed_script():
    """ideal_omega_distribution.m run as a script on U = scheme.U(grid): omega_abs = omega_0 + U.k over (grid point, angle) --
    restated here in three numpy lines from the stored U, and binned (histcounts rule) into the stored counts"""
    U = R["ideal_U"]
    t = O.matlab_linspace(0.0, 2 * np.pi, 100)             # multiply-then-divide: numpy.linspace differs in the last bit
    kv = 3.0 * np.stack([np.cos(t), np.sin(t)], axis=1)
    om = np.sqrt(F0 ** 2 + 1.0 * 9.0) + (np.outer(U[:, 0], kv[:, 0]) + np.outer(U[:, 1], kv[:, 1]))
    assert om.size == int(R["ideal_total"]) == NX * NX * 100
    assert np.array_equal(om.ravel(order="F")[::16], R["ideal_omega_abs"])
    assert np.array_equal(O.histcounts(om.ravel(order="F"), R["ideal_edges"]), R["ideal_counts"]) and R["ideal_counts"].sum() > 0.9 * om.size
    # U itself: the reference's SpectralScheme on the grid of symplectic_full_fourier.m:14-15 (linspace(0, L, nx): the last node
    # wraps onto the first)
    X = O.matlab_linspace(0.0, L, NX); XX, YY = np.meshgrid(X, X)
    planes = O.velocity_planes_k(O.g2k(O.k2g(H["psik"])), KX, KY)
    for j in range(2):
        assert np.array_equal(O.interpolate(XX.ravel(order="F"), YY.ravel(order="F"), O.k2g(planes[j]), DX, DX), U[:, j])


def test_oracle_raytrace_driver_equals_the_executed_script():
    """ray_trace_sw/raytrace.m run as a script (Childress-Soward flow with the matrix product of :36 as written, ``rand*L`` from
    MATLAB's start-up stream, 300 ``step_packet`` calls on packet 1): the restated driver gives the same doubles"""
    hist, dt, nsteps = O.raytrace_driver(np_=5, nsteps=301)
    assert dt == float(R["raytrace_dt"])
    assert int(round((1 / (4.0 * 0.1 ** 2)) / dt)) == int(R["raytrace_nsteps"]) == 3395
    for j, c in enumerate("xykl"):
        assert np.array_equal(hist[c][:, 0], R["raytrace_P0"][:, j]), c
        assert np.array_equal(hist[c][0, :301], R["raytrace_p1"][:, j]), c
    _, _, G = O.childress_soward_as_written(256, 2 * np.pi, 0.1, 4.0, 0.25)
    assert np.array_equal(G["v_x"], R["raytrace_GradU_v_x"])
    assert np.abs(R["raytrace_GradU_v_x"]).max() > 10 * 0.4 * 1.25            # the matrix product blows v_x up far beyond km*U0*(1+a)


def test_config_1_zero_background_flow_under_the_executed_reference():
    """BASELINE config 1 (1,000 packets, zero background flow, symplectic step; plumbing + analytic dispersion): five steps of
    the reference's own ode_symplectic.m over a SpectralScheme of a zero streamfunction.  The packets move in straight lines at
    the group velocity, k unchanged -- the analytic answer to 1e-13 -- and the restated stepper gives the same doubles."""
    x, y, k, l = (R["c1_" + c] for c in "xykl")
    assert x.size == 1000
    fin = R["c1_final"]
    w = np.sqrt(9.0 + (k * k + l * l))
    assert np.array_equal(fin[2], k) and np.array_equal(fin[3], l)
    assert np.abs(fin[0] - (x + 5 * 0.01 * k / w)).max() < 1e-13 and np.abs(fin[1] - (y + 5 * 0.01 * l / w)).max() < 1e-13
    assert np.allclose(R["c1_t"], 0.01 * np.arange(6), rtol=0, atol=1e-17)
    zero = [np.zeros((NX, NX))] * 6
    st = (x, y, k, l)
    for _ in range(5):
        st = O.leapfrog_step(*st, 0.01, 3.0, 1.0, lambda xx, yy: [O.interpolate(xx, yy, g, DX, DX) for g in zero])
    assert np.array_equal(np.stack(st), fin)


def test_oracle_qgsw_loop_with_packets_equals_the_executed_driver():
    """qgsw_raytrace(32, 12, 2, 6000, 0, 0.5, 3, 1) executed (packets from the first flow step; ode23 = the restated controller,
    a MATLAB builtin): the restated pieces chained the way the driver chains them -- qg_run frames, grid_U, odefun with the
    bump of the copy beside it, ode23 over [0, dt] -- give the same packets at the start of steps 1..7, and the packet files
    hold the initial frame (time -dt: packet_step_start = 0) and the wrapped frame of step 4"""
    nx, Np, nif, U_g, f, Cg = 32, 12, 2.0, 0.5, 3.0, 1.0
    K_d2 = f / Cg
    xg = O.matlab_linspace(-L / 2, L / 2, nx); X, Y = np.meshgrid(xg, xg)
    rs = O.matlab_rand_stream(146)
    qk0 = O.g2k(O.initial_q(X, Y, U_g, K_d2, rs))
    x, y, k, l = O.init_packets(Np, L, np.sqrt((nif ** 2 - 1) * f ** 2 / Cg ** 2), rs)
    fl = O.grid_U(qk0, K_d2, K2, KX, KY)
    U0 = np.sqrt((fl["u"] ** 2 + fl["v"] ** 2).max()); dt = 0.05 * (L / nx) / U0
    assert "Time step: %f" % dt in str(R["qgsw_log"]) and "(0.500000,%f)" % U0 in str(R["qgsw_log"])
    yv = np.concatenate([x, y, k, l])
    ref = R["qgsw_packets_y"]
    assert np.array_equal(yv, ref[0])
    names = ("u", "v", "ux", "uy", "vx", "vy")
    for step in range(1, ref.shape[0]):
        bf1 = O.grid_U(O.qg_run(qk0, step - 1, dt, nx, L, K_d2, f, Cg), K_d2, K2, KX, KY)
        bf2 = O.grid_U(O.qg_run(qk0, step, dt, nx, L, K_d2, f, Cg), K_d2, K2, KX, KY)
        yv, _ = O.ode23(O.generate_raytracing_ode(bf1, bf2, Np, f, Cg, dt, L / nx), [0, dt], yv)
        assert np.abs(yv - ref[step]).max() <= 1e-12, step            # qg_run vs the driver's in-place AB3: round-off only
    t = R["qgsw_file_packet_time"]
    assert t.size == 2 and t[0] == dt * (0 - 1) and abs(t[1] - 4 * dt) < 1e-15
    px = R["qgsw_file_packet_x"].reshape(2, 2, Np)                     # two frames of an Np x 2 array, column-major
    assert np.array_equal(px[0, 0], x) and np.array_equal(px[0, 1], y)
    wrapped = np.mod(ref[4][: 2 * Np] + L / 2, L) - L / 2
    assert np.array_equal(px[1].ravel(), wrapped)
    assert np.array_equal(R["qgsw_file_packet_k"].reshape(2, 2, Np)[1].ravel(), ref[4][2 * Np:])


def _swz_rhs(ev6, k, l, f, gH):
    """SW_zero_background_raytracing.m:134-145,182-184 from the six evaluated planes"""
    u, v, ux, uy, vx, vy = ev6
    w = np.sqrt(f * f + gH * (k * k + l * l))
    return np.concatenate([u + gH * k / w, v + gH * l / w, -(ux * k + vx * l), -(uy * k + vy * l)])


def test_config_1_script_right_hand_side_equals_the_nested_reference_function():
    """the ode23 right-hand side of SW_zero_background_raytracing.m (gH k/omega, not Cg k/omega as in the QG drivers) over the
    reference's own SpectralScheme object, and its local omega / grad_omega"""
    x, y, k, l = (H[c] for c in "xykl")
    fields = [O.k2g(p) for p in O.velocity_planes_k(O.g2k(O.k2g(H["psik"])), KX, KY)]
    ev6 = [O.interpolate(x, y, g, DX, DX) for g in fields]
    assert np.array_equal(_swz_rhs(ev6, k, l, F0, 1.7), R["swz_odefun"])
    w = np.sqrt(F0 * F0 + 1.7 * (k * k + l * l))
    assert np.array_equal(w, R["swz_omega"])
    assert np.array_equal(np.stack([1.7 * k / w, 1.7 * l / w], axis=1), R["swz_grad_omega"])


def test_oracle_raytrace_sw_driver_equals_the_executed_script():
    """ray_trace_sw/raytrace_sw.m run as a script on a seeded [u,v,eta] state served to its ``load``: geostrophic projection,
    gradients and H (rsw/g2k.m, k2g.m), U0 / dt / nsteps, ring of packets from the start-up random stream, 150 step_packet_xka
    calls on packet 1 with wave action -- the restated driver gives the same doubles"""
    hist, info = O.raytrace_sw_driver(R["rsw_S"], 3.0, 1.0, np_=10, nsteps=151)
    assert info["dt"] == float(R["rsw_dt"]) and info["U0"] == float(R["rsw_U0"])
    assert int(round(20 / (3.0 * info["Fr"] ** 2) / info["dt"])) == int(R["rsw_nsteps"])
    got = [info["U"]["u"], info["U"]["v"]] + [info["GradU"][c] for c in ("u_x", "u_y", "v_x", "v_y")] + [info["H"]]
    for j, g in enumerate(got):
        assert np.array_equal(g, R["rsw_fields"][j]), j
    for j, c in enumerate("xykla"):
        assert np.array_equal(hist[c][:, 0], R["rsw_P0"][:, j]), c
        assert np.array_equal(hist[c][0, :151], R["rsw_p1"][:, j]), c
    assert abs(R["rsw_p1"][-1, 4] - 1.0) > 1e-3                     # the wave action has moved


# ---------------------------------------------------------------------------------------------------------- product, on the GPU
@pytest.mark.gpu
def test_gpu_on_a_24x24_grid_with_L_20_equals_the_reference():
    import swraytracing_b200 as S
    bf1, bf2, h, (x, y, k, l) = _g24()
    names = ("u", "v", "ux", "uy", "vx", "vy")
    f, C0, dt, L24 = float(R["g24_f"]), float(R["g24_C0"]), float(R["g24_dt"]), float(R["g24_L"])
    with S.Engine(24, L24, f, C0 * C0, S.MODE_LAGRANGE6, bump=1e-10) as e:
        e.set_flow_grid(*[bf1[n] for n in names], slot=0); e.set_flow_grid(*[bf2[n] for n in names], slot=1)
        e.set_packets(x, y, k, l)
        assert np.array_equal(np.concatenate(e.rhs(0.3)), R["g24_odefun"])
    for xka, key, sch in ((True, "g24_rk4x2_xka", S.SCHEME_RK4_XKA), (False, "g24_rk4x2_packet", S.SCHEME_RK4_PACKET)):
        with S.Engine(24, L24, f, C0 * C0, S.MODE_LAGRANGE6) as e:
            e.set_flow_grid(*[bf1[n] for n in names], H=R["g24_H"] if xka else None, slot=0)
            e.set_packets(x, y, k, l)
            e.step(sch, dt, 2)
            got = np.stack(e.get_packets(with_a=True))
            assert np.array_equal(got[: R[key].shape[0]], R[key]), key


@pytest.mark.gpu
def test_gpu_two_layer_solver_equals_the_executed_driver():
    """the on-device two-layer QG solver (swrt_qg2_*: B, expm(factor_L dt) and the AB3 history on the GPU) from the executed
    driver's initial spectra: its states at the start of steps 2, 4, 7"""
    import swraytracing_b200 as S
    nx, Lq = 32, 20.0
    st = R["qg2_driver_states"]
    dt = float(str(R["qg2_driver_log"]).split("Initial time step: ")[1].split()[0])
    r = O.qg2layersw_driver(nx, 0, 2, 600, 100, 0.3, 3.0, 1.0, max_steps=0)
    assert abs(r["dt"] - dt) < 1e-6
    g2 = S.QG2Flow(nx, Lq, st[0][:, :, 0], st[0][:, :, 1], 3.0, 0.0, 0.5, 0.4, 0.1 * (Lq / nx) ** 8, 4)
    assert abs(g2.max_speed() - r["U0"]) < 1e-12 * r["U0"]
    done = 0
    for steps, ref in zip((1, 3, 6), st[1:]):
        while done < steps:
            g2.step(r["dt"]); done += 1
        got = np.stack([g2.get(0), g2.get(1)], axis=2)
        assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-12, steps
    g2.close()


@pytest.mark.gpu
def test_gpu_theoretical_omega_pdf_equals_the_executed_script():
    """reference_api.ideal_omega_distribution (swrt_ideal_omega_hist: evaluation + binning on the device) on the same scheme:
    the counts of the executed ideal_omega_distribution.m, bin for bin"""
    from swraytracing_b200 import reference_api as A
    import swraytracing_b200 as S
    sch = A.SpectralScheme(L, NX, O.k2g(H["psik"]), mode=S.MODE_LAGRANGE6, f=F0, gH=1.0)
    counts, pdf = A.ideal_omega_distribution(sch, F0, 1.0, 3.0, R["ideal_edges"])
    assert np.array_equal(np.asarray(counts, dtype=np.uint64), R["ideal_counts"].astype(np.uint64))
    assert abs(float((pdf * np.diff(R["ideal_edges"])).sum()) - R["ideal_counts"].sum() / float(R["ideal_total"])) < 1e-12


@pytest.mark.gpu
def test_gpu_raytrace_driver_equals_the_executed_script():
    """drivers.raytrace (step_packet on the device, LAGRANGE6) on the reference's own script output: 100 steps within 1e-9,
    300 within 1e-7 (k has grown eightfold by then)"""
    from swraytracing_b200 import drivers
    out = drivers.raytrace(np_=5, nsteps=301)
    P = out["P"]
    assert out["dt"] == float(R["raytrace_dt"])
    for j, c in enumerate("xykl"):
        assert np.array_equal(P[c][:, 0], R["raytrace_P0"][:, j]), c
        assert np.abs(P[c][0, :101] - R["raytrace_p1"][:101, j]).max() <= 1e-9, c
        assert np.abs(P[c][0, :301] - R["raytrace_p1"][:, j]).max() <= 1e-7, c

@pytest.mark.gpu
def test_gpu_rhs_equals_the_nested_reference_odefun():
    """generate_raytracing_ode through the product (swrt_set_packets + swrt_rhs, LAGRANGE6): bit-identical to the reference's
    odefun at t = 0 (one frame) and within 1e-12 of the plane at blended times; SPECTRAL / NUFFT modes under the degree-5
    interpolation bound"""
    from swraytracing_b200 import reference_api as A
    import swraytracing_b200 as S
    x, y, k, l = (H[n] for n in ("x", "y", "k", "l"))
    yv = np.concatenate([x, y, k, l])
    bf1, bf2 = frames()
    ode = A.generate_raytracing_ode(bf1, bf2, x.size, F0, 1.0, TMAX, DX)
    for tag, t in (("t0", 0.0), ("tmid", 0.25 * TMAX), ("tend", TMAX)):
        got = ode(t, yv)
        ref = R["odefun_" + tag]
        assert np.array_equal(got, ref), (tag, np.abs(got - ref).max())


@pytest.mark.gpu
def test_gpu_interpolate_at_the_awkward_places_equals_both_reference_copies():
    from swraytracing_b200 import reference_api as A
    from swraytracing_b200.engine import interpolate_dev
    ex, ey = R["edge_x"], R["edge_y"]
    for j in range(2):
        g = H["grids"][j]
        assert np.array_equal(A.interpolate(ex, ey, g, DX, DX), R["edge_interpolate_live"][j])
        assert np.array_equal(interpolate_dev(ex, ey, g, DX, DX, 1e-10), R["edge_interpolate_qg"][j])


@pytest.mark.gpu
def test_gpu_interpolate_par_and_grid_U_equal_the_reference():
    from swraytracing_b200 import reference_api as A
    x, y = H["x"], H["y"]
    for j, g in enumerate(H["grids"]):
        assert np.array_equal(A.interpolate_par(x, y, g, DX, DX), R["interpolate_par"][j])
    flow = A.grid_U(R["update_qk_in"], 3.0, K2, KX, KY, float(R["grid_U_shear_value"]))
    for j, nm in enumerate(NAMES):
        assert rel(flow[nm], R["grid_U_shear"][j]) <= 1e-14, nm


@pytest.mark.gpu
def test_gpu_qg_solver_first_step_equals_the_reference_update():
    """swrt_qg_create + one swrt_qg_step = Euler start-up of qgsw_raytrace.m:117-136: qk1 = Ef .* (qk + dt * update(qk, ...)),
    with ``update``, ``filter`` and ``inertial_ring`` as the reference's own local functions returned them"""
    from swraytracing_b200.engine import QGFlow
    qk = R["update_qk_in"]
    dt = 1e-3
    f, Cg = 3.0, 0.25
    upd = O.qg_update(qk, K2, 3.0, 0.3, 0.1, R["inertial_ring"], KX, KY)
    assert np.array_equal(upd, R["update"])
    want = R["filter"] * (qk + dt * R["update"])
    qg = QGFlow(NX, L, qk, 3.0, dt, f, Cg, beta=0.3, r_drag=0.1, force_strength=0.1)
    qg.step(1)
    got = qg.get()
    qg.close()
    assert rel(got, want) <= 1e-13


@pytest.mark.gpu
def test_gpu_raytrace_sw_driver_equals_the_executed_script():
    """drivers.raytrace_sw (BASELINE config 5's caller: device k2g for the projection, step_packet_xka on the device) on the
    executed script's output: fields to 1e-14 of each plane, 100 steps of packet 1 within 1e-9, 150 within 1e-8"""
    from swraytracing_b200 import drivers
    out = drivers.raytrace_sw(R["rsw_S"], 3.0, 1.0, np_=10, nsteps=151)
    assert abs(out["dt"] - float(R["rsw_dt"])) < 1e-15 and abs(out["U0"] - float(R["rsw_U0"])) < 1e-13
    got = [out["U"]["u"], out["U"]["v"]] + [out["GradU"][c] for c in ("u_x", "u_y", "v_x", "v_y")] + [out["H"]]
    for j, g in enumerate(got):
        assert rel(g, R["rsw_fields"][j]) <= 1e-14, j
    P = out["P"]
    for j, c in enumerate("xykla"):
        assert np.array_equal(P[c][:, 0], R["rsw_P0"][:, j]), c
        assert np.abs(P[c][0, :101] - R["rsw_p1"][:101, j]).max() <= 1e-9, c
        assert np.abs(P[c][0, :151] - R["rsw_p1"][:, j]).max() <= 1e-8, c


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["SPECTRAL", "NUFFT", "LAGRANGE6"])
def test_gpu_config_1_zero_background_flow_equals_the_executed_reference(mode):
    """config 1 on the device, all three modes: five fused leapfrog steps over a zero flow == the reference's own run"""
    import swraytracing_b200 as S
    x, y, k, l = (R["c1_" + c] for c in "xykl")
    with S.Engine(NX, L, 3.0, 1.0, getattr(S, "MODE_" + mode)) as e:
        e.set_flow_spectral(np.zeros((NX - 1, NX // 2), dtype=complex))
        e.set_packets(x, y, k, l)
        e.step(S.SCHEME_LEAPFROG, 0.01, 5)
        got = np.stack(e.get_packets())
    assert np.array_equal(got[2:], R["c1_final"][2:])
    assert np.abs(got[:2] - R["c1_final"][:2]).max() <= 1e-13


@pytest.mark.gpu
def test_gpu_config_1_script_right_hand_side_equals_the_nested_reference_function():
    """swrt_rhs with SWRT_FLAG_RHS_GH (dx/dt = U + gH k/omega) in LAGRANGE6 mode on the scheme's own planes"""
    import swraytracing_b200 as S
    from swraytracing_b200.engine import FLAG_RHS_GH
    x, y, k, l = (H[c] for c in "xykl")
    with S.Engine(NX, L, F0, 1.7, S.MODE_LAGRANGE6, flags=FLAG_RHS_GH) as e:
        e.set_flow_spectral(O.g2k(O.k2g(H["psik"])))
        e.set_packets(x, y, k, l)
        got = np.concatenate(e.rhs(0.0))
    assert rel(got, R["swz_odefun"]) <= 1e-12


@pytest.mark.gpu
def test_gpu_qgsw_driver_with_packets_equals_the_executed_driver(tmp_path):
    """drivers.qgsw_raytrace (device QG solver, both frames resident, ode23 with the stages on the device) in LAGRANGE6 mode:
    the packets after six flow steps and the packet files it writes, against the executed qgsw_raytrace.m"""
    import swraytracing_b200 as S
    from swraytracing_b200 import drivers
    ref = R["qgsw_packets_y"]
    out = drivers.qgsw_raytrace(32, 12, 2, 6000, 0, 0.5, 3.0, 1.0, outdir=str(tmp_path), max_steps=6, mode=S.MODE_LAGRANGE6,
                                log=lambda s: None)
    assert np.abs(np.concatenate(out["packets"]) - ref[6]).max() <= 1e-9
    for nm in ("packet_x", "packet_k", "packet_time"):
        got = np.fromfile(tmp_path / f"{nm}.bin")
        want = R["qgsw_file_" + nm]
        assert got.size == want.size and np.abs(got - want).max() <= 1e-9, nm
