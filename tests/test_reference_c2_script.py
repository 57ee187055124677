"""BASELINE config 2's driver executed: ``symplectic_full_fourier.m``, unmodified and to the end, against the oracle and the product.

``tests/golden/reference_c2_script.npz`` (``tests/golden/run_reference_c2_script.py``, ~15 minutes of ``oracle/minimat``) is what the
reference's own script leaves in its workspace when started in a folder that holds a 128^2 ``Resolution:`` line in the run log it
parses and a seeded PV frame where it reads ``analysis/pv``: U0, Fr, dt, Tend, the ring of ten packets drawn with ``rng(123)``, the
whole leapfrog history (every 8th row stored) and the relative drift of the absolute frequency omega + U.k -- the quantity the
script exists to plot.

CPU: the restated driver (``oracle.symplectic_full_fourier_driver``) gives the same doubles, history and drift series included;
the generator re-run at a small size agrees with it too.  ``-m gpu``: ``drivers.symplectic_full_fourier`` in LAGRANGE6 mode follows
the executed script (100 steps within 1e-9, the whole drift series to 1e-6), and the dense SPECTRAL mode -- the headline kernel,
which evaluates the exact Fourier series where the reference interpolates -- keeps the same frequency drift envelope.
"""
import json
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests" / "golden"))

from oracle import swrt_oracle as O          # noqa: E402

GOLD = ROOT / "tests" / "golden"
D = np.load(GOLD / "reference_c2_script.npz")
# a checkout of the original MATLAB project (ndefilippis/SWRaytracing), which this repository does not carry
REF = Path(os.environ.get("SWRT_REFERENCE_DIR", "")).absolute()
HAVE_REF = bool(os.environ.get("SWRT_REFERENCE_DIR")) and (REF / "ode_symplectic.m").exists()
NX, F, CG = int(D["nx"]), float(D["f"]), float(D["Cg"])


def test_golden_is_the_full_run_of_the_unmodified_script():
    prov = json.loads(str(D["provenance"]))
    ex = set(prov["reference_files_executed"])
    assert {"symplectic_full_fourier.m", "SpectralScheme.m", "RaytracingScheme.m", "ode_symplectic.m", "ray_trace_sw/interpolate.m",
            "qg_flow_ray_trace/read_field.m", "rsw/g2k.m", "rsw/k2g.m", "rsw/fulspec.m"} <= ex
    assert NX == 128 and F == 3.0 and CG == 1.0                                 # parse_data on the log header
    nrows = int(D["nrows"])
    assert nrows == int(np.floor(float(D["Tend"]) / float(D["dt"]))) and nrows > 1000          # ode_symplectic.m:2
    assert float(D["Tend"]) == 10 / (F * float(D["Fr"]) ** 2) and float(D["dt"]) == 0.1 * (2 * np.pi / NX) / max(CG, float(D["U0"]))
    assert D["solver_error"].shape == (nrows, 10) and np.abs(D["solver_error"][0]).max() == 0.0
    assert 1e-6 < np.abs(D["solver_error"]).max() < 0.2                         # the drift the script plots: small, not zero
    if HAVE_REF:
        import hashlib
        for rel, sha in prov["reference_files_executed"].items():
            assert hashlib.sha256((REF / rel).read_bytes()).hexdigest() == sha, rel


def test_oracle_driver_gives_the_same_doubles_as_the_executed_script():
    r = O.symplectic_full_fourier_driver(D["q"], NX, F, CG)
    assert r["U0"] == float(D["U0"]) and r["Fr"] == float(D["Fr"]) and r["dt"] == float(D["dt"]) and r["Tend"] == float(D["Tend"])
    assert r["solver_x"].shape[0] == int(D["nrows"])
    assert np.array_equal(r["solver_x"][0], D["x0"][0]) and np.array_equal(r["solver_k"][0], D["k0"][0])
    assert np.array_equal(r["solver_x"][::8], D["solver_x_every8"]) and np.array_equal(r["solver_k"][::8], D["solver_k_every8"])
    assert np.array_equal(r["solver_x"][-1], D["solver_x_last"]) and np.array_equal(r["solver_k"][-1], D["solver_k_last"])
    assert np.array_equal(np.asarray(r["solver_t"]).ravel()[::8], D["solver_t_every8"])
    assert np.array_equal(np.squeeze(r["solver_error"]), D["solver_error"])


@pytest.mark.skipif(not HAVE_REF, reason="set SWRT_REFERENCE_DIR to a checkout of the original MATLAB project")
def test_rerunning_the_script_at_a_small_size_agrees_with_the_oracle(tmp_path):
    """the same generator on a 32^2 log line and a stronger flow (56 history rows, half a minute): U0, dt, Tend, the last
    row of the history and the whole drift series equal the restated driver's bit for bit"""
    import run_reference_c2_script as G
    out = tmp_path / "c2.npz"
    G.main(["--ref", str(REF), "--nx", "32", "--amp", "4", "--out", str(out)])
    N = np.load(out)
    r = O.symplectic_full_fourier_driver(N["q"], 32, float(N["f"]), float(N["Cg"]))
    assert (r["U0"], r["dt"], r["Tend"]) == (float(N["U0"]), float(N["dt"]), float(N["Tend"]))
    assert np.array_equal(r["solver_x"][-1], N["solver_x_last"]) and np.array_equal(r["solver_k"][-1], N["solver_k_last"])
    assert np.array_equal(np.squeeze(r["solver_error"]), N["solver_error"])
    assert "Fr =" in str(N["stdout"])                                    # the script's unsuppressed  Fr = U0/Cg


@pytest.mark.gpu
def test_gpu_driver_follows_the_executed_script():
    import swraytracing_b200 as S
    from swraytracing_b200 import drivers
    r = drivers.symplectic_full_fourier(D["q"], nx=NX, f=F, Cg=CG, mode=S.MODE_LAGRANGE6)
    assert abs(r["U0"] - float(D["U0"])) <= 1e-13 * float(D["U0"]) and abs(r["dt"] - float(D["dt"])) <= 1e-15
    sx, sk = np.asarray(r["solver_x"]), np.asarray(r["solver_k"])
    assert sx.shape[0] == int(D["nrows"])
    assert np.array_equal(sx[0], D["x0"][0]) and np.array_equal(sk[0], D["k0"][0])
    rows = np.arange(0, 104, 8)                                          # stored rows within the first 100 steps
    assert np.abs(sx[rows] - D["solver_x_every8"][: rows.size]).max() <= 1e-9
    assert np.abs(sk[rows] - D["solver_k_every8"][: rows.size]).max() <= 1e-9
    err = np.squeeze(np.asarray(r["solver_error"]))
    assert np.abs(err - D["solver_error"]).max() <= 1e-6                 # the whole run: grid planes differ by cuFFT round-off
    # the headline mode evaluates the exact series instead of interpolating it: not the same trajectories, the same physics --
    # the drift of the absolute frequency stays inside the same envelope
    r2 = drivers.symplectic_full_fourier(D["q"], nx=NX, f=F, Cg=CG, mode=S.MODE_SPECTRAL)
    e2 = np.abs(np.squeeze(np.asarray(r2["solver_error"])))
    ref = np.abs(D["solver_error"])
    assert 0.5 * ref.max() < e2.max() < 2.0 * ref.max()
    assert np.abs(e2[:200] - ref[:200]).max() < 1e-4                     # and early on the two still agree closely


# ------------------------------------------------------------------------------------------------------------------ config 1
# SW_zero_background_raytracing.m executed to the end on a 32^2 frame (tests/golden/run_reference_c2_script.py --c1 ->
# reference_c1_script.npz).  Its integrator is MATLAB's ode23 (a builtin, not reference code: served by the restated controller,
# with the script's own RelTol 1e-6 / AbsTol 1e-7 and dense output at dt*(0:Nsteps)); everything else -- parse_data, read_field,
# SpectralScheme, the packet ring, initialize_raytracing / odefun, the Omega series -- is the reference's own code.
C1 = np.load(GOLD / "reference_c1_script.npz")


def test_config_1_script_ran_to_its_end():
    prov = json.loads(str(C1["provenance"]))
    assert {"SW_zero_background_raytracing.m", "SpectralScheme.m", "RaytracingScheme.m", "ray_trace_sw/interpolate.m",
            "qg_flow_ray_trace/read_field.m", "qg_flow_ray_trace/grid_U.m"} <= set(prov["reference_files_executed"])
    assert "ode23 with 1e-5 tol:" in str(C1["stdout"]) and "Nsteps =" in str(C1["stdout"])          # the script's own printing
    n = int(C1["Nsteps"])
    assert n == int(np.floor(float(C1["Tend"]) / float(C1["dt"]))) and float(C1["Tend"]) == 1 / (3.0 * float(C1["Fr"]) ** 2)
    assert C1["solver_x"].shape == (n + 1, 2, 10) and C1["solver_error"].shape == (10, n + 1) and C1["w"].shape == (n + 1, 10)
    assert int(C1["ode23_nsteps"]) > n                                    # RelTol 1e-6 takes several steps per output interval
    if HAVE_REF:
        import hashlib
        for rel, sha in prov["reference_files_executed"].items():
            assert hashlib.sha256((REF / rel).read_bytes()).hexdigest() == sha, rel


def test_oracle_config_1_driver_gives_the_same_doubles_as_the_executed_script():
    r = O.sw_zero_background_driver(C1["q"], 32, float(C1["f"]), float(C1["Cg"]))
    assert (r["U0"], r["dt"], r["Nsteps"]) == (float(C1["U0"]), float(C1["dt"]), int(C1["Nsteps"]))
    assert (r["stats"]["nsteps"], r["stats"]["nfailed"]) == (int(C1["ode23_nsteps"]), int(C1["ode23_nfailed"]))
    assert np.array_equal(r["t_hist"], C1["t_hist"])
    assert np.array_equal(r["solver_x"], C1["solver_x"]) and np.array_equal(r["solver_k"], C1["solver_k"])
    assert np.array_equal(np.squeeze(r["solver_error"]), C1["solver_error"].T)


@pytest.mark.gpu
def test_gpu_config_1_driver_follows_the_executed_script():
    """drivers.SW_zero_background_raytracing: ode23 with its stages, error norm and dense output on the device (LAGRANGE6 mode,
    SWRT_FLAG_RHS_GH): the same accept / reject decisions as the executed script's run and its history within 1e-9"""
    import swraytracing_b200 as S
    from swraytracing_b200 import drivers
    r = drivers.SW_zero_background_raytracing(C1["q"], nx=32, f=float(C1["f"]), Cg=float(C1["Cg"]), mode=S.MODE_LAGRANGE6)
    assert r["Nsteps"] == int(C1["Nsteps"]) and abs(r["dt"] - float(C1["dt"])) < 1e-15
    assert (r["stats"]["nsteps"], r["stats"]["nfailed"]) == (int(C1["ode23_nsteps"]), int(C1["ode23_nfailed"]))
    assert np.abs(np.asarray(r["solver_x"]) - C1["solver_x"]).max() <= 1e-9
    assert np.abs(np.asarray(r["solver_k"]) - C1["solver_k"]).max() <= 1e-9
    assert np.abs(np.squeeze(np.asarray(r["solver_error"])) - C1["solver_error"].T).max() <= 1e-9
