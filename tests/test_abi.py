"""The C-ABI library loads and exports every symbol include/swrt.h declares (no compute calls)."""
import ctypes
import re
from pathlib import Path

import pytest

import swraytracing_b200 as S
from swraytracing_b200 import engine

ROOT = Path(__file__).resolve().parent.parent


def _declared_symbols():
    text = (ROOT / "include" / "swrt.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(swrt_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported():
    lib = S.load_library()
    syms = _declared_symbols()
    assert len(syms) >= 25
    for name in syms:
        assert hasattr(lib, name), f"{name} declared in swrt.h but not exported by libswrt.so"


def test_ctypes_table_matches_header():
    assert sorted(engine.SIGNATURES) == _declared_symbols()


def test_version_and_struct_layout():
    lib = S.load_library()
    assert lib.swrt_version() == 200
    assert ctypes.sizeof(engine._Params) == 56      # 4 x int32 + 4 x double + 2 x int32 (ngpu, reserved), as swrt_params


def test_no_cpu_fallback_without_device():
    lib = S.load_library()
    if lib.swrt_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(S.SwrtError) as ei:
        S.Engine(32, 6.28, 3.0, 1.0)
    assert ei.value.code == -3 and "no CPU path" in str(ei.value)
    import numpy as np
    with pytest.raises(S.SwrtError):
        S.interpolate_dev(np.zeros(4), np.zeros(4), np.zeros((8, 8)), 1.0, 1.0)


def test_create_argument_validation():
    lib = S.load_library()
    h = ctypes.c_void_p()
    bad = engine._Params(7, 0, 0, 0, 6.28, 3.0, 1.0, 1e-13)      # odd nx
    assert lib.swrt_create(ctypes.byref(bad), ctypes.byref(h)) == -1
    assert b"nx" in lib.swrt_last_error(None)
    bad = engine._Params(32, 5, 0, 0, 6.28, 3.0, 1.0, 1e-13)     # unknown mode
    assert lib.swrt_create(ctypes.byref(bad), ctypes.byref(h)) == -1
    assert lib.swrt_create(None, ctypes.byref(h)) == -1
    bad = engine._Params(32, 0, 0, 0, 6.28, 3.0, 1.0, 1e-13, -2, 0)     # negative device count
    assert lib.swrt_create(ctypes.byref(bad), ctypes.byref(h)) == -1
    assert b"ngpu" in lib.swrt_last_error(None)
    assert lib.swrt_destroy(None) == 0


def test_product_does_not_import_oracle():
    for py in (ROOT / "swraytracing_b200").glob("*.py"):
        src = py.read_text()
        assert "import oracle" not in src and "from oracle" not in src, py
    for cu in (ROOT / "swraytracing_b200" / "csrc").glob("*"):
        assert "oracle" not in cu.read_text().lower(), cu


def test_library_is_sm100a_with_dmma_and_bulk_copy():
    import shutil, subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    out = subprocess.run(["cuobjdump", "-sass", str(engine.LIB_PATH)], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "DMMA.8x8x4" in out          # fp64 tensor pipe
    assert "UBLKCP" in out              # cp.async.bulk (TMA engine) staging of the coefficient stack


def test_mex_gateway_compiles():
    """matlab/swrt_mex.c against the stub mex.h (neither mkoctfile nor mex exists in this image)"""
    import shutil, subprocess
    if not shutil.which("gcc"):
        pytest.skip("gcc not on PATH")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", f"-I{ROOT / 'matlab' / 'stub'}",
                        f"-I{ROOT / 'include'}", str(ROOT / "matlab" / "swrt_mex.c")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    text = (ROOT / "matlab" / "swrt_mex.c").read_text()
    # every command the .m shims send exists in the gateway
    import re
    cmds = set()
    for m in (ROOT / "matlab" / "shims").glob("*.m"):
        cmds |= set(re.findall(r"swrt_mex\('([a-z0-9_]+)'", m.read_text()))
    assert cmds and all(f'"{c}"' in text for c in cmds), cmds


def test_spectral_geometry_fits_shared_memory_for_every_size():
    """host-only: for every even grid size up to 130, a selection up to 1024, and every plane count / m-tile choice the dense kernel's dynamic
    shared memory (chunk ring + barriers + twiddle table) stays inside the 227 KB a CTA may opt into, the ring has at
    least three chunks, chunks tile a pass, and the twiddle table (when on) has one double per lane per k-step per warp"""
    from swraytracing_b200.engine import spectral_geometry
    seen_on = seen_off = 0
    for nx in list(range(4, 132, 2)) + [160, 192, 200, 250, 256, 258, 320, 384, 500, 512, 640, 768, 1000, 1024]:
        for npl in range(1, 8):
            for mt in (1, 2):
                g = spectral_geometry(nx, npl, mt)
                assert g["smem_bytes"] <= 227 * 1024, (nx, npl, mt, g)
                assert g["nstages"] >= 3 and g["nstages"] <= 8
                assert g["ksteps"] % g["kc"] == 0 and g["kc"] % 4 == 0
                assert 2 * g["ksteps"] >= nx // 2                                  # kx = 0..kmax, two per k-step
                assert g["chunk_bytes"] == g["kc"] * g["ntiles"] * 256
                assert g["stack_bytes"] == g["npass"] * g["ksteps"] * g["ntiles"] * 256
                assert g["smem_bytes"] == g["nstages"] * g["chunk_bytes"] + 128 + g["table_bytes"]
                if g["twiddle_table"] == 1:                 # table in shared memory, beside the ring
                    assert mt == 1 and g["table_bytes"] == g["ksteps"] * 32 * 8 * 8
                    seen_on += 1
                else:                                       # 2: table in the global / L2 scratch; 0 (two m-tiles): rotation
                    assert g["table_bytes"] == 0 and g["twiddle_table"] == (2 if mt == 1 else 0)
                    seen_off += 1
    assert seen_on and seen_off
    assert spectral_geometry(128, 3, 1)["twiddle_table"] == 1
    assert spectral_geometry(256, 3, 1)["twiddle_table"] == 2 and spectral_geometry(256, 3, 1)["chunk_bytes"] == 48 * 1024
    assert spectral_geometry(512, 3, 1)["twiddle_table"] == 2
    lib = S.load_library()
    assert lib.swrt_spectral_geometry(7, 3, 1, (ctypes.c_int64 * 10)()) == -1
