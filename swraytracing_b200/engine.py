"""ctypes binding of libswrt.so (include/swrt.h) -- the tested skin of the C ABI.

``Engine`` is a thin 1:1 wrapper: every method is one C call on host numpy buffers.  There is no
CPU fallback: if the library is missing or no CUDA device is present the constructor raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libswrt.so"

MODE_SPECTRAL, MODE_LAGRANGE6, MODE_NUFFT = 0, 1, 2
SCHEME_LEAPFROG, SCHEME_RK4_PACKET, SCHEME_RK4_XKA = 0, 1, 2
HIST_INTRINSIC, HIST_ABSOLUTE = 0, 1
FLAG_RHS_GH = 1
EVENT_X, EVENT_Y, EVENT_K, EVENT_L, EVENT_KMAG, EVENT_OMEGA = 0, 1, 2, 3, 4, 5
MAX_EVENTS = 8
Q_XMOD, Q_YMOD, Q_K, Q_L, Q_KMAG, Q_THETA, Q_OMEGA, Q_OMEGA_ABS = 0, 1, 2, 3, 4, 5, 6, 7
W_ACTION, W_ENERGY, W_PSEUDO_K, W_PSEUDO_L = 0, 1, 2, 3
MAX_WEIGHTS = 4

_dp = C.POINTER(C.c_double)


class _Event(C.Structure):
    _fields_ = [("kind", C.c_int32), ("direction", C.c_int32), ("terminal", C.c_int32), ("reserved", C.c_int32),
                ("level", C.c_double)]


class SwrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libswrt error {code}: {msg}")
        self.code = code


class _Params(C.Structure):
    _fields_ = [("nx", C.c_int32), ("mode", C.c_int32), ("device", C.c_int32), ("flags", C.c_int32),
                ("L", C.c_double), ("f", C.c_double), ("gH", C.c_double), ("bump", C.c_double),
                ("ngpu", C.c_int32), ("reserved", C.c_int32)]


# name -> (restype, argtypes); every symbol include/swrt.h declares
SIGNATURES = {
    "swrt_version": (C.c_int, []),
    "swrt_device_count": (C.c_int, []),
    "swrt_create": (C.c_int, [C.POINTER(_Params), C.POINTER(C.c_void_p)]),
    "swrt_destroy": (C.c_int, [C.c_void_p]),
    "swrt_last_error": (C.c_char_p, [C.c_void_p]),
    "swrt_set_flow_spectral": (C.c_int, [C.c_void_p, C.c_int, _dp, _dp, C.c_int, C.c_int, C.c_double]),
    "swrt_set_flow_planes_spectral": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(_dp), C.POINTER(_dp), C.c_int, C.c_int, C.c_int]),
    "swrt_set_flow_grid": (C.c_int, [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int]),
    "swrt_set_packets": (C.c_int, [C.c_void_p, C.c_int64, _dp, _dp, _dp, _dp, _dp]),
    "swrt_get_packets": (C.c_int, [C.c_void_p, _dp, _dp, _dp, _dp, _dp]),
    "swrt_num_packets": (C.c_int64, [C.c_void_p]),
    "swrt_num_devices": (C.c_int, [C.c_void_p]),
    "swrt_shard_info": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "swrt_packets_alloc_dev": (C.c_int, [C.c_void_p, C.c_int64]),
    "swrt_packets_dev": (C.c_int, [C.c_void_p] + [C.POINTER(C.c_void_p)] * 5),
    "swrt_eval": (C.c_int, [C.c_void_p, C.c_double] + [_dp] * 6),
    "swrt_eval_at": (C.c_int, [C.c_void_p, C.c_double, C.c_int64, _dp, _dp] + [_dp] * 7),
    "swrt_rhs": (C.c_int, [C.c_void_p, C.c_double] + [_dp] * 4),
    "swrt_interpolate": (C.c_int, [C.c_int, _dp, _dp, C.c_int64, _dp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, _dp]),
    "swrt_step": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double]),
    "swrt_step_async": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double]),
    "swrt_step_host": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int64] + [_dp] * 10),
    "swrt_hist_omega": (C.c_int, [C.c_void_p, C.c_int, C.c_double, _dp, C.c_int, C.POINTER(C.c_uint64), C.c_int]),
    "swrt_bs23_begin": (C.c_int, [C.c_void_p, C.c_double, C.c_double, _dp]),
    "swrt_bs23_attempt": (C.c_int, [C.c_void_p, C.c_double, _dp, C.c_double, _dp]),
    "swrt_bs23_accept": (C.c_int, [C.c_void_p]),
    "swrt_bs23_interp": (C.c_int, [C.c_void_p, C.c_double, C.c_double] + [_dp] * 4),
    "swrt_ode23": (C.c_int, [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _dp, C.POINTER(C.c_int64), _dp, C.c_int]),
    "swrt_ode23_packets": (C.c_int, [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _dp, C.POINTER(C.c_int32), _dp,
                                     C.POINTER(C.c_int64)]),
    "swrt_ode23_packets_tspans": (C.c_int, [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _dp, C.POINTER(C.c_int32),
                                            _dp, C.POINTER(C.c_int64)]),
    "swrt_ode23_packets_events": (C.c_int, [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_double, C.POINTER(_Event), C.c_int,
                                            C.c_int, _dp, C.POINTER(C.c_int32), _dp, _dp, _dp, C.POINTER(C.c_int32),
                                            C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "swrt_ode23_packets_tspans_events": (C.c_int, [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_double, C.POINTER(_Event),
                                                   C.c_int, C.c_int, _dp, C.POINTER(C.c_int32), _dp, _dp, _dp, C.POINTER(C.c_int32),
                                                   C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "swrt_hist_omega_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_double, _dp, C.c_int, C.POINTER(C.c_void_p)]),
    "swrt_hist_omega_launch": (C.c_int, [C.c_void_p, C.c_int, C.c_double, _dp, C.c_int, C.POINTER(C.c_void_p)]),
    "swrt_hist_omega_wait": (C.c_int, [C.c_void_p]),
    "swrt_ideal_omega_hist": (C.c_int, [C.c_void_p, C.c_double, C.c_int64, _dp, _dp, _dp, _dp, C.c_int, C.c_double, _dp, C.c_int,
                                        C.POINTER(C.c_uint64)]),
    "swrt_diag": (C.c_int, [C.c_void_p, C.c_double, _dp]),
    "swrt_omega": (C.c_int, [C.c_void_p, C.c_double, _dp, _dp]),
    "swrt_packet_quantity": (C.c_int, [C.c_void_p, C.c_int, C.c_double, _dp]),
    "swrt_hist2": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_double, C.POINTER(C.c_uint64), C.c_int]),
    "swrt_weight_scale": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_int, C.c_double, C.POINTER(C.c_int32)]),
    "swrt_hist2_sums": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_double, C.POINTER(C.c_int32),
                                  C.c_int, C.POINTER(C.c_int32), _dp, C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]),
    "swrt_fixed_sums_to_double": (C.c_int, [C.POINTER(C.c_int64), C.c_int64, C.c_int, C.POINTER(C.c_int32), _dp]),
    "swrt_g2k": (C.c_int, [C.c_int, _dp, C.c_int, _dp, _dp]),
    "swrt_k2g": (C.c_int, [C.c_int, _dp, _dp, C.c_int, _dp]),
    "swrt_qg_create": (C.c_int, [C.c_int, C.c_int] + [C.c_double] * 8 + [_dp, _dp, C.POINTER(C.c_void_p)]),
    "swrt_qg_step": (C.c_int, [C.c_void_p, C.c_int]),
    "swrt_qg_get": (C.c_int, [C.c_void_p, _dp, _dp]),
    "swrt_qg_get_grid": (C.c_int, [C.c_void_p, _dp]),
    "swrt_qg_destroy": (C.c_int, [C.c_void_p]),
    "swrt_set_flow_from_qg": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_double]),
    "swrt_qg2_create": (C.c_int, [C.c_int, C.c_int] + [C.c_double] * 7 + [_dp] * 4 + [C.POINTER(C.c_void_p)]),
    "swrt_qg2_max_speed": (C.c_int, [C.c_void_p, _dp]),
    "swrt_qg2_step": (C.c_int, [C.c_void_p, C.c_double]),
    "swrt_qg2_get": (C.c_int, [C.c_void_p, C.c_int, _dp, _dp]),
    "swrt_qg2_destroy": (C.c_int, [C.c_void_p]),
    "swrt_set_flow_from_qg2": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "swrt_launch_count": (C.c_int64, [C.c_void_p, C.c_int]),
    "swrt_last_kernel_ms": (C.c_double, [C.c_void_p, C.POINTER(C.c_int)]),
    "swrt_work_per_eval": (C.c_double, [C.c_void_p, C.c_int]),
    "swrt_synchronize": (C.c_int, [C.c_void_p]),
    "swrt_set_tuning": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "swrt_contracted_planes": (C.c_int, [C.c_void_p]),
    "swrt_spectral_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64)]),
    "swrt_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "swrt_gather_probe": (C.c_int, [C.c_int, C.c_int64, C.c_int, _dp]),
    "swrt_timer_start": (C.c_int, [C.c_void_p]),
    "swrt_timer_stop": (C.c_double, [C.c_void_p]),
}

_lib = None


def load_library(path: os.PathLike | None = None):
    """dlopen libswrt.so and declare every prototype.  Raises if the library is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else Path(os.environ.get("SWRT_LIB", LIB_PATH))   # SWRT_LIB: developer A/B builds
    if not p.exists():
        raise FileNotFoundError(f"{p} not found: build it with `make` or `python -c 'import __graft_entry__ as g; g.build()'`"
                                " (libswrt has no CPU fallback)")
    lib = C.CDLL(str(p))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


_nccl_preloaded = False


def _preload_nccl():
    """A multi-device handle makes libswrt dlopen("libnccl.so.2").  The dynamic loader keeps ONE library per soname in a
    process, so whichever NCCL is mapped first also serves everybody else -- e.g. a later ``import torch``, whose
    libtorch_cuda.so needs the symbols of the NCCL release it was built against.  When a pip-installed NCCL (the one torch
    bundles: site-packages/nvidia/nccl/lib) is present, map that one first; otherwise the system library is used."""
    global _nccl_preloaded
    if _nccl_preloaded or os.environ.get("SWRT_NCCL_LIB"):
        return
    _nccl_preloaded = True
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for root in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
            cand = Path(root) / "lib" / "libnccl.so.2"
            if cand.exists():
                C.CDLL(str(cand), mode=C.RTLD_GLOBAL)
                return
    except Exception:
        pass


def spectral_geometry(nx, nplanes=3, mtiles=1):
    """launch geometry of the dense kernel (host-only diagnostic, swrt_spectral_geometry)"""
    out = (C.c_int64 * 10)()
    rc = load_library().swrt_spectral_geometry(int(nx), int(nplanes), int(mtiles), out)
    if rc != 0:
        raise SwrtError(rc, load_library().swrt_last_error(None).decode())
    keys = ("ntiles", "npass", "ksteps", "kc", "nstages", "chunk_bytes", "twiddle_table", "table_bytes", "smem_bytes", "stack_bytes")
    return dict(zip(keys, (int(v) for v in out)))


def gather_probe(table_bytes=1 << 24, reps=5, device=0):
    """measured scattered-gather rate (GB/s) from an L2-resident table: the roofline denominator of the gather modes"""
    out = C.c_double(0.0)
    rc = load_library().swrt_gather_probe(int(device), int(table_bytes), int(reps), C.byref(out))
    if rc != 0:
        raise SwrtError(rc, load_library().swrt_last_error(None).decode())
    return out.value


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _i32p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32)) if a is not None else None


def _weight_kinds(weights):
    """one W_* kind or a sequence of 1..MAX_WEIGHTS of them -> int32 array (checked before any library call)"""
    w = np.atleast_1d(np.asarray(weights))
    if w.ndim != 1 or not 1 <= w.size <= MAX_WEIGHTS or not np.issubdtype(w.dtype, np.integer):
        raise ValueError(f"weights must be 1..{MAX_WEIGHTS} of W_ACTION, W_ENERGY, W_PSEUDO_K, W_PSEUDO_L, got {weights!r}")
    if not np.all((w >= W_ACTION) & (w <= W_PSEUDO_L)):
        raise ValueError(f"unknown weight kind in {weights!r}")
    return np.ascontiguousarray(w, dtype=np.int32)


def fixed_sums_to_double(acc, scale_exp):
    """swrt_fixed_sums_to_double on the host (no device): ``acc`` int64 of shape ``(nw, nbx, nby, 4)`` as
    ``Engine.hist2_sums(..., return_acc=True)`` returns it (or a sum of such arrays), ``scale_exp`` the nw exponents
    -> the ``(nw, nbx, nby)`` sums, each rounded once"""
    acc = np.asarray(acc)
    if acc.dtype != np.int64 or acc.ndim != 4 or acc.shape[3] != 4:
        raise ValueError(f"acc must be an int64 array of shape (nw, nbx, nby, 4), got {acc.dtype} {acc.shape}")
    nw, nbx, nby, _ = acc.shape
    e = np.ascontiguousarray(np.atleast_1d(scale_exp), dtype=np.int32)
    if e.shape != (nw,):
        raise ValueError(f"scale_exp must hold {nw} exponents, got {e.shape}")
    raw = np.ascontiguousarray(acc.transpose(0, 2, 1, 3))                  # C: acc[4*((v*nby + j)*nbx + i) + c]
    out = np.empty((nw, nby, nbx))
    rc = load_library().swrt_fixed_sums_to_double(raw.ctypes.data_as(C.POINTER(C.c_int64)), nbx * nby, nw, _i32p(e), _ptr(out))
    if rc != 0:
        raise SwrtError(rc, "swrt_fixed_sums_to_double")
    return out.transpose(0, 2, 1)


def _colmajor(a):
    """host array -> flat column-major (MATLAB) float64 copy"""
    return np.asfortranarray(np.asarray(a, dtype=np.float64)).ravel(order="F").copy()


class Engine:
    """One handle = ``ngpu`` CUDA devices (default one) + device-resident packets + flow stacks.  With ``ngpu > 1`` the
    packets are sharded over the devices ``device .. device+ngpu-1`` inside libswrt (one host thread, in-library NCCL
    all-reduce of histograms / diagnostics / the ode23 norm); every method keeps its meaning for the whole ensemble."""

    def __init__(self, nx, L, f, gH, mode=MODE_SPECTRAL, device=0, bump=1e-13, flags=0, ngpu=1):
        self.lib = load_library()
        self.nx, self.L, self.f, self.gH, self.mode, self.device = int(nx), float(L), float(f), float(gH), int(mode), int(device)
        self.ngpu = int(ngpu)
        if self.ngpu > 1:
            _preload_nccl()
        self._h = C.c_void_p()
        prm = _Params(self.nx, self.mode, self.device, int(flags), self.L, self.f, self.gH, float(bump), self.ngpu, 0)
        rc = self.lib.swrt_create(C.byref(prm), C.byref(self._h))
        if rc != 0:
            raise SwrtError(rc, (self.lib.swrt_last_error(None) or b"").decode())
        self.n = 0

    # -- plumbing --
    def _check(self, rc):
        if rc != 0:
            raise SwrtError(rc, (self.lib.swrt_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.swrt_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- flow --
    def set_flow_spectral(self, psik, slot=0, u_mean=0.0):
        """psik: complex (nkx, nky) array in g2k layout (kx = first index)."""
        psik = np.asarray(psik, dtype=np.complex128)
        nkx, nky = psik.shape
        re, im = _colmajor(psik.real), _colmajor(psik.imag)
        self._check(self.lib.swrt_set_flow_spectral(self._h, slot, _ptr(re), _ptr(im), nkx, nky, float(u_mean)))

    def set_flow_planes_spectral(self, planes, slot=0):
        planes = [np.asarray(p, dtype=np.complex128) for p in planes]
        nkx, nky = planes[0].shape
        res = [_colmajor(p.real) for p in planes]
        ims = [_colmajor(p.imag) for p in planes]
        n = len(planes)
        tr = (_dp * n)(*[_ptr(a) for a in res])
        ti = (_dp * n)(*[_ptr(a) for a in ims])
        self._check(self.lib.swrt_set_flow_planes_spectral(self._h, slot, tr, ti, n, nkx, nky))

    def set_flow_grid(self, u, v, ux, uy, vx, vy, H=None, slot=0):
        """gridded planes F[ix, iy] (x = first index, as MATLAB)."""
        arrs = [_colmajor(a) for a in (u, v, ux, uy, vx, vy)]
        h = _colmajor(H) if H is not None else None
        nx = np.asarray(u).shape[0]
        self._check(self.lib.swrt_set_flow_grid(self._h, slot, *[_ptr(a) for a in arrs], _ptr(h), nx))

    # -- packets --
    def set_packets(self, x, y, k, l, a=None):
        x, y, k, l = map(_f64, (x, y, k, l))
        a = _f64(a) if a is not None else None
        self.n = x.size
        self._check(self.lib.swrt_set_packets(self._h, self.n, _ptr(x), _ptr(y), _ptr(k), _ptr(l), _ptr(a)))

    def get_packets(self, with_a=False):
        n = self.n
        out = [np.empty(n) for _ in range(5 if with_a else 4)]
        ptrs = [_ptr(o) for o in out] + ([] if with_a else [None])
        self._check(self.lib.swrt_get_packets(self._h, *ptrs))
        return tuple(out)

    def alloc_packets_dev(self, n):
        self._check(self.lib.swrt_packets_alloc_dev(self._h, int(n)))
        self.n = int(n)

    def packets_dev(self):
        """raw device pointers (ints) of the SoA buffers x,y,k,l,a"""
        ps = [C.c_void_p() for _ in range(5)]
        self._check(self.lib.swrt_packets_dev(self._h, *[C.byref(p) for p in ps]))
        return tuple(p.value for p in ps)

    # -- evaluation --
    def eval(self, alpha=0.0):
        outs = [np.empty(self.n) for _ in range(6)]
        self._check(self.lib.swrt_eval(self._h, float(alpha), *[_ptr(o) for o in outs]))
        return np.stack(outs)

    def eval_at(self, x, y, alpha=0.0, with_H=False):
        x, y = _f64(x).ravel(), _f64(y).ravel()
        n = x.size
        outs = [np.empty(n) for _ in range(7 if with_H else 6)]
        ptrs = [_ptr(o) for o in outs] + ([] if with_H else [None])
        self._check(self.lib.swrt_eval_at(self._h, float(alpha), n, _ptr(x), _ptr(y), *ptrs))
        return np.stack(outs)

    def rhs(self, alpha=0.0):
        outs = [np.empty(self.n) for _ in range(4)]
        self._check(self.lib.swrt_rhs(self._h, float(alpha), *[_ptr(o) for o in outs]))
        return tuple(outs)

    def step(self, scheme, dt, nsteps, alpha0=0.0, dalpha=0.0):
        self._check(self.lib.swrt_step(self._h, int(scheme), float(dt), int(nsteps), float(alpha0), float(dalpha)))

    def step_host(self, scheme, dt, nsteps, x, y, k, l, a=None, alpha0=0.0, dalpha=0.0, out=None):
        """host arrays in -> ``nsteps`` steps -> host arrays out in ONE C call (swrt_step_host: upload, compute and
        download pipelined over packet chunks).  ``out``: optional (x, y, k, l[, a]) arrays to receive the result."""
        x, y, k, l = map(_f64, (x, y, k, l))
        a = _f64(a) if a is not None else None
        self.n = x.size
        if out is None:
            out = [np.empty(self.n) for _ in range(5 if a is not None else 4)]
        ptrs = [_ptr(o) for o in out] + [None] * (5 - len(out))
        self._check(self.lib.swrt_step_host(self._h, int(scheme), float(dt), int(nsteps), float(alpha0), float(dalpha), self.n,
                                            _ptr(x), _ptr(y), _ptr(k), _ptr(l), _ptr(a), *ptrs))
        return tuple(out)

    def shard_info(self, i):
        """(device, lo, n) of shard ``i`` of a multi-device handle"""
        d, lo, n = C.c_int(0), C.c_int64(0), C.c_int64(0)
        self._check(self.lib.swrt_shard_info(self._h, int(i), C.byref(d), C.byref(lo), C.byref(n)))
        return d.value, lo.value, n.value

    def step_async(self, scheme, dt, nsteps, alpha0=0.0, dalpha=0.0):
        """queue the step's kernels and return at once (``synchronize()`` or any blocking call completes them)"""
        self._check(self.lib.swrt_step_async(self._h, int(scheme), float(dt), int(nsteps), float(alpha0), float(dalpha)))

    # -- ode23 building blocks (the controller lives in reference_api.ode23) --
    def bs23_begin(self, alpha, threshold):
        out = C.c_double(0.0)
        self._check(self.lib.swrt_bs23_begin(self._h, float(alpha), float(threshold), C.byref(out)))
        return out.value

    def bs23_attempt(self, hstep, alphas, threshold):
        al = (C.c_double * 3)(*[float(a) for a in alphas])
        out = C.c_double(0.0)
        self._check(self.lib.swrt_bs23_attempt(self._h, float(hstep), al, float(threshold), C.byref(out)))
        return out.value

    def bs23_accept(self):
        self._check(self.lib.swrt_bs23_accept(self._h))

    def bs23_interp(self, hstep, s):
        """ntrp23 dense output of the last attempted step at t + s*hstep -> (x, y, k, l)"""
        out = [np.empty(self.n) for _ in range(4)]
        self._check(self.lib.swrt_bs23_interp(self._h, float(hstep), float(s), *[_ptr(o) for o in out]))
        return tuple(out)

    def ode23(self, tspan, tmax, rtol=1e-3, atol=1e-6, *, trace=0):
        """a whole ``[~, Y] = ode23(ray_ode, tspan, y0)`` solve in one call (swrt_ode23): the decisions of
        ``reference_api.ode23`` made by a controller in device memory, the host waiting a few times per solve instead of
        twice per attempt.  ``tmax`` None / 0 = steady flow.  Returns the same dict as ``reference_api.ode23`` (``Y`` when
        ``tspan`` has more than two entries) plus ``host_waits``, and ``h`` (the first ``trace`` accepted step sizes, signed)
        when ``trace`` > 0.  A decreasing ``tspan`` (``[T 0]``) integrates backward in time, as MATLAB's ode23 does; an
        entry that steps against the direction from ``tspan[0]`` to ``tspan[-1]`` raises SwrtError (SWRT_ERR_ARG).  A step
        size below hmin raises SwrtError (SWRT_ERR_STATE) naming t."""
        ts = _f64(tspan)
        dense = ts.size > 2
        Y = np.empty((ts.size, 4, self.n)) if dense else None
        st = (C.c_int64 * 4)()
        hs = np.empty(max(int(trace), 0))
        self._check(self.lib.swrt_ode23(self._h, _ptr(ts), int(ts.size), float(tmax or 0.0), float(rtol), float(atol),
                                        _ptr(Y) if dense else None, st, _ptr(hs) if trace > 0 else None, int(hs.size)))
        out = {"nsteps": st[0], "nfailed": st[1], "nfevals": st[2], "t": float(ts[-1]), "host_waits": st[3]}
        if dense:
            out["Y"] = Y
        if trace > 0:
            out["h"] = hs[:min(st[0], hs.size)].copy()
        return out

    def ode23_packets(self, tspan, tmax, rtol=1e-3, atol=1e-6, events=None, ev_cap=4):
        """``ode23`` once per packet (swrt_ode23_packets): every packet under its own step-size controller, exactly as
        ``ode23`` advances an ensemble holding that packet alone, so a packet's result does not depend on the others.
        Returns ``ode23``'s dict with ``nsteps``, ``nfailed`` and ``nfevals`` summed over packets, plus ``stopped``
        (packets whose step size fell below hmin: they keep their last accepted state, the others carry on),
        ``host_waits``, and the per-packet arrays ``steps``, ``rejected``, ``status`` (0 reached tfinal, 1 stopped) and
        ``t_end`` (where each packet stopped).  ``Y`` when ``tspan`` has more than two entries (NaN in the rows a stopped
        packet did not reach).  A decreasing ``tspan`` integrates backward in time, as in ``ode23``.

        ``events``: MATLAB's ``odeset('Events', ...)`` per packet (swrt_ode23_packets_events), a list of
        ``(kind, level, direction=0, terminal=False)`` with ``kind`` one of ``EVENT_X``, ``EVENT_Y``, ``EVENT_K``,
        ``EVENT_L``, ``EVENT_KMAG`` (|k|) and ``EVENT_OMEGA`` (omega as ``omega()`` computes it); tspan must be strictly
        increasing.  The result then also holds ``te`` (ev_cap, n), ``ye`` (ev_cap, 4, n) and ``ie`` (ev_cap, n, 1-based
        event index): each packet's first ``ev_cap`` records in ascending (te, ie) order, NaN / 0 where unused; ``ne``
        (events found per packet, may exceed ev_cap); ``events`` (their total) and ``terminated`` (packets stopped by a
        terminal event: status 2, state and ``t_end`` those of the event).

        A 2-D ``tspan`` of shape ``(ntspan, n)`` gives every packet its own (swrt_ode23_packets_tspans): column ``i`` is
        packet ``i``'s tspan, so ``Y[j, :, i]`` is its state at ``tspan[j, i]``, as ``ode23(odefun, tspan(:, i), y0(:, i))``
        gives it.  Each column has its own direction (backward when it decreases); a constant column keeps its packet
        where it is.  ``t`` is then the per-packet array ``tspan[-1]``.  Events need a 1-D ``tspan`` here; with a
        per-packet or decreasing ``tspan`` use ``ode23_packets_tspans_events``."""
        ts = _f64(tspan)
        if ts.ndim == 2:
            if events is not None:
                raise ValueError("ode23_packets: events need one shared (1-D) tspan")
            if ts.shape[0] < 2 or ts.shape[1] != self.n:
                raise ValueError(f"ode23_packets: a per-packet tspan must be (ntspan >= 2, n = {self.n}), got {ts.shape}")
        elif ts.ndim != 1:
            raise ValueError(f"ode23_packets: tspan must be 1-D (shared) or 2-D (ntspan, n), got shape {ts.shape}")
        if events is not None:
            return self._ode23_events(self.lib.swrt_ode23_packets_events, ts, tmax, rtol, atol, events, ev_cap)
        nt = ts.shape[0]
        dense = nt > 2
        Y = np.empty((nt, 4, self.n)) if dense else None
        pstat = np.empty((3, self.n), dtype=np.int32)          # the C side's n x 3 column-major block
        t_end = np.empty(self.n)
        i32 = C.POINTER(C.c_int32)
        if ts.ndim == 2:                                        # C order (ntspan, n) = the C side's n x ntspan column-major
            st = (C.c_int64 * 5)()
            self._check(self.lib.swrt_ode23_packets_tspans(self._h, _ptr(ts), int(nt), float(tmax or 0.0), float(rtol),
                                                           float(atol), _ptr(Y) if dense else None, pstat.ctypes.data_as(i32),
                                                           _ptr(t_end), st))
        else:
            st = (C.c_int64 * 5)()
            self._check(self.lib.swrt_ode23_packets(self._h, _ptr(ts), int(ts.size), float(tmax or 0.0), float(rtol), float(atol),
                                                    _ptr(Y) if dense else None, pstat.ctypes.data_as(i32), _ptr(t_end), st))
        out = {"nsteps": st[0], "nfailed": st[1], "nfevals": st[2], "t": ts[-1].copy() if ts.ndim == 2 else float(ts[-1]),
               "stopped": st[3], "host_waits": st[4],
               "steps": pstat[0].copy(), "rejected": pstat[1].copy(), "status": pstat[2].copy(), "t_end": t_end}
        if dense:
            out["Y"] = Y
        return out

    def ode23_packets_tspans_events(self, tspan, tmax, events, rtol=1e-3, atol=1e-6, ev_cap=4):
        """``ode23`` with ``odeset('Events', ...)`` once per packet, every packet with its own tspan in either direction
        (swrt_ode23_packets_tspans_events): ``for i = 1:n, ode23(odefun, tspan(:, i), y0(:, i), odeset('Events', ...))``.
        ``tspan`` is ``(ntspan, n)`` (column ``i`` is packet ``i``'s, as in ``ode23_packets``) or 1-D, shared by every
        packet in either direction.  ``events`` and ``ev_cap`` as in ``ode23_packets``; everything about them follows each
        packet's direction of integration: rising means rising as the packet integrates (as t decreases when it goes
        backward), records come in order of encounter, and a terminal event stops the packet at the first terminal
        crossing it meets.  Returns ``ode23_packets(events=...)``'s dict with ``t`` the per-packet ``tspan[-1]``."""
        ts = _f64(tspan)
        if ts.ndim == 1 and ts.shape[0] >= 2:           # shared: the same row for every packet
            ts = np.ascontiguousarray(np.broadcast_to(ts[:, None], (ts.shape[0], self.n)))
        elif ts.ndim != 2 or ts.shape[0] < 2 or ts.shape[1] != self.n:
            raise ValueError(f"ode23_packets_tspans_events: tspan must be (ntspan >= 2,) or (ntspan >= 2, n = {self.n}), "
                             f"got shape {ts.shape}")
        return self._ode23_events(self.lib.swrt_ode23_packets_tspans_events, ts, tmax, rtol, atol, events, ev_cap)

    def _ode23_events(self, fn, ts, tmax, rtol, atol, events, ev_cap):
        """the call and result dict of the per-packet solves with events; ts is 1-D (shared) or (ntspan, n)"""
        nt = ts.shape[0]
        dense = nt > 2
        Y = np.empty((nt, 4, self.n)) if dense else None
        pstat = np.empty((3, self.n), dtype=np.int32)          # the C side's n x 3 column-major block
        t_end = np.empty(self.n)
        i32 = C.POINTER(C.c_int32)
        evs = [tuple(e) + (0, False)[len(e) - 2:] for e in events]      # direction 0, not terminal by default
        arr = (_Event * max(len(evs), 1))(*[_Event(int(kind), int(d), int(term), 0, float(level)) for kind, level, d, term in evs])
        cap = max(int(ev_cap), 0)
        te, ye, ie = np.empty((cap, self.n)), np.empty((cap, 4, self.n)), np.empty((cap, self.n), dtype=np.int32)
        ne = np.empty(self.n, dtype=np.int32)
        st = (C.c_int64 * 7)()
        self._check(fn(self._h, _ptr(ts), int(nt), float(tmax or 0.0), float(rtol), float(atol), arr, len(evs), int(ev_cap),
                       _ptr(Y) if dense else None, pstat.ctypes.data_as(i32), _ptr(t_end), _ptr(te), _ptr(ye),
                       ie.ctypes.data_as(i32), ne.ctypes.data_as(i32), st))
        out = {"nsteps": st[0], "nfailed": st[1], "nfevals": st[2], "t": ts[-1].copy() if ts.ndim == 2 else float(ts[-1]),
               "stopped": st[3], "host_waits": st[4],
               "steps": pstat[0].copy(), "rejected": pstat[1].copy(), "status": pstat[2].copy(), "t_end": t_end}
        if dense:
            out["Y"] = Y
        out.update(te=te, ye=ye, ie=ie, ne=ne, events=st[5], terminated=st[6])
        return out

    # -- diagnostics --
    def hist_omega(self, edges, kind=HIST_INTRINSIC, alpha=0.0, counts=None):
        edges = _f64(edges)
        acc = counts is not None
        if counts is None:
            counts = np.zeros(edges.size - 1, dtype=np.uint64)
        self._check(self.lib.swrt_hist_omega(self._h, kind, float(alpha), _ptr(edges), edges.size,
                                             counts.ctypes.data_as(C.POINTER(C.c_uint64)), int(acc)))
        return counts

    def hist_omega_dev(self, edges, kind=HIST_INTRINSIC, alpha=0.0):
        """histogram left on the device: returns (device pointer, nbins) of the handle-owned u64 counts"""
        edges = _f64(edges)
        ptr = C.c_void_p()
        self._check(self.lib.swrt_hist_omega_dev(self._h, kind, float(alpha), _ptr(edges), edges.size, C.byref(ptr)))
        return ptr.value, edges.size - 1

    def hist_omega_launch(self, edges, kind=HIST_INTRINSIC, alpha=0.0):
        """non-blocking: queue the histogram kernel on the handle's stream -> (device pointer, nbins)"""
        edges = _f64(edges)
        ptr = C.c_void_p()
        self._check(self.lib.swrt_hist_omega_launch(self._h, kind, float(alpha), _ptr(edges), edges.size, C.byref(ptr)))
        return ptr.value, edges.size - 1

    def hist_omega_wait(self):
        self._check(self.lib.swrt_hist_omega_wait(self._h))

    def ideal_omega_hist(self, x, y, kvx, kvy, omega0, edges, alpha=0.0):
        x, y, kvx, kvy, edges = (_f64(a).ravel() for a in (x, y, kvx, kvy, edges))
        counts = np.zeros(edges.size - 1, dtype=np.uint64)
        self._check(self.lib.swrt_ideal_omega_hist(self._h, float(alpha), x.size, _ptr(x), _ptr(y), _ptr(kvx), _ptr(kvy), kvx.size,
                                                   float(omega0), _ptr(edges), edges.size, counts.ctypes.data_as(C.POINTER(C.c_uint64))))
        return counts

    def diag(self, alpha=0.0):
        out = np.empty(8)
        self._check(self.lib.swrt_diag(self._h, float(alpha), _ptr(out)))
        return out

    def omega(self, alpha=0.0, absolute=True):
        om = np.empty(self.n)
        Om = np.empty(self.n) if absolute else None
        self._check(self.lib.swrt_omega(self._h, float(alpha), _ptr(om), _ptr(Om)))
        return om, Om

    def packet_quantity(self, q, alpha=0.0):
        """quantity ``q`` (``Q_XMOD``, ``Q_YMOD``, ``Q_K``, ``Q_L``, ``Q_KMAG``, ``Q_THETA``, ``Q_OMEGA``, ``Q_OMEGA_ABS``) of
        every packet, exactly the values ``hist2`` bins; ``alpha`` is the flow time of the two frequencies"""
        out = np.empty(self.n)
        self._check(self.lib.swrt_packet_quantity(self._h, int(q), float(alpha), _ptr(out)))
        return out

    def hist2(self, qx, xedges, qy, yedges, alpha=0.0, counts=None):
        """MATLAB's ``histcounts2(Qx, Qy, xedges, yedges)`` of two packet quantities on the device (swrt_hist2): a
        ``(nxe-1, nye-1)`` uint64 array, ``N[i, j]`` the packets with ``xedges[i] <= Qx < xedges[i+1]`` and
        ``yedges[j] <= Qy < yedges[j+1]`` (the last bin of each axis closed); NaN or out-of-range packets are not counted.
        ``counts`` (uint64, that shape) is added to and returned."""
        xe, ye = _f64(xedges).ravel(), _f64(yedges).ravel()
        shape = (max(xe.size - 1, 0), max(ye.size - 1, 0))
        acc = counts is not None
        if acc and (not isinstance(counts, np.ndarray) or counts.dtype != np.uint64 or counts.shape != shape):
            raise ValueError(f"hist2: counts must be a uint64 array of shape {shape}")
        buf = np.zeros(shape, dtype=np.uint64, order="F") if not acc else np.asfortranarray(counts)   # C: counts[i + j*(nxe-1)]
        self._check(self.lib.swrt_hist2(self._h, int(qx), _ptr(xe), xe.size, int(qy), _ptr(ye), ye.size, float(alpha),
                                        buf.ctypes.data_as(C.POINTER(C.c_uint64)), int(acc)))
        if acc and buf is not counts:
            counts[...] = buf
            return counts
        return buf

    def weight_scale(self, weights, alpha=0.0):
        """swrt_weight_scale: for each kind in ``weights`` (``W_ACTION``, ``W_ENERGY``, ``W_PSEUDO_K``, ``W_PSEUDO_L``) the least
        E with |w| < 2^E over every finite weight of the ensemble (0 when there is none); int32 array"""
        w = _weight_kinds(weights)
        out = np.zeros(w.size, dtype=np.int32)
        self._check(self.lib.swrt_weight_scale(self._h, _i32p(w), w.size, float(alpha), _i32p(out)))
        return out

    def hist2_sums(self, qx, xedges, qy, yedges, weights, alpha=0.0, scale_exp=None, return_acc=False):
        """per-bin sums of packet weights over ``hist2``'s bins (swrt_hist2_sums): ``(sums, counts)``, sums float64 of shape
        ``(nw, nxe-1, nye-1)`` (``sums[v, i, j]``: kind ``weights[v]`` summed over bin (i, j)), counts as ``hist2``
        returns them.  Each sum is the fixed-point total of the weights scaled by 2^(95-E), rounded once: exactly rounded
        when all weights are within 2^42 of the largest, else fixed-point to 2^(E-95); NaN where a binned packet's weight
        is not finite.  ``scale_exp``: the nw exponents E to use (default: ``weight_scale``'s).  ``return_acc``: also the
        int64 accumulators, shape ``(nw, nxe-1, nye-1, 4)`` (three digit counters and the non-finite count), which
        ``fixed_sums_to_double`` finishes."""
        w = _weight_kinds(weights)
        xe, ye = _f64(xedges).ravel(), _f64(yedges).ravel()
        nbx, nby = max(xe.size - 1, 0), max(ye.size - 1, 0)
        e = None
        if scale_exp is not None:
            e = np.ascontiguousarray(np.atleast_1d(scale_exp), dtype=np.int32)
            if e.shape != (w.size,):
                raise ValueError(f"hist2_sums: scale_exp must hold {w.size} exponents, got {e.shape}")
        sums = np.empty((w.size, nby, nbx))                      # C: sums[(v*nby + j)*nbx + i]
        counts = np.empty((nby, nbx), dtype=np.uint64)
        acc = np.empty((w.size, nby, nbx, 4), dtype=np.int64) if return_acc else None
        self._check(self.lib.swrt_hist2_sums(self._h, int(qx), _ptr(xe), xe.size, int(qy), _ptr(ye), ye.size, float(alpha),
                                             _i32p(w), w.size, _i32p(e), _ptr(sums), counts.ctypes.data_as(C.POINTER(C.c_uint64)),
                                             acc.ctypes.data_as(C.POINTER(C.c_int64)) if return_acc else None))
        out = (sums.transpose(0, 2, 1), counts.T)
        return out + (acc.transpose(0, 2, 1, 3),) if return_acc else out

    # -- instrumentation --
    def launch_count(self, reset=False):
        return int(self.lib.swrt_launch_count(self._h, int(reset)))

    def last_kernel_ms(self):
        n = C.c_int(0)
        ms = self.lib.swrt_last_kernel_ms(self._h, C.byref(n))
        return float(ms), int(n.value)

    def work_per_eval(self, nplanes=6):
        return float(self.lib.swrt_work_per_eval(self._h, nplanes))

    def synchronize(self):
        self._check(self.lib.swrt_synchronize(self._h))

    def set_stream(self, cuda_stream_ptr):
        self._check(self.lib.swrt_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def timer_start(self):
        self._check(self.lib.swrt_timer_start(self._h))

    def timer_stop(self):
        ms = float(self.lib.swrt_timer_stop(self._h))
        if ms < 0:
            raise SwrtError(-3, "timer failed")
        return ms

    def set_tuning(self, mtiles=0, use_psi_moments=True, preblend_grid=False, unfused_rk4=False, twiddles=0):
        """``preblend_grid`` (LAGRANGE6): blend two frames on the grid before the gather (faster) instead of
        interpolating both frames and blending the results as interpolate_U.m does (default, bit-faithful);
        ``unfused_rk4`` (SPECTRAL, NUFFT): step_packet* as evaluation + stage launches instead of the fused kernel;
        ``twiddles`` (SPECTRAL): 0 automatic, 1 rotate in registers, 2 global (L2) table, 3 shared-memory table else global"""
        self._check(self.lib.swrt_set_tuning(self._h, int(mtiles), (0 if use_psi_moments else 1) | (2 if preblend_grid else 0)
                                             | (4 if unfused_rk4 else 0) | ((int(twiddles) & 3) << 3)))

    def contracted_planes(self):
        return int(self.lib.swrt_contracted_planes(self._h))


class QGFlow:
    """On-device one-layer QG solver producing the background-flow frames (qgsw_raytrace.m:111-137,
    :270-286): q-hat lives on the GPU; ``to_flow(engine, slot)`` fills a flow slot without a host copy."""

    def __init__(self, nx, L, qk, K_d2, dt, f, Cg, beta=0.0, r_drag=0.1, force_strength=0.1, device=0):
        self.lib = load_library()
        self.nx, self.L = int(nx), float(L)
        qk = np.asarray(qk, dtype=np.complex128)
        re, im = _colmajor(qk.real), _colmajor(qk.imag)
        self._q = C.c_void_p()
        rc = self.lib.swrt_qg_create(int(device), self.nx, self.L, float(K_d2), float(beta), float(r_drag), float(force_strength),
                                     float(f), float(Cg), float(dt), _ptr(re), _ptr(im), C.byref(self._q))
        if rc != 0:
            raise SwrtError(rc, (self.lib.swrt_last_error(None) or b"").decode())

    def step(self, nsteps=1):
        rc = self.lib.swrt_qg_step(self._q, int(nsteps))
        if rc != 0:
            raise SwrtError(rc, "swrt_qg_step failed")

    def get(self):
        nkx, nky = self.nx - 1, self.nx // 2
        re = np.empty(nkx * nky); im = np.empty(nkx * nky)
        rc = self.lib.swrt_qg_get(self._q, _ptr(re), _ptr(im))
        if rc != 0:
            raise SwrtError(rc, "swrt_qg_get failed")
        return (re + 1j * im).reshape((nkx, nky), order="F")

    def get_grid(self):
        """q = k2g(qk) (nx, nx), transformed on the device with the solver's own FFT plan"""
        out = np.empty(self.nx * self.nx)
        rc = self.lib.swrt_qg_get_grid(self._q, _ptr(out))
        if rc != 0:
            raise SwrtError(rc, "swrt_qg_get_grid failed")
        return out.reshape((self.nx, self.nx), order="F")

    def to_flow(self, engine, slot=0, u_mean=0.0):
        engine._check(self.lib.swrt_set_flow_from_qg(engine._h, int(slot), self._q, float(u_mean)))

    def close(self):
        if getattr(self, "_q", None) and self._q.value:
            self.lib.swrt_qg_destroy(self._q)
            self._q = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class QG2Flow:
    """On-device two-layer QG solver (qg2layersw_raytrace.m:120-181, :309-323): both layer PV spectra, the
    inversion matrix B and expm(factor_L*dt) live on the GPU; ``to_flow`` fills a flow slot with
    ``grid_U(qk(:,:,1), ..., shear_strength)`` of the top layer without a host copy."""

    def __init__(self, nx, L, q1k, q2k, K_d2, beta, shear_strength, r, nu, alpha, device=0):
        self.lib = load_library()
        self.nx, self.L = int(nx), float(L)
        parts = []
        for qk in (q1k, q2k):
            qk = np.asarray(qk, dtype=np.complex128)
            parts += [_colmajor(qk.real), _colmajor(qk.imag)]
        self._q = C.c_void_p()
        rc = self.lib.swrt_qg2_create(int(device), self.nx, self.L, float(K_d2), float(beta), float(shear_strength), float(r),
                                      float(nu), float(alpha), *[_ptr(a) for a in parts], C.byref(self._q))
        if rc != 0:
            raise SwrtError(rc, (self.lib.swrt_last_error(None) or b"").decode())

    def _check(self, rc, what):
        if rc != 0:
            raise SwrtError(rc, f"{what} failed")

    def max_speed(self):
        out = C.c_double(0.0)
        self._check(self.lib.swrt_qg2_max_speed(self._q, C.byref(out)), "swrt_qg2_max_speed")
        return out.value

    def step(self, dt):
        self._check(self.lib.swrt_qg2_step(self._q, float(dt)), "swrt_qg2_step")

    def get(self, layer):
        nkx, nky = self.nx - 1, self.nx // 2
        re = np.empty(nkx * nky); im = np.empty(nkx * nky)
        self._check(self.lib.swrt_qg2_get(self._q, int(layer), _ptr(re), _ptr(im)), "swrt_qg2_get")
        return (re + 1j * im).reshape((nkx, nky), order="F")

    def to_flow(self, engine, slot=0):
        engine._check(self.lib.swrt_set_flow_from_qg2(engine._h, int(slot), self._q))

    def close(self):
        if getattr(self, "_q", None) and self._q.value:
            self.lib.swrt_qg2_destroy(self._q)
            self._q = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# -- handle-free helpers ---------------------------------------------------------------------------

def interpolate_dev(x, y, F, dx, dy, bump=1e-13, device=0):
    lib = load_library()
    x = _f64(x); shp = x.shape
    x = x.ravel(); y = _f64(y).ravel()
    if x.size != y.size:
        raise ValueError(f"interpolate: x has {x.size} elements, y has {y.size}")
    F = np.asarray(F, dtype=np.float64)
    nx, ny = F.shape
    Ff = _colmajor(F)
    out = np.empty(x.size)
    rc = lib.swrt_interpolate(device, _ptr(x), _ptr(y), x.size, _ptr(Ff), nx, ny, float(dx), float(dy), float(bump), _ptr(out))
    if rc != 0:
        raise SwrtError(rc, (lib.swrt_last_error(None) or b"").decode())
    return out.reshape(shp)


def g2k_dev(fg, device=0):
    lib = load_library()
    fg = np.asarray(fg, dtype=np.float64)
    nx = fg.shape[0]
    nkx, nky = nx - 1, nx // 2
    re = np.empty(nkx * nky); im = np.empty(nkx * nky)
    f = _colmajor(fg)
    rc = lib.swrt_g2k(device, _ptr(f), nx, _ptr(re), _ptr(im))
    if rc != 0:
        raise SwrtError(rc, (lib.swrt_last_error(None) or b"").decode())
    return (re + 1j * im).reshape((nkx, nky), order="F")


def k2g_dev(fk, device=0):
    lib = load_library()
    fk = np.asarray(fk, dtype=np.complex128)
    nx = fk.shape[0] + 1
    re, im = _colmajor(fk.real), _colmajor(fk.imag)
    out = np.empty(nx * nx)
    rc = lib.swrt_k2g(device, _ptr(re), _ptr(im), nx, _ptr(out))
    if rc != 0:
        raise SwrtError(rc, (lib.swrt_last_error(None) or b"").decode())
    return out.reshape((nx, nx), order="F")
