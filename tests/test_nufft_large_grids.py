"""NUFFT mode above 64^2, and at the smallest grids, against the C oracle's long-double Fourier sums.

The NUFFT evaluation deconvolves u-hat, v-hat (and H-hat) by 1/phi-hat(k) (nufft_init: up to ~250x at kmax), unfolds the
half plane (the ky = 0 row by conjugation) into an nf = 2 nx spectrum, transforms it with cuFFT and gathers an 18 x 18
stencil of the fine grid with the ES kernel and its analytic derivative.  Each size of NUFFT_SIZES takes a path the others
miss: 8 (nf = 16 < 18: the stencil wraps twice), 10 / 30 / 130 / 258 (nx/2 odd), 96 / 192 / 384 / 1000 (off powers of
two, small primes), 194 / 1018 (nf = 4*97, 4*509: cuFFT's non-radix kernels) and the powers of two.

* evaluation at every size: C3 and C4 flows uploaded as psi-hat, six planes, seven planes (the (u, v, H, 0) grid) and
  grids (device g2k), at seeded, edge, fine-node, next-to-fine-node and coarse-node positions;
* flows that weight every wavenumber alike (white psi-hat with |u-hat|^2 + |v-hat|^2 flat, and single modes up to
  kx = +-kmax, ky = kmax): the ones on which a per-wavenumber error is not diluted by a K^-3 spectrum;
* the leapfrog: one step, 8 two-frame sub-steps, and 40 sub-steps (two fused runs, the second at j0 = 32);
* the fused RK4 steppers (nufft_rk4_kernel) and their composed twin (unfused_rk4), steady and two-frame;
* ode23 at 256^2: coupled, dense output, backward, per packet and per-packet tspans (the MIX blend), and at 512^2;
* gradients 0.03 - 0.045 fine cells from fine nodes, where the kernel's end node is near its singular derivative;
* Omega = omega + U.k on the white flow;
* CPU guards: NUFFT_SIZES reaches every size class, and the sparse long-double reference equals the C oracle."""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
from oracle import c_oracle as CO
from oracle import swrt_oracle as O
import test_spectral_large_grids as L
from test_spectral_large_grids import sample, edge_positions, planes_at, scaled_err, TOL_SUBSTEPS

NUFFT_SIZES = [8, 10, 30, 64, 96, 128, 130, 192, 194, 256, 258, 384, 512, 1000, 1018, 1024]
NUFFT_W = 18                         # ES-kernel width in fine-grid points (swrt_internal.h kNufftW)
TOL_FIELD = 1e-12                    # evaluation: of max|plane|, the README contract
TOL_STEP = 1e-12                     # one leapfrog step: of the increment
TOL_RK4 = 1e-11                      # 2 RK4 steps: of the increment, the bound that holds at 64^2 and 128^2


# ------------------------------------------------------------------------------------------------
# CPU guard: every class of size
# ------------------------------------------------------------------------------------------------
def largest_prime_factor(n):
    p, big = 2, 1
    while n > 1:
        while n % p == 0:
            n //= p
            big = p
        p += 1
    return big


SIZE_CLASSES = {
    "nf = 2 nx < 18: the stencil wraps twice": lambda nx: 2 * nx < NUFFT_W,
    "nx/2 odd": lambda nx: (nx // 2) % 2 == 1,
    "power of two": lambda nx: nx & (nx - 1) == 0,
    "smooth, not a power of two": lambda nx: nx & (nx - 1) != 0 and largest_prime_factor(nx // 2) < 11,
    "nx/2 has a prime factor >= 11": lambda nx: largest_prime_factor(nx // 2) >= 11,
}


def test_nufft_sizes_reach_every_size_class():
    assert all(nx % 2 == 0 and 8 <= nx <= 1024 for nx in NUFFT_SIZES)
    missing = [c for c, member in SIZE_CLASSES.items() if not any(member(nx) for nx in NUFFT_SIZES)]
    assert not missing, f"no size in NUFFT_SIZES for: {missing}"
    # a class with at least two members above 128^2, where the fine grid no longer fits in L1 / shared memory
    for c in ("nx/2 odd", "power of two", "smooth, not a power of two", "nx/2 has a prime factor >= 11"):
        assert sum(SIZE_CLASSES[c](nx) for nx in NUFFT_SIZES if nx > 128) >= 2, c


# ------------------------------------------------------------------------------------------------
# flows that weight every wavenumber, and their long-double reference
# ------------------------------------------------------------------------------------------------
def hermitian_row0(fk):
    """the ky = 0 row made conjugate-symmetric (kx < 0 from kx > 0, a real mean): the half plane the engine sees"""
    kmax = fk.shape[1] - 1
    fk = fk.copy()
    fk[:kmax, 0] = np.conj(fk[:kmax:-1, 0])
    fk[kmax, 0] = fk[kmax, 0].real
    return fk


def flow_workload(nx, psik, psik2, etak, etak2, name, L=2 * np.pi, u_mean=0.0, nrand=40, seed=5):
    """a Workload holding the two frames (psi-hat, eta-hat) and seeded positions; k, l on a ring of |k| = 10"""
    f, Cg = 3.0, 1.0
    dx = L / nx
    xe, ye = edge_positions(L, dx)
    rs = np.random.RandomState(seed)
    x = np.concatenate([rs.uniform(-3 * L, 3 * L, nrand), xe])
    y = np.concatenate([rs.uniform(-3 * L, 3 * L, nrand), ye])
    th = rs.uniform(0, 2 * np.pi, x.size)
    k, l = 10 * np.cos(th), 10 * np.sin(th)
    return W.Workload(name, nx, L, f, Cg, x.size, psik, psik2, u_mean, x, y, k, l, 0.05 * dx / 0.5, 0.5,
                      extra={"etak_frames": (etak, etak2)})


def white_flow(nx, seed=7):
    """psi-hat ~ e^{i theta} / |K|: |u-hat|^2 + |v-hat|^2 is the same at every (kx, ky) up to the truncation, kx = +-kmax,
    ky = kmax and the ky = 0 row included; eta-hat flat with random phases.  Frame 1 turns every phase by up to 0.3."""
    kx, ky = W.wavenumbers(nx)
    K = np.hypot(kx, ky)                              # L = 2 pi: kappa = 1
    K[K == 0] = 1.0
    rs = np.random.RandomState(seed)
    psik = np.exp(2j * np.pi * rs.rand(*kx.shape)) / K
    psik[nx // 2 - 1, 0] = 0.0
    etak = np.exp(2j * np.pi * rs.rand(*kx.shape))
    etak[nx // 2 - 1, 0] = 0.0
    psik2 = psik * np.exp(1j * rs.uniform(-0.3, 0.3, kx.shape))
    etak2 = etak * np.exp(1j * rs.uniform(-0.3, 0.3, kx.shape))
    psik, psik2, etak, etak2 = (hermitian_row0(a) for a in (psik, psik2, etak, etak2))
    pl = W.planes_from_psik(psik, 2 * np.pi)
    U0 = np.hypot(W._fulspec_ifft(pl[0]), W._fulspec_ifft(pl[1])).max()
    E0 = np.abs(W._fulspec_ifft(etak)).max()
    s, t = 0.5 / U0, 0.3 / E0
    return flow_workload(nx, s * psik, s * psik2, t * etak, t * etak2, "white")


def single_modes(nx):
    """(kx, ky) in {0, 1, kmax/2, kmax-1, kmax}^2 with kx of both signs; on the ky = 0 row -kx is the mode kx"""
    kmax = nx // 2 - 1
    ks = sorted({0, 1, kmax // 2, kmax - 1, kmax})
    return [(sx * kx, ky) for ky in ks for kx in ks for sx in ((1, -1) if kx and ky else (1,)) if kx or ky]


def single_mode_flow(nx, kx, ky, seed=3):
    """psi-hat and eta-hat of the one mode (kx, ky), max|u|, max|v| ~ 0.5, |eta| <= 0.3; frame 1 turns the phase by 0.2"""
    kmax = nx // 2 - 1
    rs = np.random.RandomState(seed + 4096 * (kx + nx) + ky)
    c = np.exp(2j * np.pi * rs.rand())
    psik = np.zeros((nx - 1, nx // 2), dtype=np.complex128)
    etak = np.zeros_like(psik)
    psik[kx + kmax, ky] = 0.25 / max(abs(kx), ky) * c
    etak[kx + kmax, ky] = 0.15 * c.conjugate()
    return flow_workload(nx, psik, psik * np.exp(0.2j), etak, etak * np.exp(-0.2j), f"mode({kx},{ky})", nrand=16)


def flow_planes(w, alpha=0.0, seven=False):
    """the coefficient planes of (1 - alpha)*frame 0 + alpha*frame 1: the gradients from O.velocity_planes_k, H = 1 + eta"""
    if "etak_frames" not in w.extra:
        return planes_at(w, alpha, seven)
    e0, e1 = w.extra["etak_frames"]
    psik = w.psik if alpha == 0.0 else (1.0 - alpha) * w.psik + alpha * w.psik2
    kap = 2 * np.pi / w.L
    kx, ky = O.wavenumbers(w.nx)
    pl = O.velocity_planes_k(psik, kap * kx, kap * ky)
    pl[0] = pl[0].copy(); pl[0][w.nx // 2 - 1, 0] += w.u_mean
    if seven:
        Hk = e0 if alpha == 0.0 else (1.0 - alpha) * e0 + alpha * e1
        Hk = Hk.copy(); Hk[w.nx // 2 - 1, 0] += 1.0
        pl.append(Hk)
    return pl


PI_LD = np.longdouble("3.14159265358979323846264338327950288")


def sparse_eval(x, y, planes_k, dx, nx):
    """CO.spectral_eval's long-double sum taken over the nonzero coefficients only (a single-mode flow at 1024^2 costs
    one term instead of half a million): F = sum_kx F(kx,0) e^{i kx tx} (conjugate-symmetrised) + 2 Re sum_{ky>=1} ...,
    tx = 2 pi mod(x/dx, nx) / nx"""
    def red(v):
        r = np.fmod(np.asarray(v, dtype=np.float64) / dx, float(nx))
        return np.where(r < 0.0, r + nx, r).astype(np.longdouble)
    tx = 2 * PI_LD * red(x) / nx
    ty = 2 * PI_LD * red(y) / nx
    kmax = nx // 2 - 1
    out = []
    for p in planes_k:
        acc = np.zeros(tx.shape, dtype=np.longdouble)
        for i, ky in zip(*np.nonzero(p)):
            kx = int(i) - kmax
            re, im = np.longdouble(p[i, ky].real), np.longdouble(p[i, ky].imag)
            if ky == 0 and kx == 0:
                acc += re
            elif ky > 0 or kx > 0:
                a = kx * tx + int(ky) * ty
                acc += 2 * (re * np.cos(a) - im * np.sin(a))
        out.append(acc.astype(np.float64))
    return np.stack(out)


def test_sparse_reference_equals_the_c_oracle():
    """the single-mode reference is CO.spectral_eval: every mode of single_modes at 30^2 and 64^2, and a sparse random
    flow, to 1e-17 of the plane (both sums are long double)"""
    for nx in (30, 64):
        flows = [single_mode_flow(nx, kx, ky) for kx, ky in single_modes(nx)]
        w = white_flow(nx)
        rs = np.random.RandomState(1)
        keep = rs.rand(*w.psik.shape) < 0.05
        w.psik, w.psik2 = (np.where(keep, p, 0.0) for p in (w.psik, w.psik2))
        w.extra["etak_frames"] = tuple(np.where(keep, e, 0.0) for e in w.extra["etak_frames"])
        for f in flows + [w]:
            pl = flow_planes(f, 0.3, seven=True)
            ref = CO.spectral_eval(f.x, f.y, pl, f.dx, nx, precise=True)
            assert scaled_err(sparse_eval(f.x, f.y, pl, f.dx, nx), ref) < 1e-15, f.name


# ------------------------------------------------------------------------------------------------
# engines and positions
# ------------------------------------------------------------------------------------------------
def nufft_engine(w, form, two=False):
    """form: psi (psi-hat upload), planes (six planes), seven (six + H: the (u, v, H, 0) fine grid), grid (seven gridded
    planes through the device g2k)"""
    e = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_NUFFT)
    for slot in (0, 1) if two else (0,):
        al = float(slot)
        if form == "psi":
            e.set_flow_spectral(w.psik if slot == 0 else w.psik2, slot, w.u_mean)
        elif form == "grid":
            e.set_flow_grid(*[O.k2g(p) for p in flow_planes(w, al, seven=True)], slot=slot)
        else:
            e.set_flow_planes_spectral(flow_planes(w, al, seven=form == "seven"), slot)
    return e


def node_positions(L, nx, seed=9):
    """24 positions: fine-grid nodes (i + 1/2) dx, one ulp either side of them, and coarse nodes i dx"""
    dx = L / nx
    rs = np.random.RandomState(seed)
    i, j = rs.randint(-nx, 2 * nx, (2, 8))
    fx, fy = (i + 0.5) * dx, (j + 0.5) * dx
    x = np.concatenate([fx, np.nextafter(fx[:4], np.inf), np.nextafter(fx[4:], -np.inf), i * dx])
    y = np.concatenate([fy, np.nextafter(fy[:4], -np.inf), np.nextafter(fy[4:], np.inf), j * dx])
    return x, y


def eval_positions(w):
    """the workload's positions, plus the node positions from 256^2 on"""
    if w.nx < 256:
        return w.x, w.y
    xn, yn = node_positions(w.L, w.nx)
    return np.concatenate([w.x, xn]), np.concatenate([w.y, yn])


def nufft_eval_errors(w, forms, ref_fn):
    """{form: error of eval_at against ref_fn's planes}; a reversed ensemble must give the same doubles, reversed"""
    x, y = eval_positions(w)
    ref = ref_fn(x, y, flow_planes(w, seven=True), w.dx, w.nx)
    xr, yr = x[::-1].copy(), y[::-1].copy()
    errs = {}
    for form in forms:
        seven = form in ("seven", "grid")
        with nufft_engine(w, form) as e:
            got = e.eval_at(x, y, with_H=seven)
            errs[form] = scaled_err(got, ref[:7 if seven else 6])
            rev = e.eval_at(xr, yr, with_H=seven)
            assert np.array_equal(rev[:, ::-1], got), form
    return errs


# ------------------------------------------------------------------------------------------------
# evaluation at every size
# ------------------------------------------------------------------------------------------------
def workload_sample(name, nx):
    """the workload with 64 seeded and the edge positions in w.x, w.y; 40 from 512^2 on, where the node positions make
    73 long-double points"""
    w, (x, y, _, _) = sample(name, nx, 64 if nx < 512 else 40)
    w.x, w.y = x, y
    return w


def cexact(x, y, planes, dx, nx):
    return CO.spectral_eval(x, y, planes, dx, nx, precise=True)


@pytest.mark.gpu
@pytest.mark.parametrize("nx", NUFFT_SIZES)
@pytest.mark.parametrize("name", ["C3", "C4"])
def test_eval_every_size_and_upload(nx, name):
    w = workload_sample(name, nx)
    errs = nufft_eval_errors(w, ("psi", "planes", "seven", "grid"), cexact)
    bad = {k: v for k, v in errs.items() if not v < TOL_FIELD}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# flows that weight every wavenumber
# ------------------------------------------------------------------------------------------------
FLAT_SIZES = [256, 512, 1018, 1024]


@pytest.mark.gpu
@pytest.mark.parametrize("nx", FLAT_SIZES)
def test_white_flow(nx):
    errs = nufft_eval_errors(white_flow(nx), ("psi", "planes", "seven", "grid"), cexact)
    bad = {k: v for k, v in errs.items() if not v < TOL_FIELD}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("nx", FLAT_SIZES)
def test_single_modes(nx):
    """every mode on its own: psi-hat and seven planes; the error of each plane against its own max"""
    bad = {}
    for kx, ky in single_modes(nx):
        errs = nufft_eval_errors(single_mode_flow(nx, kx, ky), ("psi", "seven"), sparse_eval)
        bad.update({(kx, ky, f): v for f, v in errs.items() if not v < TOL_FIELD})
    assert not bad, bad


@pytest.mark.gpu
def test_gradients_next_to_fine_nodes_carry_no_multiple_of_the_field():
    """Near |z| = 1 phi' is singular, so es_kernel drops a stencil end node while sqrt(1 - z^2) < 1e-3.  A node dropped
    (or mis-weighted) farther in takes phi'(z) g away from the derivative sum, and g there is the field itself for a k = 1
    mode: the error of vx (uy) gains a part proportional to v (u).  At 1024^2, where dscale / kappa = nx / (9 pi) is
    largest, 2000 packets 0.03 and 0.045 fine cells either side of fine nodes: the least-squares multiple of the field in
    the gradient's error, times max|field|, within 1e-13 of max|gradient|.  Measured on a B200: <= 4.1e-14 (the largest
    single error is ~1.7e-13, the bound of the other tests is 1e-12); dropping the nodes with 1 - z^2 < 1e-2 gives 3e-13."""
    nx = 1024
    rs = np.random.RandomState(8)
    i = rs.randint(0, 2 * nx, 2000)
    t = rs.rand(2000) * 2 * nx
    bias = {}
    for kx, ky, field, grad in ((1, 0, 1, 4), (0, 1, 0, 3)):        # (1, 0): v and vx; (0, 1): u and uy
        w = single_mode_flow(nx, kx, ky)
        hf = w.dx / 2
        with nufft_engine(w, "psi") as e:
            for d in (0.045, -0.045, 0.03, -0.03):
                x, y = ((i + d) * hf, t * hf) if kx else (t * hf, (i + d) * hf)
                ref = sparse_eval(x, y, flow_planes(w), w.dx, nx)
                err = e.eval_at(x, y)[grad] - ref[grad]
                c = err @ ref[field] / (ref[field] @ ref[field])
                bias[(kx, ky, d)] = abs(c) * np.abs(ref[field]).max() / np.abs(ref[grad]).max()
    assert max(bias.values()) < 1e-13, bias


@pytest.mark.gpu
def test_omega_absolute_on_the_white_flow():
    """Omega = omega + u k + v l (swrt_omega) at 512^2 against the exact-sum U, to 1e-12 of max|U.k|"""
    w = white_flow(512)
    with nufft_engine(w, "psi") as e:
        e.set_packets(w.x, w.y, w.k, w.l)
        om, Om = e.omega()
    u, v = CO.spectral_eval(w.x, w.y, flow_planes(w)[:2], w.dx, w.nx, precise=True)
    Uk = u * w.k + v * w.l
    assert np.array_equal(om, np.sqrt(w.f ** 2 + w.gH * (w.k * w.k + w.l * w.l)))
    assert np.abs(Om - (om + Uk)).max() < TOL_FIELD * np.abs(Uk).max()


# ------------------------------------------------------------------------------------------------
# the leapfrog (nufft_leapfrog_kernel on the axpby_multi arena of fine grids)
# ------------------------------------------------------------------------------------------------
LEAPFROG_SIZES = [8, 10, 130, 194, 256, 512, 1024]


@pytest.mark.gpu
@pytest.mark.parametrize("nx", LEAPFROG_SIZES)
@pytest.mark.parametrize("name", ["C3", "C4"])
def test_leapfrog_against_the_exact_sum(nx, name):
    e1, em = L.leapfrog_errors(nx, name, "psi", make=nufft_engine)
    assert e1 < TOL_STEP and em < TOL_SUBSTEPS, (e1, em)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["C3", "C4"])
def test_leapfrog_40_substeps_cross_the_fused_blend_limit(name):
    """40 two-frame sub-steps are two fused runs (32 + 8 pre-blended grids); the second blends from j0 = 32"""
    _, em = L.leapfrog_errors(130, name, "psi", m=40, make=nufft_engine)
    assert em < TOL_SUBSTEPS, em


# ------------------------------------------------------------------------------------------------
# the fused RK4 steppers (nufft_rk4_kernel) and the composed launches
# ------------------------------------------------------------------------------------------------
RK4_SIZES = [64, 128, 130, 194, 256, 512]            # 64 and 128 calibrate TOL_RK4
RK4_CASES = [("rk4_packet", "psi"), ("rk4_packet", "planes"), ("rk4_packet", "two-frame"), ("rk4_xka", "planes"),
             ("rk4_xka", "two-frame")]


@pytest.mark.gpu
@pytest.mark.parametrize("nx", RK4_SIZES)
@pytest.mark.parametrize("scheme,flow", RK4_CASES)
@pytest.mark.parametrize("unfused", [False, True])
def test_rk4_against_the_exact_sum(nx, scheme, flow, unfused):
    err = L.rk4_error(nx, scheme, flow, make=nufft_engine, unfused=unfused)
    assert err < TOL_RK4, err


# ------------------------------------------------------------------------------------------------
# ode23: nufft_eval_dev_kernel (the controller's frame) and nufft_eval_pkt_kernel (per-packet alphas, MIX)
# ------------------------------------------------------------------------------------------------
def ode23_sample(nx):
    """sample's C3 packets (8 seeded and the edge positions) without the two at 1e6, so that every other packet is 8
    packets.  The backward solve's step-size controller turns an evaluation error of 1e-13 (the exact sums perturbed by
    that much, on the oracle alone) into steps that differ in the 9th digit, and a packet at 1e6, where one ulp is 3e-10
    of its increment, then lands a few ulps away: 1.4e-9 of the increment on the oracle, 1.35e-9 in NUFFT mode"""
    w, pk = sample("C3", nx, 8)
    pk = np.stack(pk)
    return w, pk[:, np.abs(pk[:2]).max(axis=0) < 1e3]


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["psi", "planes"])
@pytest.mark.parametrize("two", [False, True])
def test_ode23_256(form, two):
    errs = L.ode23_errors(256, form, two, make=nufft_engine, packets=ode23_sample, tspans=True)
    assert max(errs.values()) < TOL_SUBSTEPS, errs


@pytest.mark.gpu
def test_ode23_512_steady():
    err = L.ode23_steady_error(512, make=nufft_engine, packets=ode23_sample)
    assert err < TOL_SUBSTEPS, err
