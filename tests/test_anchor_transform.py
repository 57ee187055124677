"""K1 of the anchored leapfrog (anchor_transform_kernel, DESIGN.md section 3e): the expansion blocks of every anchor cell by
a pre-twiddle and an M-point Stockham FFT per pre-twiddle phase s, instead of a dense contraction per cell.

CPU: a numpy mirror of the kernel's arithmetic -- the S/D unfold, sincospi pre-twiddles and twiddle table, the radix-8
(radix-4 last at M = 256) butterflies in the kernel's order, 1/r! and i^r at the output -- must be as accurate as the direct
double sum against an extended-precision reference (the bar of test_anchored_expansion.py), and the mirror's stack
reads and block writes, index for index as the kernel forms them, must give the contraction K2 expects.

GPU: one packet per anchor cell with k = l = 0 (keyed where it is placed), so every output cell of the transform is used,
against the dense six-plane kernel: one step, and 16 two-frame sub-steps.
"""
from math import factorial, pi

import numpy as np
import pytest

R = 8
S_PHASES = 64          # N / M


def _cells(nx):
    return {256: 14, 512: 15}[nx]


def _dft4(v0, v1, v2, v3):
    t0, t1, t2, t3 = v0 + v2, v0 - v2, v1 + v3, 1j * (v1 - v3)
    return t0 + t2, t1 + t3, t0 - t2, t1 - t3


def _dft(v):
    if len(v) == 4:
        return list(_dft4(*v))
    h = 0.70710678118654752440
    e0, e1, e2, e3 = _dft4(v[0], v[2], v[4], v[6])
    o0, o1, o2, o3 = _dft4(v[1], v[3], v[5], v[7])
    o1 = ((o1.real - o1.imag) * h) + 1j * ((o1.real + o1.imag) * h)
    o2 = 1j * o2
    o3 = ((-o3.real - o3.imag) * h) + 1j * ((o3.real - o3.imag) * h)
    return [e0 + o0, e1 + o1, e2 + o2, e3 + o3, e0 - o0, e1 - o1, e2 - o2, e3 - o3]


def _radices(M):
    return [8, 8, 8] if M == 512 else [8, 8, 4]


def _twiddles(M):
    m = np.arange(M)
    return np.cos(pi * (m * (2.0 / M))) + 1j * np.sin(pi * (m * (2.0 / M)))


def _fft_pos(y):
    """Stockham FFT along the last axis with the positive exponent, the kernel's passes and twiddles"""
    M = y.shape[-1]
    tw = _twiddles(M)
    L = 1
    for Rx in _radices(M):
        bpt = M // Rx
        b = np.arange(bpt)
        v = []
        for i in range(Rx):
            vi = y[..., b + i * bpt]
            if L > 1 and i > 0:
                vi = vi * tw[(i * (b % L)) * (M // (L * Rx))]
            v.append(vi)
        v = _dft(v)
        out = np.empty_like(y)
        q0 = (b // L) * L * Rx + b % L
        for m in range(Rx):
            out[..., q0 + m * L] = v[m]
        y = out
        L *= Rx
    return y


def _unfold(S, D, M):
    """residues mod M of C(kx): C(+kx) = (S + D)/2, C(-kx) = (S - D)/2, C(0) = S; S, D of shape (..., kmax + 1)"""
    x = np.zeros(S.shape[:-1] + (M,), complex)
    x[..., 0] = S[..., 0]
    x[..., 1:M // 2] = 0.5 * (S[..., 1:] + D[..., 1:])
    x[..., M - 1:M // 2:-1] = 0.5 * (S[..., 1:] - D[..., 1:])
    return x


def _hprime(S, D, nx, r, s):
    """H'_r at the cells 64 q + s, q = 0..M-1 (last axis), for columns S, D (..., kmax + 1)"""
    M = nx
    N = S_PHASES * M
    kmax = nx // 2 - 1
    k = np.arange(M)
    kx = np.where(k < M // 2, k, k - M)
    w = kx / float(kmax)
    wr = np.ones(M)
    for _ in range(r):
        wr = wr * w
    arg = (kx * (2 * s + 1)) * (1.0 / N)
    pre = np.cos(pi * arg) + 1j * np.sin(pi * arg)
    y = _unfold(S, D, M) * pre
    y = wr * y.real + 1j * (wr * y.imag)
    X = _fft_pos(y)
    X = X.real / factorial(r) + 1j * (X.imag / factorial(r))
    return (1j) ** r * X


@pytest.mark.parametrize("nx", [256, 512])
def test_transform_route_is_as_accurate_as_the_direct_sum(nx):
    rs = np.random.default_rng(1)
    kmax, ncol = nx // 2 - 1, 6
    kx = np.arange(0, kmax + 1)
    amp = 1.0 / np.maximum(kx, 1.0) ** 2
    Cp = amp * (rs.standard_normal((ncol, kmax + 1)) + 1j * rs.standard_normal((ncol, kmax + 1)))
    Cm = amp * (rs.standard_normal((ncol, kmax + 1)) + 1j * rs.standard_normal((ncol, kmax + 1)))
    Cm[:, 0] = 0.0
    S, D = Cp + Cm, Cp - Cm
    m = _cells(nx)
    h2 = 2.0 ** (1 - m)
    ts = rs.uniform(0.0, 2.0, 300)
    ts = np.concatenate([ts, [0.0, 2.0 - h2 / 3, h2 * 0.999]])
    cells = np.floor(ts / h2).astype(int)
    scale = (np.abs(Cp) + np.abs(Cm)).sum(1)
    Cp_l, Cm_l, kx_l = Cp.astype(np.clongdouble), Cm.astype(np.clongdouble), kx.astype(np.longdouble)
    H = {}
    for s in sorted(set(cells % S_PHASES)):
        H[s] = np.stack([_hprime(S, D, nx, r, s) for r in range(R)])       # (R, ncol, M)
    worst_a = worst_d = 0.0
    for t, c in zip(ts, cells):
        q, s = divmod(c, S_PHASES)
        ta = (c + 0.5) * h2
        z = pi * kmax * (t - ta)
        G = sum(z ** r * H[s][r, :, q] for r in range(R))
        tl = np.longdouble(t) * np.pi
        ref = (Cp_l * np.exp(1j * kx_l * tl) + Cm_l * np.exp(-1j * kx_l * tl)).sum(1)
        direct = (Cp * np.exp(1j * kx * np.pi * t) + Cm * np.exp(-1j * kx * np.pi * t)).sum(1)
        worst_a = max(worst_a, float((np.abs(G - ref) / scale).max()))
        worst_d = max(worst_d, float((np.abs(direct - ref) / scale).max()))
    assert worst_a < 2e-15 + 2 * worst_d, (worst_a, worst_d)


def _pack_stack(C, nx, ksteps):
    """the psi-hat stack layout [pass][kstep][tp][lane][which] (pack_kernel) from C[plane][ky][kx + kmax], weights
    included; the ky = 0 symmetrisation is not needed for a layout check"""
    kmax, G, NT = nx // 2 - 1, 8, 24
    npass = (nx // 2 + 4 * G - 1) // (4 * G)
    st = np.zeros((npass, ksteps, NT // 2, 32, 2))
    for lane in range(32):
        krow, ncol = lane & 3, lane >> 2
        part_k, j, part_n = krow & 1, ncol >> 1, ncol & 1
        for which in range(2):
            for tp in range(NT // 2):
                t = 2 * tp + which
                c, gg = t // G, t % G
                for p in range(npass):
                    ky = p * 4 * G + 4 * gg + j
                    sk = np.arange(ksteps)
                    kxs = 2 * sk + (krow >> 1)
                    ok = (kxs <= kmax) & (ky <= kmax)
                    if not ok.any() or ky > kmax:
                        continue
                    kxv = kxs[ok]
                    cp = C[c, ky, kxv + kmax]
                    cm = np.where(kxv == 0, 0.0, C[c, ky, -kxv + kmax])
                    Sv = np.where(kxv == 0, cp, cp + cm)
                    Dv = np.where(kxv == 0, 0.0, cp - cm)
                    w = 1.0 if ky == 0 else 2.0
                    v = (Sv.real if part_n == 0 else Sv.imag) if part_k == 0 else (-Dv.imag if part_n == 0 else Dv.real)
                    st[p, sk[ok], tp, lane, which] = w * v
    return st


@pytest.mark.parametrize("nx", [256, 512])
def test_kernel_indexing_gives_the_blocks_k2_reads(nx):
    """the kernel's reads of the stack and writes of the blocks, mirrored index for index, against the definition
    H'_r(c)[pass][ks][tp][lane = (2 j + part) * 4 + r % 4][which] = i^r / r! sum_kx (kx/kmax)^r w_ky C(kx, ky) e^{i pi kx t_c}"""
    rs = np.random.default_rng(3)
    kmax, M = nx // 2 - 1, nx
    ksteps = (kmax + 2) // 2
    C = rs.standard_normal((3, nx // 2, 2 * kmax + 1)) + 1j * rs.standard_normal((3, nx // 2, 2 * kmax + 1))
    st = _pack_stack(C, nx, ksteps)
    N = S_PHASES * M
    cells = np.array([0, 1, 63, 64, 12345 % N, N // 2 + 7, N - 1])
    for (p, tp, j) in [(0, 0, 0), (1, 5, 2), (3, 11, 3)]:
        # the kernel's reads: v[part_k][part_n] at lane 2 (kx & 1) + part_k + 4 (2 j + part_n)
        kxa = np.arange(kmax + 1)
        src = st[p, kxa >> 1, tp]                                   # (kmax + 1, 32, 2)
        l0 = 2 * (kxa & 1) + 8 * j
        v00, v01 = src[kxa, l0], src[kxa, l0 + 4]
        v10, v11 = src[kxa, l0 + 1], src[kxa, l0 + 5]
        Sv = (v00 + 1j * v01).T                                     # (which, kx)
        Dv = (v11 - 1j * v10).T
        for ks in range(2):
            lines = np.zeros((M, 16))                               # line of cell 64 q + s, for one s at a time
            for s in sorted(set(cells % S_PHASES)):
                for krow in range(4):
                    r = 4 * ks + krow
                    Hp = _hprime(Sv, Dv, nx, r, s)                  # (which, M)
                    for which in range(2):
                        lines[:, krow * 2 + which] = Hp[which].real
                        lines[:, 8 + krow * 2 + which] = Hp[which].imag
                for c in cells[cells % S_PHASES == s]:
                    q = c // S_PHASES
                    t_c = (2 * c + 1) / N
                    for which in range(2):
                        tt = 2 * tp + which
                        pl, gg = tt // 8, tt % 8
                        ky = p * 32 + 4 * gg + j
                        if ky > kmax:
                            continue
                        wky = 1.0 if ky == 0 else 2.0
                        kxs = np.arange(-kmax, kmax + 1)
                        for krow in range(4):
                            r = 4 * ks + krow
                            ht = (wky * (kxs / kmax) ** r * C[pl, ky, kxs + kmax] * np.exp(1j * pi * kxs * t_c)).sum()
                            want = (1j) ** r / factorial(r) * ht
                            got = lines[q, krow * 2 + which] + 1j * lines[q, 8 + krow * 2 + which]
                            tol = 1e-12 * wky * np.abs(C[pl, ky]).sum()
                            assert abs(got - want) < tol, (nx, p, tp, j, ks, c, which, r, got, want)


def _one_per_cell(w, nx, rs):
    m = _cells(nx)
    N = 2 ** m
    u = rs.uniform(0.0, 1.0, N)
    x = (np.arange(N) + u) * 2.0 ** -m * w.L
    x = np.concatenate([x, [0.0, np.nextafter(2.0 ** -m * w.L, 0.0), (N - 1) * 2.0 ** -m * w.L, np.nextafter(w.L, 0.0)]])
    y = rs.uniform(-w.L / 2, w.L / 2, x.size)
    return x, y, np.zeros_like(x), np.zeros_like(x)


def _rel_increment_err(got, ref, start):
    d_got = np.stack(got) - np.stack(start)
    d_ref = np.stack(ref) - np.stack(start)
    scale = np.abs(d_ref).max(axis=1, keepdims=True)
    scale[scale == 0] = 1.0
    return float((np.abs(d_got - d_ref) / scale).max())


def _stepped(w, x, y, k, l, psi, m, a0=0.0, da=0.0, dt=None):
    import swraytracing_b200 as S
    eng = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL, device=0)
    eng.set_flow_spectral(w.psik, slot=0, u_mean=w.u_mean)
    if da != 0.0:
        eng.set_flow_spectral(w.psik2, slot=1, u_mean=w.u_mean)
    eng.set_tuning(use_psi_moments=psi)
    eng.set_packets(x, y, k, l)
    eng.step(S.SCHEME_LEAPFROG, dt if dt is not None else w.dt, m, a0, da)
    out = eng.get_packets()
    eng.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [256, 512])
def test_every_anchor_cell_one_step_against_the_dense_kernel(nx):
    from swraytracing_b200 import workloads as W
    w = W.make_workload("C4", n_packets=16, nx=nx)
    x, y, k, l = _one_per_cell(w, nx, np.random.default_rng(11))
    got = _stepped(w, x, y, k, l, True, 1)
    ref = _stepped(w, x, y, k, l, False, 1)
    err = _rel_increment_err(got, ref, (x, y, k, l))
    assert err < 1e-12, f"anchored vs dense, one packet per anchor cell: {err:.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [256, 512])
def test_every_anchor_cell_two_frame_substeps_against_the_dense_kernel(nx):
    from swraytracing_b200 import workloads as W
    w = W.make_workload("C4", n_packets=16, nx=nx)
    x, y, k, l = _one_per_cell(w, nx, np.random.default_rng(12))
    m = 16
    got = _stepped(w, x, y, k, l, True, m, 0.5 / m, 1.0 / m, w.dt / m)
    ref = _stepped(w, x, y, k, l, False, m, 0.5 / m, 1.0 / m, w.dt / m)
    err = _rel_increment_err(got, ref, (x, y, k, l))
    assert err < 1e-9, f"16 anchored two-frame sub-steps vs dense, one packet per anchor cell: {err:.3e}"
