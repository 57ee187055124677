"""Extended-precision references of the QG frame producers (swrt_qg.inc), for test_qg_producers_large.py.

The float64 oracle (oracle.swrt_oracle: qg_run, qg2_operators / qg2_expL, g2k / k2g) restates the reference's
arithmetic; its own rounding (~1e-13 for the eig-based two-layer exponential) is too close to the device's to tell
a subtly wrong kernel from noise.  The helpers here compute the same operations in ``np.longdouble`` /
``np.clongdouble`` (64-bit significand on x86-64), from the same float64 inputs the device receives -- the wave
numbers ``(2 pi / L) * integer`` rounded to double, as the kernels form them -- so that what remains in a comparison
is the device's own rounding:

* ``qg2_factor_ld``: factor_L of qg2layersw_raytrace.m:136-146, (2, 2, nkx, nky);
* ``expm2_ld``: page-wise exp(t M) by scaling and squaring plus Taylor (``expm2_mp`` is the mpmath check of it);
* ``qg_linear_ld``: the one-layer Euler / AB2 / AB3 recurrence with the filter, restricted to its linear part
  Qn = -beta i kx psi-hat (the whole recurrence when the Jacobian underflows to zero);
* ``g2k_ld`` / ``k2g_ld``: g2k.m / k2g.m as matrix DFTs with long-double twiddles."""
import numpy as np

from oracle import swrt_oracle as O

LD, CLD = np.longdouble, np.clongdouble
PI_LD = np.arccos(LD(-1))
EXTENDED = np.finfo(LD).eps < 1e-18                   # False where long double is only double (then the tests skip)


def wavenumbers(nx, L):
    """(kx, ky) as float64 (nkx, nky) arrays, rounded exactly as the kernels form them: (2.0*M_PI/L) * integer"""
    kx_, ky_ = O.wavenumbers(nx)
    kap = 2.0 * np.pi / L
    return kx_ * kap, ky_ * kap


# ------------------------------------------------------------------------------------------------
# two layers: factor_L and its exponential
# ------------------------------------------------------------------------------------------------
def qg2_factor_ld(kx, ky, K_d2, beta, shear, r, nu, alpha):
    """factor_L = shear_factor .* M + B .* diffusion_factor (qg2layersw_raytrace.m:136-146) in clongdouble"""
    kx, ky = kx.astype(LD), ky.astype(LD)
    K2 = kx * kx + ky * ky
    F = LD(K_d2) / 2
    det = K2 * (K2 + 2 * F)
    zero = K2 == 0
    det[zero] = 1
    B11 = np.where(zero, LD(0), (-F - K2) / det)
    B12 = np.where(zero, LD(0), -F / det)
    dfac = (LD(nu) * K2 ** LD(alpha) + LD(r)) * K2 - 1j * kx * LD(beta)
    sh = 1j * kx * LD(shear)
    m11, m12 = -(1 + 2 * F * B11), -2 * F * B12
    M = np.empty((2, 2) + kx.shape, dtype=CLD)
    M[0, 0] = sh * m11 + dfac * B11
    M[0, 1] = sh * m12 + dfac * B12
    M[1, 0] = sh * (-m12) + dfac * B12
    M[1, 1] = sh * (-m11) + dfac * B11
    return M


def _mul2(A, B):
    return np.stack([np.stack([A[0, 0] * B[0, 0] + A[0, 1] * B[1, 0], A[0, 0] * B[0, 1] + A[0, 1] * B[1, 1]]),
                     np.stack([A[1, 0] * B[0, 0] + A[1, 1] * B[1, 0], A[1, 0] * B[0, 1] + A[1, 1] * B[1, 1]])])


def _split(x, bits):
    """Veltkamp: x = hi + lo with hi holding the leading 64 - ``bits`` bits of the long-double significand"""
    c = x * LD(2.0 ** bits + 1)
    hi = c - (c - x)
    return hi, x - hi


def _exp_real_times(x, t):
    """exp(x t) for long-double x and float64 t, with x t formed without rounding (two-product): at the top modes of
    512^2 |x t| reaches ~700, where the rounding of the product alone would move the result by 4e-17"""
    t = LD(t)
    hi = x * t
    x1, x2 = _split(x, 32)
    t1, t2 = _split(t, 38)                          # t: 53 bits -> 26 + 27
    lo = (((x1 * t1 - hi) + x1 * t2) + x2 * t1) + x2 * t2
    return np.exp(hi) * (1 + lo)


def expm2_ld(M, t):
    """exp(t M) of every 2x2 page of M (2, 2, ...) as exp(t s) exp(t N), s = trace/2, N = [p b; c -p],
    p = (M11 - M22)/2.  exp(t N) by scaling to A = t N / 2^k with |A|_1 <= 1/4, 18 Taylor terms (the remainder is
    below 1e-21 of the sum) and k squarings.  Shifting out the trace keeps k small for the hyperviscous modes, whose
    exponentials decay like exp(-949 t) at 512^2: their squarings would otherwise multiply the rounding of exp(A) by
    2^k."""
    M = np.asarray(M, dtype=CLD)
    s, p = (M[0, 0] + M[1, 1]) / 2, (M[0, 0] - M[1, 1]) / 2
    A = np.stack([np.stack([p, M[0, 1]]), np.stack([M[1, 0], -p])]) * LD(t)
    nrm = np.abs(A).sum(axis=0).max(axis=0).astype(np.float64)
    k = np.maximum(0, np.ceil(np.log2(np.maximum(nrm, 1e-300) / 0.25))).astype(np.int64)
    A = A / np.ldexp(LD(1), k)
    E = np.zeros_like(A)
    E[0, 0] = 1; E[1, 1] = 1
    T = E.copy()
    for j in range(1, 19):
        T = _mul2(T, A) / LD(j)
        E = E + T
    for r in range(int(k.max(initial=0))):
        E = np.where(k > r, _mul2(E, E), E)
    return _exp_real_times(s.real, t) * np.exp(1j * (s.imag * LD(t))) * E


def discriminant(M):
    """D of expm2 (swrt_qg.inc): D^2 = ((a - d)/2)^2 + b c, page-wise; exp(t M) switches branch at |t D| = 1e-4"""
    p = (M[0, 0] - M[1, 1]) / 2
    return np.sqrt((p * p + M[0, 1] * M[1, 0]).astype(np.complex128))


def _mpc(z):
    """clongdouble -> mpmath mpc, exactly (also below the float64 range): significand as an integer times 2^e"""
    import mpmath
    parts = []
    for x in (LD(z.real), LD(z.imag)):
        m, e = np.frexp(x)
        parts.append(mpmath.ldexp(mpmath.mpf(int(np.ldexp(m, 64))), int(e) - 64))
    return mpmath.mpc(*parts)


def expm2_mp(M2, t, dps=40):
    """exp(t M2) of one 2x2 clongdouble page with mpmath.expm at ``dps`` digits; returns a 2x2 list of mpc"""
    import mpmath
    with mpmath.workdps(dps):
        A = mpmath.matrix([[_mpc(M2[i, j]) for j in range(2)] for i in range(2)]) * mpmath.mpf(float(t))
        E = mpmath.expm(A)
        return [[E[i, j] for j in range(2)] for i in range(2)]


def expm2_mp_error(E_ld, M2, t, dps=40):
    """max |E_ld - exp(t M2)| / max |exp(t M2)| over one page, evaluated in mpmath"""
    import mpmath
    with mpmath.workdps(dps):
        ref = expm2_mp(M2, t, dps)
        diff = max(abs(_mpc(E_ld[i, j]) - ref[i][j]) for i in range(2) for j in range(2))
        scale = max(abs(ref[i][j]) for i in range(2) for j in range(2))
        return float(diff / scale)


def apply2(E, q):
    """mmult3: (E q)_i = E[i, 0] q[0] + E[i, 1] q[1] for q (2, nkx, nky)"""
    return np.stack([E[0, 0] * q[0] + E[0, 1] * q[1], E[1, 0] * q[0] + E[1, 1] * q[1]])


# ------------------------------------------------------------------------------------------------
# one layer: filter and the linear AB3 recurrence
# ------------------------------------------------------------------------------------------------
def qg_filter_ld(kx, ky, dx):
    """Ef of qgsw_raytrace.m:222-230: exp(log(1e-15)/(pi/4)^4 (kstar - 3 pi/4)^4) for kstar >= 3 pi/4"""
    kxd, kyd = kx.astype(LD) * LD(dx), ky.astype(LD) * LD(dx)
    kstar = np.sqrt(kxd * kxd + kyd * kyd)
    kc = LD(3) * PI_LD / 4
    cst = np.log(LD("1e-15")) / (PI_LD / 4) ** 4
    return np.where(kstar >= kc, np.exp(cst * (kstar - kc) ** 4), LD(1))


def qg_linear_ld(q0, nsteps, dt, nx, L, K_d2, beta):
    """q-hat after ``nsteps`` steps of qgsw_raytrace.m:111-137 with Qn = -beta i kx psi-hat, psi-hat = -q/(K_d2 + K2)
    (update() without the Jacobian, r_drag = 0, no forcing): Euler, AB2, then AB3, the filter after every step"""
    kx, ky = wavenumbers(nx, L)
    Ef = qg_filter_ld(kx, ky, L / nx)
    kx, ky = kx.astype(LD), ky.astype(LD)
    den = LD(K_d2) + (kx * kx + ky * ky)
    q = np.asarray(q0).astype(CLD)
    dt = LD(dt)
    Qm1 = Qm2 = np.zeros_like(q)
    for step in range(1, nsteps + 1):
        Qn = -LD(beta) * (1j * kx * (-q / den))
        if step == 1:
            dq = dt * Qn
        elif step == 2:
            dq = dt / 2 * (3 * Qn - Qm1)
        else:
            dq = dt / 12 * (23 * Qn - 16 * Qm1 + 5 * Qm2)
        Qm2, Qm1 = Qm1, Qn
        q = Ef * (q + dq)
    return q


# ------------------------------------------------------------------------------------------------
# g2k / k2g as long-double matrix DFTs
# ------------------------------------------------------------------------------------------------
def _twiddles(nx, freqs, sign):
    """cos and sign*sin of 2 pi f x / nx for f in ``freqs`` (rows) and x = 0..nx-1 (columns); the phase index is
    reduced mod nx in integers, so every entry is one correctly rounded long-double value of a table"""
    m = np.arange(nx, dtype=LD)
    c, s = np.cos(2 * PI_LD * m / nx), np.sin(2 * PI_LD * m / nx)
    idx = np.outer(np.asarray(freqs, dtype=np.int64), np.arange(nx, dtype=np.int64)) % nx
    return c[idx], sign * s[idx]


def g2k_ld(fg):
    """g2k.m: fftshift(fft2(fg))/nx^2 at kx = -kmax..kmax, ky = 0..kmax, as a long-double DFT"""
    fg = np.asarray(fg).astype(LD)
    nx = fg.shape[0]
    kmax = nx // 2 - 1
    cx, sx = _twiddles(nx, np.arange(-kmax, kmax + 1), -1)      # e^{-i theta} = c + i s with s = -sin
    cy, sy = _twiddles(nx, np.arange(0, kmax + 1), -1)
    gr, gi = fg @ cy.T, fg @ sy.T                                # (nx, nky)
    fr = cx @ gr - sx @ gi
    fi = cx @ gi + sx @ gr
    return (fr + 1j * fi) / LD(nx * nx)


def fulspec_ld(fk):
    """fulspec.m (oracle.swrt_oracle.fulspec) without the cast to complex128"""
    nkx, nky = fk.shape
    nx, kmax = nkx + 1, nky - 1
    fkf = np.zeros((nx, nx), dtype=CLD)
    fup = np.asarray(fk).astype(CLD).copy()
    fup[kmax - 1::-1, 0] = np.conj(fup[kmax + 1:nkx, 0])
    fdn = np.conj(fup[::-1, nky - 1:0:-1])
    fkf[1:nx, nky:nx] = fup
    fkf[1:nx, 1:nky] = fdn
    return fkf


def k2g_ld(fk):
    """k2g.m: nx^2 ifft2(ifftshift(fulspec(fk))) as a long-double DFT.  fulspec's spectrum is Hermitian with a zero
    Nyquist row and column, so the sum is its ky >= 0 half, ky = 0 once and ky > 0 twice, real part"""
    fkf = fulspec_ld(fk)
    nx = fkf.shape[0]
    half = fkf[1:, nx // 2:]                                      # kx = -kmax..kmax, ky = 0..kmax
    half = half * np.where(np.arange(half.shape[1]) == 0, LD(1), LD(2))
    kmax = nx // 2 - 1
    cx, sx = _twiddles(nx, np.arange(-kmax, kmax + 1), 1)         # (freq, x): e^{+i theta}
    cy, sy = _twiddles(nx, np.arange(0, kmax + 1), 1)
    fr, fi = half.real.astype(LD), half.imag.astype(LD)
    pr = cx.T @ fr - sx.T @ fi                                    # (x, ky)
    pi = cx.T @ fi + sx.T @ fr
    return pr @ cy - pi @ sy


def qg_update_ld(qk, nx, L, K_d2, beta, r_drag, forces):
    """update() of qgsw_raytrace.m:270-286 (oracle.swrt_oracle.qg_update) in long double, the FFTs replaced by
    g2k_ld / k2g_ld; ``forces`` is the float64 inertial-ring forcing"""
    kx, ky = wavenumbers(nx, L)
    kx, ky = kx.astype(LD), ky.astype(LD)
    K2 = kx * kx + ky * ky
    qk = np.asarray(qk).astype(CLD)
    psik = -qk / (LD(K_d2) + K2)
    psikx, psiky = 1j * kx * psik, 1j * ky * psik
    J = k2g_ld(psikx) * k2g_ld(1j * ky * qk) - k2g_ld(psiky) * k2g_ld(1j * kx * qk)
    return g2k_ld(J) - LD(beta) * psikx + LD(r_drag) * K2 + np.asarray(forces).astype(LD)
