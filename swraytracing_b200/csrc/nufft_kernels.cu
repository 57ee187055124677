// nufft_kernels.cu -- NUFFT mode of libswrt: the SAME exact Fourier-series semantics as SPECTRAL mode
// (F(x,y) = sum over the half-plane spectrum, SURVEY.md 7.0), evaluated as a type-2 non-uniform FFT instead of a
// dense sum:
//   setup (per flow frame, untimed):  u-hat, v-hat  ->  divide by the kernel's Fourier transform (deconvolution)
//       ->  zero-pad to an oversampled nf = 2 nx grid  ->  cuFFT inverse  ->  fine grids u_f, v_f (interleaved);
//   per evaluation:  F(x,y) = sum_{a,b=0..15} phi(z_a(x)) phi(z_b(y)) g[i0+a, j0+b],  an 18 x 18 gather with the
//       "exponential of semicircle" kernel phi(z) = exp(beta (sqrt(1 - z^2) - 1)), beta = 2.30 w, w = 18
//       (Barnett, Magland & af Klinteberg, SIAM J. Sci. Comput. 41, 2019); the four velocity gradients come from the
//       ANALYTIC derivative phi'(z) applied to the same u_f, v_f nodes, i.e. they are the spectral derivatives
//       i kx u-hat, ... of SpectralScheme.m:20-23 / grid_U.m:6-9.
// Accuracy (tests/test_gpu_parity.py): <= 1e-12 of max|plane| against the exact trigonometric sum (CPU checker) on all six planes
// (measured 1e-14 for u,v and 2e-13 for the gradients).  Work per evaluation is 324 nodes x 16 bytes, independent of
// nx, against 6 nx^2 flops for the dense contraction: the crossover is below nx = 64.  An optional H plane
// (step_packet_xka, cg_sw.m) rides on a second fine grid of 32-byte nodes (u, v, H, 0) gathered with the same weights:
// one 256-bit load per node, a quad's four loads are one aligned-or-straddling 128-byte segment.
// Replaces: SpectralScheme.U / grad_U (SpectralScheme.m:45-68), interpolate_U.m:5-23, ode_symplectic.m:13-37.
#include "swrt_internal.h"

namespace swrt {

namespace {

constexpr int W = kNufftW;          // kernel width in fine-grid points
constexpr double HALF_W = W / 2.0;
constexpr int kBlock = 128;         // four lanes per packet: 32 packets per block

__device__ __forceinline__ double reduced_coord(double x, double dx, double nxd) {
    // xl = mod(x/dx, nx), the reduced coordinate of interpolate.m:21 (same as the other two modes)
    double r = fmod(x / dx, nxd);
    if (r < 0.0) r += nxd;
    return r;
}

// phi and dphi/dz of the ES kernel at z in [-1, 1]
__device__ __forceinline__ void es_kernel(double z, double beta, double& p0, double& p1) {
    const double s2 = fma(-z, z, 1.0);
    // The end of the support: phi = e^-beta ~ 1e-18 of the peak there, but phi' = -phi beta z / sqrt(1 - z^2) has an
    // (integrable) singularity at |z| = 1.  A packet that sits on a fine-grid node -- or within rounding of one, which is
    // what x = i*dx gives -- puts a stencil node at |z| = 1 - O(1e-16), where the formula returns ~1e-18 * beta / 1e-8:
    // a spurious 2e-10 of the gradient (found by the node test of tests/test_octave_goldens.py).  The node is dropped while
    // sqrt(1 - z^2) < 1e-3: what is dropped is below e^-beta * beta / 1e-3 = 4e-14 of the peak in phi' and 1e-18 in phi.
    if (s2 <= 1e-6) { p0 = 0.0; p1 = 0.0; return; }
    const double s = sqrt(s2);
    const double e = exp(beta * (s - 1.0));
    p0 = e;
    p1 = -e * beta * z / s;
}

// first fine-grid index of the stencil and t0 = i0 - xf, so that z_a = (t0 + a) / (w/2)
__device__ __forceinline__ void stencil_origin(double xl, int nf, int& base, double& t0) {
    const double xf = xl * kNufftSigma;                  // sigma = 2: exact
    const double c = ceil(xf - HALF_W);
    t0 = c - xf;
    int i0 = (int)c % nf;
    if (i0 < 0) i0 += nf;
    base = i0;
}

// u,v,ux,uy,vx,vy at one point, computed by a QUAD of lanes (4 lanes per packet, 8 packets per warp).
// grid: double2 (u,v) at [(iy*nf + ix)], x fastest (cuFFT's output order).  Lane q of the quad owns the stencil
// columns a = q, q+4, q+8, ... (so the quad's four loads of one round are four consecutive 16-byte nodes: one 64-byte
// segment instead of four scattered lines -- the kernel is bound by L1 data-pipe wavefronts) and evaluates the kernel
// for those columns and for the rows b = q, q+4, ...; row weights travel inside the quad by shuffle.  All four lanes end
// with bit-identical sums (the butterfly adds are commutative), so the redundant packet state stays consistent.
#ifndef SWRT_NUFFT_LPP
#define SWRT_NUFFT_LPP 4
#endif
// lanes per packet: 4 = quad (shipped).  8 = octet (a 128-byte segment per round, 3 rounds instead of 5) was measured and
// is slower: 1.62e9 against 1.85e9 packet-steps/s at C3, the extra redundant per-packet work outweighs the wider segments
constexpr int LPP = SWRT_NUFFT_LPP;
constexpr int LPP_SHIFT = LPP == 8 ? 3 : 2;
static_assert(LPP == 4 || LPP == 8, "lanes per packet");
constexpr int QR = (W + LPP - 1) / LPP;          // columns (and rows) owned per lane, the last round partly empty

struct __align__(32) Node4 { double u, v, h, pad; };
__device__ __forceinline__ Node4 ldg_node4(const Node4* p) {        // SASS LDG.E.256 (read-only path)
    Node4 r;
    asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.u), "=d"(r.v), "=d"(r.h), "=d"(r.pad) : "l"(p));
    return r;
}

// MIX (swrt_ode23_packets): with mix set, every node is (1 - al) * grid + al * grid1 formed as axpby_dev_kernel forms the
// blended fine grid, so the sums equal those over that grid; without it the quad reads `grid` alone
template <bool WITH_H, bool WITH_GRAD = true, bool MIX = false>
__device__ __forceinline__ void nufft_eval6(const double2* __restrict__ grid, const double* __restrict__ uvh, int nf,
                                            double beta, double dscale, double xl, double yl, int q, int quad_base, double* F,
                                            const double2* __restrict__ grid1 = nullptr, double al = 0.0, bool mix = false) {
    int ib, jb; double tx, ty;
    stencil_origin(xl, nf, ib, tx);
    stencil_origin(yl, nf, jb, ty);
    double wx0[QR], wx1[QR], my0[QR], my1[QR];
    int ixr[QR];
#pragma unroll
    for (int r = 0; r < QR; r++) {
        const int a = q + LPP * r;
        const bool on = a < W;
        es_kernel((tx + (double)a) * (1.0 / HALF_W), beta, wx0[r], wx1[r]);
        es_kernel((ty + (double)a) * (1.0 / HALF_W), beta, my0[r], my1[r]);
        if (!on) { wx0[r] = 0.0; wx1[r] = 0.0; my0[r] = 0.0; my1[r] = 0.0; }
        if constexpr (!WITH_GRAD) { wx1[r] = 0.0; my1[r] = 0.0; }     // u, v (, H) only: the derivative sums fold away
        int ix = ib + (on ? a : 0);
        if (ix >= nf) ix -= nf;
        if (ix >= nf) ix -= nf;                // nx = 8: nf = 16 < w, the stencil wraps twice
        ixr[r] = ix;
    }
    const bool last_on = q + LPP * (QR - 1) < W;
    double U = 0, V = 0, Ux = 0, Uy = 0, Vx = 0, Vy = 0, Hs = 0;
#pragma unroll
    for (int b = 0; b < W; b++) {
        const double wy0 = __shfl_sync(0xffffffffu, my0[b >> LPP_SHIFT], quad_base | (b & (LPP - 1)));
        const double wy1 = WITH_GRAD ? __shfl_sync(0xffffffffu, my1[b >> LPP_SHIFT], quad_base | (b & (LPP - 1))) : 0.0;
        int iy = jb + b;
        if (iy >= nf) iy -= nf;
        if (iy >= nf) iy -= nf;
        double su0 = 0, su1 = 0, sv0 = 0, sv1 = 0, sh0 = 0;
#pragma unroll
        for (int r = 0; r < QR; r++) {
            double2 g = make_double2(0.0, 0.0);
            if (r < QR - 1 || last_on) {            // lanes whose column of the last round is past the stencil issue no load
                if constexpr (WITH_H) {
                    const Node4 nd = ldg_node4(reinterpret_cast<const Node4*>(uvh) + (size_t)iy * nf + ixr[r]);
                    g.x = nd.u; g.y = nd.v;
                    sh0 = fma(wx0[r], nd.h, sh0);
                } else if (MIX && mix) {
                    const double2 g0 = __ldg(grid + (size_t)iy * nf + ixr[r]), g1 = __ldg(grid1 + (size_t)iy * nf + ixr[r]);
                    const double wa = __dsub_rn(1.0, al);
                    g.x = fma(wa, g0.x, __dmul_rn(al, g1.x));
                    g.y = fma(wa, g0.y, __dmul_rn(al, g1.y));
                } else {
                    g = __ldg(grid + (size_t)iy * nf + ixr[r]);
                }
            }
            su0 = fma(wx0[r], g.x, su0); sv0 = fma(wx0[r], g.y, sv0);
            if constexpr (WITH_GRAD) { su1 = fma(wx1[r], g.x, su1); sv1 = fma(wx1[r], g.y, sv1); }
        }
        U = fma(wy0, su0, U);  V = fma(wy0, sv0, V);
        if constexpr (WITH_GRAD) {
            Ux = fma(wy0, su1, Ux); Uy = fma(wy1, su0, Uy);
            Vx = fma(wy0, sv1, Vx); Vy = fma(wy1, sv0, Vy);
        }
        if constexpr (WITH_H) Hs = fma(wy0, sh0, Hs);
    }
    double o[7] = {U, V, Ux * dscale, Uy * dscale, Vx * dscale, Vy * dscale, Hs};
#pragma unroll
    for (int c = 0; c < (WITH_H ? 7 : 6); c++) {
        if (!WITH_GRAD && c >= 2 && c < 6) { F[c] = 0.0; continue; }
        double v = o[c];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if constexpr (LPP == 8) v += __shfl_xor_sync(0xffffffffu, v, 4);
        F[c] = v;
    }
}

template <bool WITH_H>
__global__ void __launch_bounds__(kBlock) nufft_eval_kernel(const NufftArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> LPP_SHIFT;
    const int lane = threadIdx.x & 31, q = lane & (LPP - 1), qb = lane & ~(LPP - 1);
    const long long pc = p < a.n ? p : a.n - 1;              // idle quads of the last warp still take part in the shuffles
    double F[7];
    nufft_eval6<WITH_H>(a.grid, a.hgrid, a.nf, a.beta, a.dscale, reduced_coord(a.xin[pc], a.dx, a.nxd),
                        reduced_coord(a.yin[pc], a.dx, a.nxd), q, qb, F);
    if (p < a.n && q == 0) {
#pragma unroll
        for (int c = 0; c < (WITH_H ? 7 : 6); c++)
            if (a.out[c]) a.out[c][p] = F[c];
    }
}

// swrt_ode23's evaluation of the six planes: the fine grid active_nufft_grid picks for the controller's alpha (frame 0,
// frame 1 or the blend that axpby_dev_kernel wrote); nothing to do once the solve is done
__global__ void __launch_bounds__(kBlock) nufft_eval_dev_kernel(const NufftArgs a, const Ode23Sel sel) {
    if (ode23_idle(sel.ctl)) return;
    const double al = sel.ctl->al[sel.stage];
    const double2* grid = a.grid;
    if (al == 1.0 && sel.frame1) grid = static_cast<const double2*>(sel.frame1);
    else if (al != 0.0 && sel.blend) grid = static_cast<const double2*>(sel.blend);
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> LPP_SHIFT;
    const int lane = threadIdx.x & 31, q = lane & (LPP - 1), qb = lane & ~(LPP - 1);
    const long long pc = p < a.n ? p : a.n - 1;
    double F[7];
    nufft_eval6<false>(grid, nullptr, a.nf, a.beta, a.dscale, reduced_coord(a.xin[pc], a.dx, a.nxd),
                       reduced_coord(a.yin[pc], a.dx, a.nxd), q, qb, F);
    if (p < a.n && q == 0) {
#pragma unroll
        for (int c = 0; c < 6; c++)
            if (a.out[c]) a.out[c][p] = F[c];
    }
}

// swrt_ode23_packets' evaluation of the six planes at each packet's own alpha: frame 0, frame 1, or both blended node by
// node.  The choice is per quad; every quad takes part in the shuffles, finished packets store nothing.
__global__ void __launch_bounds__(kBlock) nufft_eval_pkt_kernel(const NufftArgs a, const double2* __restrict__ grid1,
                                                                const Ode23Pkt s, int stage) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> LPP_SHIFT;
    const int lane = threadIdx.x & 31, q = lane & (LPP - 1), qb = lane & ~(LPP - 1);
    const long long pc = p < a.n ? p : a.n - 1;
    const double al = grid1 ? ode23_pkt_alpha(s, stage)[pc] : 0.0;
    const double2* grid = al == 1.0 ? grid1 : a.grid;
    double F[7];
    nufft_eval6<false, true, true>(grid, nullptr, a.nf, a.beta, a.dscale, reduced_coord(a.xin[pc], a.dx, a.nxd),
                                   reduced_coord(a.yin[pc], a.dx, a.nxd), q, qb, F, grid1, al, al != 0.0 && al != 1.0);
    if (p < a.n && q == 0 && !ode23_pkt_idle(s, p)) {
#pragma unroll
        for (int c = 0; c < 6; c++)
            if (a.out[c]) a.out[c][p] = F[c];
    }
}

// ode_symplectic.m:13-21,33-37 with the six planes from the NUFFT evaluation at x1
#ifndef SWRT_NUFFT_MINB
#define SWRT_NUFFT_MINB 5     /* 96 registers: 4 / 5 / 6 / 8 blocks per SM give 1.75 / 1.84 / 1.70 / 1.15e9 packet-steps/s at C3 */
#endif
__global__ void __launch_bounds__(kBlock, SWRT_NUFFT_MINB) nufft_leapfrog_kernel(const NufftArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> LPP_SHIFT;
    const int lane = threadIdx.x & 31, q = lane & (LPP - 1), qb = lane & ~(LPP - 1);
    const long long pc = p < a.n ? p : a.n - 1;
    double x = a.x[pc], y = a.y[pc], k = a.k[pc], l = a.l[pc];
    const double h = 0.5 * a.dt;
    for (int st = 0; st < a.nsteps; st++) {
        double om = sqrt(a.f2 + a.gH * (k * k + l * l));
        x = x + h * (a.gH * k / om);
        y = y + h * (a.gH * l / om);
        double F[6];
        nufft_eval6<false>(a.grid + (size_t)st * a.gstride, nullptr, a.nf, a.beta, a.dscale, reduced_coord(x, a.dx, a.nxd), reduced_coord(y, a.dx, a.nxd), q, qb, F);
        x = x + a.dt * F[0];
        y = y + a.dt * F[1];
        const double k0 = k, l0 = l;
        k = k0 - a.dt * (F[2] * k0 + F[4] * l0);
        l = l0 - a.dt * (F[3] * k0 + F[5] * l0);
        om = sqrt(a.f2 + a.gH * (k * k + l * l));
        x = x + h * (a.gH * k / om);
        y = y + h * (a.gH * l / om);
    }
    if (p < a.n && q == 0) { a.x[p] = x; a.y[p] = y; a.k[p] = k; a.l[p] = l; }
}

// step_packet.m:37-78 / step_packet_xka.m:38-91 with the continuous fields of this mode: RK4 in x with k frozen (u, v and,
// for xka, H at the four stage positions), then RK4 in k (and a) with the gradients frozen -- at the OLD position for
// step_packet (:58-61), at the NEW one for step_packet_xka (:62-70, with cg_sw.m:22-31 evaluated at the point).  One
// launch runs `nsteps` whole steps with the packet in registers; the stage arithmetic is the expression-for-expression
// twin of rk4_stage_kernel / rk4_final_kernel (misc_kernels.cu), which the dense mode composes from separate launches.
#ifndef SWRT_NUFFT_RK4_MINB
#define SWRT_NUFFT_RK4_MINB 4
#endif
template <bool XKA>
__global__ void __launch_bounds__(kBlock, SWRT_NUFFT_RK4_MINB) nufft_rk4_kernel(const NufftArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> LPP_SHIFT;
    const int lane = threadIdx.x & 31, q = lane & (LPP - 1), qb = lane & ~(LPP - 1);
    const long long pc = p < a.n ? p : a.n - 1;
    double x = a.x[pc], y = a.y[pc], k = a.k[pc], l = a.l[pc];
    double am = XKA ? a.a[pc] : 0.0;
    const double dt = a.dt;
    for (int st = 0; st < a.nsteps; st++) {
        const double2* __restrict__ grid = a.grid + (size_t)st * a.gstride;      // fused run on pre-blended frames
        const double* __restrict__ hgrid = XKA ? a.hgrid + (size_t)st * a.hstride : nullptr;
        const double K2 = k * k + l * l;
        double F[7];
        double gux = 0, guy = 0, gvx = 0, gvy = 0;       // step_packet: gradients at the old position
        double xs = x, ys = y, ax = 0, ay = 0;
#pragma unroll 1
        for (int stage = 0; stage < 4; stage++) {
            const double xl = reduced_coord(xs, a.dx, a.nxd), yl = reduced_coord(ys, a.dx, a.nxd);
            if (!XKA && stage == 0) {
                nufft_eval6<false, true>(grid, nullptr, a.nf, a.beta, a.dscale, xl, yl, q, qb, F);
                gux = F[2]; guy = F[3]; gvx = F[4]; gvy = F[5];
            } else {
                nufft_eval6<XKA, false>(grid, hgrid, a.nf, a.beta, a.dscale, xl, yl, q, qb, F);
            }
            const double gH = XKA ? a.C0 * a.C0 * F[6] : a.C0 * a.C0;
            const double om = sqrt(a.f * a.f + gH * K2);
            const double dxs = dt * (F[0] + gH * k / om);
            const double dys = dt * (F[1] + gH * l / om);
            switch (stage) {
                case 0: ax = dxs; ay = dys; xs = x + dxs / 2; ys = y + dys / 2; break;
                case 1: ax += 2 * dxs; ay += 2 * dys; xs = x + dxs / 2; ys = y + dys / 2; break;
                case 2: ax += 2 * dxs; ay += 2 * dys; xs = x + dxs; ys = y + dys; break;
                default: {
                    const double sx = ax + dxs, sy = ay + dys;
                    xs = x + sx / 6; ys = y + sy / 6;
                }
            }
        }
        double oxi = 0.0, oyi = 0.0, dci = 0.0;
        if constexpr (XKA) {
            nufft_eval6<true, true>(grid, hgrid, a.nf, a.beta, a.dscale, reduced_coord(xs, a.dx, a.nxd),
                                    reduced_coord(ys, a.dx, a.nxd), q, qb, F);
            gux = F[2]; guy = F[3]; gvx = F[4]; gvy = F[5];
            const double gH = a.C0 * a.C0 * F[6];
            const double om = sqrt(a.f * a.f + gH * K2);
            const double cx = gH * k / om, cy = gH * l / om;
            oxi = a.f * K2 * F[1] / (2 * om);
            oyi = -a.f * K2 * F[0] / (2 * om);
            dci = (k * a.f * F[1] - l * a.f * F[0] - cx * cx - cy * cy) / om;
        }
        const double k1 = dt * (-gux * k - gvx * l - oxi);
        const double l1 = dt * (-guy * k - gvy * l - oyi);
        const double k2 = dt * (-gux * (k + k1 / 2) - gvx * (l + l1 / 2) - oxi);
        const double l2 = dt * (-guy * (k + k1 / 2) - gvy * (l + l1 / 2) - oyi);
        const double k3 = dt * (-gux * (k + k2 / 2) - gvx * (l + l2 / 2) - oxi);
        const double l3 = dt * (-guy * (k + k2 / 2) - gvy * (l + l2 / 2) - oyi);
        const double k4 = dt * (-gux * (k + k3) - gvx * (l + l3) - oxi);
        const double l4 = dt * (-guy * (k + k3) - gvy * (l + l3) - oyi);
        k = k + (k1 + 2 * k2 + 2 * k3 + k4) / 6;
        l = l + (l1 + 2 * l2 + 2 * l3 + l4) / 6;
        if constexpr (XKA) {
            const double a1 = dt * (-am * dci);
            const double a2 = dt * (-(am + a1 / 2) * dci);
            const double a3 = dt * (-(am + a2 / 2) * dci);
            const double a4 = dt * (-(am + a3) * dci);
            am = am + (a1 + 2 * a2 + 2 * a3 + a4) / 6;
        }
        x = xs; y = ys;
    }
    if (p < a.n && q == 0) {
        a.x[p] = x; a.y[p] = y; a.k[p] = k; a.l[p] = l;
        if (XKA) a.a[p] = am;
    }
}

// half-plane coefficients (g2k layout, the ky = 0 symmetrisation of fulspec.m:16 applied) -> deconvolved, zero-padded
// full spectrum of the nf x nf fine grid in FFT order: full[ky'*nf + kx'] (x fastest)
__global__ void nufft_spread_kernel(const double2* __restrict__ half, int nx, int nf, const double* __restrict__ invphi,
                                    double2* __restrict__ full) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)nf * nf) return;
    const int nkx = nx - 1, kmax = nx / 2 - 1;
    const int ixp = (int)(idx % nf), iyp = (int)(idx / nf);
    const int kx = ixp <= nf / 2 ? ixp : ixp - nf;
    const int ky = iyp <= nf / 2 ? iyp : iyp - nf;
    double2 v = make_double2(0.0, 0.0);
    if (kx >= -kmax && kx <= kmax && ky >= -kmax && ky <= kmax) {
        if (ky > 0) v = half[(size_t)ky * nkx + kx + kmax];
        else if (ky < 0) { v = half[(size_t)(-ky) * nkx + (-kx) + kmax]; v.y = -v.y; }
        else if (kx >= 0) { v = half[kx + kmax]; if (kx == 0) v.y = 0.0; }
        else { v = half[-kx + kmax]; v.y = -v.y; }
        const double s = invphi[kx < 0 ? -kx : kx] * invphi[ky < 0 ? -ky : ky];
        v.x *= s; v.y *= s;
    }
    full[idx] = v;
}
// real part of the inverse transform -> component c of a fine grid with `stride` doubles per node
__global__ void nufft_store_kernel(const double2* __restrict__ full, size_t n, int c, int stride, double* __restrict__ grid2) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) grid2[(size_t)stride * i + c] = full[i].x;
}

}  // namespace

void launch_nufft_spread(const double2* half, int nx, int nf, const double* invphi_dev, double2* full, cudaStream_t st) {
    size_t n = (size_t)nf * nf;
    nufft_spread_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(half, nx, nf, invphi_dev, full);
}
void launch_nufft_store(const double2* full, int nf, int c, int stride, double* grid2, cudaStream_t st) {
    size_t n = (size_t)nf * nf;
    nufft_store_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(full, n, c, stride, grid2);
}
cudaError_t launch_nufft_eval(const NufftArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    if (a.hgrid) nufft_eval_kernel<true><<<(unsigned)(((long long)LPP * a.n + kBlock - 1) / kBlock), kBlock, 0, st>>>(a);
    else nufft_eval_kernel<false><<<(unsigned)(((long long)LPP * a.n + kBlock - 1) / kBlock), kBlock, 0, st>>>(a);
    return cudaGetLastError();
}
cudaError_t launch_nufft_eval_dev(const NufftArgs& a, const Ode23Sel& sel, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    nufft_eval_dev_kernel<<<(unsigned)(((long long)LPP * a.n + kBlock - 1) / kBlock), kBlock, 0, st>>>(a, sel);
    return cudaGetLastError();
}
cudaError_t launch_nufft_eval_pkt(const NufftArgs& a, const double2* grid1, const Ode23Pkt& s, int stage, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    nufft_eval_pkt_kernel<<<(unsigned)(((long long)LPP * a.n + kBlock - 1) / kBlock), kBlock, 0, st>>>(a, grid1, s, stage);
    return cudaGetLastError();
}
cudaError_t launch_nufft_leapfrog(const NufftArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    nufft_leapfrog_kernel<<<(unsigned)(((long long)LPP * a.n + kBlock - 1) / kBlock), kBlock, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_nufft_rk4(const NufftArgs& a, bool xka, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    const unsigned nb = (unsigned)(((long long)LPP * a.n + kBlock - 1) / kBlock);
    if (xka) nufft_rk4_kernel<true><<<nb, kBlock, 0, st>>>(a);
    else nufft_rk4_kernel<false><<<nb, kBlock, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace swrt
