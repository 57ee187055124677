// misc_kernels.cu -- elementwise glue and diagnostics of libswrt: the ode23 RHS of
// qgsw_raytrace.m:259-265, the point-wise RK4 glue used by the SPECTRAL mode of step_packet /
// step_packet_xka, omega / Omega (symplectic_full_fourier.m:41,54-56), histcounts
// (analysis/load_data.m:39-47) and the reduction diagnostics.
#include "../../include/swrt.h"
#include "swrt_internal.h"

namespace swrt {

namespace {
inline unsigned nblk(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }

__global__ void fill_kernel(double* p, double v, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// odefun: dxdt = U + Cg*k/sqrt(f^2 + Cg^2 |k|^2), dkdt = -(grad U)^T k
struct E6 { const double* p[6]; };
// cgfac = Cg (qgsw_raytrace.m:262) or gH (SW_zero_background_raytracing.m:182-184)
__device__ __forceinline__ void rhs_at(long long i, const double* __restrict__ k, const double* __restrict__ l, const E6& e,
                                       double f, double gH, double cgfac, double* dxdt, double* dydt, double* dkdt, double* dldt) {
    const double kk = k[i], ll = l[i];
    // every product and sum rounded on its own (no FMA contraction): with the LAGRANGE6 evaluation in front, odefun is then
    // the reference's double arithmetic operation for operation (qgsw_raytrace.m:262-263)
    const double w = sqrt(__dadd_rn(__dmul_rn(f, f), __dmul_rn(gH, __dadd_rn(__dmul_rn(kk, kk), __dmul_rn(ll, ll)))));
    if (dxdt) dxdt[i] = __dadd_rn(e.p[0][i], __dmul_rn(cgfac, kk) / w);
    if (dydt) dydt[i] = __dadd_rn(e.p[1][i], __dmul_rn(cgfac, ll) / w);
    if (dkdt) dkdt[i] = -__dadd_rn(__dmul_rn(e.p[2][i], kk), __dmul_rn(e.p[4][i], ll));
    if (dldt) dldt[i] = -__dadd_rn(__dmul_rn(e.p[3][i], kk), __dmul_rn(e.p[5][i], ll));
}
// the view's idle packets write nothing.  two: the planes come from two evaluations, e at alpha 0 and e1 at alpha 1;
// between the frames they are blended at the packet's alpha, in place in e (packet i's entries are this thread's own scratch)
template <class View>
__global__ void rhs_kernel(View v, int stage, long long n, const double* __restrict__ k, const double* __restrict__ l, E6 e,
                           E6 e1, bool two, double f, double gH, double cgfac, double* dxdt, double* dydt, double* dkdt,
                           double* dldt) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || v.done() || v.idle(i)) return;
    const double al = two ? v.alpha(stage, i) : 0.0;
    E6 src;
#pragma unroll
    for (int c = 0; c < 6; c++) {
        src.p[c] = al == 1.0 ? e1.p[c] : e.p[c];
        if (al != 0.0 && al != 1.0)
            const_cast<double*>(e.p[c])[i] = __dadd_rn(__dmul_rn(__dsub_rn(1.0, al), e.p[c][i]), __dmul_rn(al, e1.p[c][i]));
    }
    rhs_at(i, k, l, src, f, gH, cgfac, dxdt, dydt, dkdt, dldt);
}

__global__ void omega_kernel(long long n, const double* __restrict__ k, const double* __restrict__ l,
                             const double* __restrict__ u, const double* __restrict__ v, double f, double gH,
                             double* omega, double* Omega_abs) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double kk = k[i], ll = l[i];
    // un-fused, in the reference's order (load_data.m:33: sqrt(f^2 + Cg^2.*dot(k,k,2))) so that omega --
    // and therefore the histogram built from it -- is bit-identical to a host evaluation
    const double w = sqrt(__dadd_rn(__dmul_rn(f, f), __dmul_rn(gH, __dadd_rn(__dmul_rn(kk, kk), __dmul_rn(ll, ll)))));
    if (omega) omega[i] = w;
    if (Omega_abs) Omega_abs[i] = __dadd_rn(w, __dadd_rn(__dmul_rn(u[i], kk), __dmul_rn(v[i], ll)));   // omega + dot(U,k)
}

// SPECTRAL-mode RK4 position stage: the continuous ray equations composed point-wise.
//   velocity = U + C with C = gH k/omega, gH = C0^2 (packet) or C0^2*H(x) (xka)
// stage 0..3 of step_packet.m:41-54; accumulates (x1 + 2x2 + 2x3 + x4) and writes the next stage
// position into xs,ys.
__global__ void rk4_stage_kernel(Rk4Args a) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const double k = a.k[i], l = a.l[i];
    const double K2 = k * k + l * l;
    const double gH = a.xka ? a.C0 * a.C0 * a.H[i] : a.C0 * a.C0;
    const double om = sqrt(a.f * a.f + gH * K2);
    const double dxs = a.dt * (a.u[i] + gH * k / om);
    const double dys = a.dt * (a.v[i] + gH * l / om);
    const double x = a.x[i], y = a.y[i];
    switch (a.stage) {
        case 0: a.ax[i] = dxs; a.ay[i] = dys; a.xs[i] = x + dxs / 2; a.ys[i] = y + dys / 2; break;
        case 1: a.ax[i] += 2 * dxs; a.ay[i] += 2 * dys; a.xs[i] = x + dxs / 2; a.ys[i] = y + dys / 2; break;
        case 2: a.ax[i] += 2 * dxs; a.ay[i] += 2 * dys; a.xs[i] = x + dxs; a.ys[i] = y + dys; break;
        default: {
            const double sx = a.ax[i] + dxs, sy = a.ay[i] + dys;
            a.xs[i] = x + sx / 6; a.ys[i] = y + sy / 6;   // = Pout.x, Pout.y
        }
    }
}

// k (and a) update with frozen gradients; commits the new position held in xs,ys.
__global__ void rk4_final_kernel(Rk4Args a) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const double k = a.k[i], l = a.l[i], dt = a.dt;
    const double uxi = a.ux[i], uyi = a.uy[i], vxi = a.vx[i], vyi = a.vy[i];
    double oxi = 0.0, oyi = 0.0, dci = 0.0;
    if (a.xka) {   // cg_sw.m:22-31 evaluated at the point
        const double K2 = k * k + l * l;
        const double gH = a.C0 * a.C0 * a.H[i];
        const double om = sqrt(a.f * a.f + gH * K2);
        const double cx = gH * k / om, cy = gH * l / om;
        const double u = a.u[i], v = a.v[i];
        oxi = a.f * K2 * v / (2 * om);
        oyi = -a.f * K2 * u / (2 * om);
        dci = (k * a.f * v - l * a.f * u - cx * cx - cy * cy) / om;
    }
    const double k1 = dt * (-uxi * k - vxi * l - oxi);
    const double l1 = dt * (-uyi * k - vyi * l - oyi);
    const double k2 = dt * (-uxi * (k + k1 / 2) - vxi * (l + l1 / 2) - oxi);
    const double l2 = dt * (-uyi * (k + k1 / 2) - vyi * (l + l1 / 2) - oyi);
    const double k3 = dt * (-uxi * (k + k2 / 2) - vxi * (l + l2 / 2) - oxi);
    const double l3 = dt * (-uyi * (k + k2 / 2) - vyi * (l + l2 / 2) - oyi);
    const double k4 = dt * (-uxi * (k + k3) - vxi * (l + l3) - oxi);
    const double l4 = dt * (-uyi * (k + k3) - vyi * (l + l3) - oyi);
    a.k[i] = k + (k1 + 2 * k2 + 2 * k3 + k4) / 6;
    a.l[i] = l + (l1 + 2 * l2 + 2 * l3 + l4) / 6;
    if (a.xka) {
        const double am = a.a[i];
        const double a1 = dt * (-am * dci);
        const double a2 = dt * (-(am + a1 / 2) * dci);
        const double a3 = dt * (-(am + a2 / 2) * dci);
        const double a4 = dt * (-(am + a3) * dci);
        a.a[i] = am + (a1 + 2 * a2 + 2 * a3 + a4) / 6;
    }
    a.x[i] = a.xs[i];
    a.y[i] = a.ys[i];
}

// histcounts(w, edges): bin i = [e_i, e_{i+1}), last bin closed; NaN / out of range dropped.
constexpr int kMaxSmemBins = 4096;
// the bin of v, e[0] <= v <= e[nb]: the last a with e[a] <= v; v == e[nb] lands in a = nb-1 because b never drops below nb
__device__ __forceinline__ int bin_index(const double* e, int nb, double v) {
    int a = 0, b = nb;
    while (b - a > 1) {
        int m = (a + b) >> 1;
        if (e[m] <= v) a = m; else b = m;
    }
    return a;
}
__global__ void hist_kernel(long long n, const double* __restrict__ w, const double* __restrict__ edges, int nedges,
                            unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned char hs[];
    double* se = reinterpret_cast<double*>(hs);
    unsigned int* sc = reinterpret_cast<unsigned int*>(se + nedges);
    const int nb = nedges - 1;
    for (int i = threadIdx.x; i < nedges; i += blockDim.x) se[i] = edges[i];
    for (int i = threadIdx.x; i < nb; i += blockDim.x) sc[i] = 0;
    __syncthreads();
    const double lo = se[0], hi = se[nb];
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double v = w[i];
        if (!(v >= lo && v <= hi)) continue;   // also drops NaN
        atomicAdd(&sc[bin_index(se, nb, v)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += blockDim.x)
        if (sc[i]) atomicAdd(&counts[i], (unsigned long long)sc[i]);
}

// ideal_omega_distribution.m:3-11: omega_abs = omega_0 + U(:,1)*kx' + U(:,2)*ky' over (grid point, angle),
// histogrammed with explicit edges.  Un-fused arithmetic in the reference's order, so the counts are
// bit-identical to a host histogram of the same U.
__global__ void ideal_hist_kernel(long long npts, const double* __restrict__ u, const double* __restrict__ v,
                                  const double* __restrict__ kvx, const double* __restrict__ kvy, int nang, double omega0,
                                  const double* __restrict__ edges, int nedges, unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned char hs[];
    double* se = reinterpret_cast<double*>(hs);
    double* sk = se + nedges;                       // kvx then kvy
    unsigned int* sc = reinterpret_cast<unsigned int*>(sk + 2 * nang);
    const int nb = nedges - 1;
    for (int i = threadIdx.x; i < nedges; i += blockDim.x) se[i] = edges[i];
    for (int i = threadIdx.x; i < nang; i += blockDim.x) { sk[i] = kvx[i]; sk[nang + i] = kvy[i]; }
    for (int i = threadIdx.x; i < nb; i += blockDim.x) sc[i] = 0;
    __syncthreads();
    const double lo = se[0], hi = se[nb];
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += stride) {
        const double uu = u[i], vv = v[i];
        for (int j = 0; j < nang; j++) {
            const double w = __dadd_rn(omega0, __dadd_rn(__dmul_rn(uu, sk[j]), __dmul_rn(vv, sk[nang + j])));
            if (!(w >= lo && w <= hi)) continue;
            atomicAdd(&sc[bin_index(se, nb, w)], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += blockDim.x)
        if (sc[i]) atomicAdd(&counts[i], (unsigned long long)sc[i]);
}

// ---- swrt_packet_quantity / swrt_hist2 ------------------------------------------------------------------------------
// x periodic in [0, L): every operation rounded on its own (this file is compiled with FMA contraction)
__device__ __forceinline__ double wrap_period(double x, double L) {
    double r = __dsub_rn(x, __dmul_rn(L, floor(__ddiv_rn(x, L))));
    if (r < 0.0) r = __dadd_rn(r, L);
    return r >= L ? 0.0 : r;
}
// quantity q of packet i: the one definition both swrt_packet_quantity and the histogram bin, so a binned value is
// exactly the value the caller reads back.  OMEGA / OMEGA_ABS are omega_kernel's outputs (bit-identical to swrt_omega).
__device__ __forceinline__ double packet_quantity(int q, const PktQ& p, long long i) {
    switch (q) {
        case SWRT_Q_XMOD: return wrap_period(p.x[i], p.L);
        case SWRT_Q_YMOD: return wrap_period(p.y[i], p.L);
        case SWRT_Q_K: return p.k[i];
        case SWRT_Q_L: return p.l[i];
        case SWRT_Q_KMAG: { const double k = p.k[i], l = p.l[i]; return __dsqrt_rn(__dadd_rn(__dmul_rn(k, k), __dmul_rn(l, l))); }
        case SWRT_Q_THETA: return atan2(p.l[i], p.k[i]);
        case SWRT_Q_OMEGA: return p.om[i];
        default: return p.Om[i];
    }
}
__global__ void packet_quantity_kernel(long long n, int q, PktQ p, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = packet_quantity(q, p, i);
}
// histcounts2: bin (i, j) = [xe_i, xe_i+1) x [ye_j, ye_j+1), last bin closed on each axis, counts[i + j*nbx].  Both edge
// arrays sit in shared memory; SMEM: so do the CTA's u32 counters, flushed (non-zero bins) with u64 global atomics, else
// every count goes to the global u64 counters.  The lanes of a warp holding the same bin are counted by one atomic of
// their number (__match_any_sync), so a histogram whose packets crowd into a few bins -- a wavenumber ring -- does not
// serialise on those addresses.  The loop is warp-uniform so that every lane takes part in the match.
template <bool SMEM>
__global__ void __launch_bounds__(1024) hist2_kernel(long long n, int qx, int qy, PktQ p, const double* __restrict__ edges,
                                                    int nxe, int nye, unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned char hs[];
    double* ex = reinterpret_cast<double*>(hs);
    double* ey = ex + nxe;
    unsigned int* sc = reinterpret_cast<unsigned int*>(ey + nye);
    const int nbx = nxe - 1, nby = nye - 1;
    for (int i = threadIdx.x; i < nxe + nye; i += blockDim.x) ex[i] = edges[i];
    if (SMEM)
        for (int i = threadIdx.x; i < nbx * nby; i += blockDim.x) sc[i] = 0;
    __syncthreads();
    const double xlo = ex[0], xhi = ex[nbx], ylo = ey[0], yhi = ey[nby];
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < n; i0 += stride) {
        const long long i = i0 + lane;
        int bin = -1;
        if (i < n) {
            const double vx = packet_quantity(qx, p, i), vy = packet_quantity(qy, p, i);
            if (vx >= xlo && vx <= xhi && vy >= ylo && vy <= yhi)             // also drops NaN
                bin = bin_index(ex, nbx, vx) + bin_index(ey, nby, vy) * nbx;
        }
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && lane == __ffs(peers) - 1) {
            if (SMEM) atomicAdd(&sc[bin], (unsigned)__popc(peers));
            else atomicAdd(&counts[bin], (unsigned long long)__popc(peers));
        }
    }
    if (SMEM) {
        __syncthreads();
        for (int i = threadIdx.x; i < nbx * nby; i += blockDim.x)
            if (sc[i]) atomicAdd(&counts[i], (unsigned long long)sc[i]);
    }
}

// ---- swrt_weight_scale / swrt_hist2_sums ----------------------------------------------------------------------------
__device__ __forceinline__ double packet_weight(int kind, const PktQ& p, const double* a, long long i) {
    const double ai = a[i];
    switch (kind) {
        case SWRT_W_ACTION: return ai;
        case SWRT_W_ENERGY: return __dmul_rn(p.om[i], ai);
        case SWRT_W_PSEUDO_K: return __dmul_rn(p.k[i], ai);
        default: return __dmul_rn(p.l[i], ai);
    }
}
// the largest finite |w| of each kind -> its frexp exponent E (max |w| < 2^E), biased: a block reduction, then one
// atomicMax per kind
__global__ void __launch_bounds__(256) weight_scale_kernel(long long n, WeightKinds w, PktQ p, const double* __restrict__ a,
                                                           int* __restrict__ exp_dev) {
    __shared__ int se[SWRT_MAX_WEIGHTS];
    if (threadIdx.x < SWRT_MAX_WEIGHTS) se[threadIdx.x] = 0;
    __syncthreads();
    double m[SWRT_MAX_WEIGHTS] = {0.0, 0.0, 0.0, 0.0};
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
#pragma unroll
        for (int v = 0; v < SWRT_MAX_WEIGHTS; v++) {
            if (v >= w.n) break;
            const double x = fabs(packet_weight(w.kind[v], p, a, i));
            if (x <= 1.7976931348623157e308) m[v] = fmax(m[v], x);         // finite only (NaN compares false)
        }
    }
#pragma unroll
    for (int v = 0; v < SWRT_MAX_WEIGHTS; v++) {
        if (v >= w.n) break;
        int e = 0;
        if (m[v] > 0.0) { frexp(m[v], &e); e += kScaleBias; }
        e = __reduce_max_sync(0xffffffffu, e);
        if ((threadIdx.x & 31) == 0 && e) atomicMax(&se[v], e);
    }
    __syncthreads();
    if (threadIdx.x < w.n && se[threadIdx.x]) atomicMax(&exp_dev[threadIdx.x], se[threadIdx.x]);
}
// 2^s for -1022 <= s <= 1023
__device__ __forceinline__ double pow2(int s) { return __longlong_as_double((long long)(s + 1023) << 52); }
// Per-bin fixed-point sums.  The loop and the bin of a packet are hist2_kernel's.  Each weight w of a binned packet
// becomes |q| = rint(|w| 2^(95-E)) < 2^95 (the scaling, by two powers of two so that each stays a normal number, is
// exact; rint is the one rounding) and three 32-bit digits of |q|, split by exact fp64 operations and signed like w.  The
// lanes of a warp that share a bin (__match_any_sync) add their digits as signed 16-bit halves with one redux each
// (32 lanes * 2^16 fits an int), and the lowest of them adds the digit sums (< 2^37 in magnitude) to the bin's int64
// counters.  A weight that is not finite or not below 2^E counts in the bin's fourth counter instead.
__global__ void __launch_bounds__(1024) hist2_sums_kernel(long long n, int qx, int qy, PktQ p, const double* __restrict__ a,
                                                         WeightKinds w, const int* __restrict__ exp_dev,
                                                         const double* __restrict__ edges, int nxe, int nye,
                                                         long long* __restrict__ acc, unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned char hs[];
    double* ex = reinterpret_cast<double*>(hs);
    double* ey = ex + nxe;
    const int nbx = nxe - 1, nby = nye - 1;
    const long long nb = (long long)nbx * nby;
    for (int i = threadIdx.x; i < nxe + nye; i += blockDim.x) ex[i] = edges[i];
    double f1[SWRT_MAX_WEIGHTS], f2[SWRT_MAX_WEIGHTS];
#pragma unroll
    for (int v = 0; v < SWRT_MAX_WEIGHTS; v++) {
        const int be = v < w.n ? exp_dev[v] : 0;
        const int s = 95 - (be ? be - kScaleBias : 0), s1 = s >> 1;     // -1073 <= E <= 1024: both halves are normal
        f1[v] = pow2(s1); f2[v] = pow2(s - s1);
    }
    __syncthreads();
    const double xlo = ex[0], xhi = ex[nbx], ylo = ey[0], yhi = ey[nby];
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < n; i0 += stride) {
        const long long i = i0 + lane;
        int bin = -1;
        if (i < n) {
            const double vx = packet_quantity(qx, p, i), vy = packet_quantity(qy, p, i);
            if (vx >= xlo && vx <= xhi && vy >= ylo && vy <= yhi)             // also drops NaN
                bin = bin_index(ex, nbx, vx) + bin_index(ey, nby, vy) * nbx;
        }
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin < 0) continue;
        const bool leader = lane == __ffs(peers) - 1;
        if (leader && counts) atomicAdd(&counts[bin], (unsigned long long)__popc(peers));
#pragma unroll
        for (int v = 0; v < SWRT_MAX_WEIGHTS; v++) {
            if (v >= w.n) break;
            const double wt = packet_weight(w.kind[v], p, a, i);
            const double qd = __dmul_rn(__dmul_rn(fabs(wt), f1[v]), f2[v]);
            const bool bad = !(qd < 0x1p95);                                    // NaN, inf, or |w| >= 2^E
            int piece[6] = {0, 0, 0, 0, 0, 0};
            if (!bad) {
                const double q = rint(qd);
                const double h2 = floor(__dmul_rn(q, 0x1p-64));
                const double r = __dsub_rn(q, __dmul_rn(h2, 0x1p64));
                const double h1 = floor(__dmul_rn(r, 0x1p-32));
                const double h0 = __dsub_rn(r, __dmul_rn(h1, 0x1p32));
                const unsigned d[3] = {(unsigned)h0, (unsigned)h1, (unsigned)h2};
                const int sg = wt < 0.0 ? -1 : 1;
#pragma unroll
                for (int c = 0; c < 3; c++) { piece[2 * c] = sg * (int)(d[c] & 0xffffu); piece[2 * c + 1] = sg * (int)(d[c] >> 16); }
            }
            long long* cell = acc + 4 * ((long long)v * nb + bin);
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const long long s = (long long)__reduce_add_sync(peers, piece[2 * c]) +
                                    (long long)__reduce_add_sync(peers, piece[2 * c + 1]) * 65536;
                if (leader && s) atomicAdd(reinterpret_cast<unsigned long long*>(cell + c), (unsigned long long)s);
            }
            const int nbad = __reduce_add_sync(peers, bad ? 1 : 0);
            if (leader && nbad) atomicAdd(reinterpret_cast<unsigned long long*>(cell + 3), (unsigned long long)nbad);
        }
    }
}

// partial sums per block, then one block reduces the partials in a fixed order (deterministic)
constexpr int kDiagBlocks = 296;
__global__ void __launch_bounds__(256) diag_partial_kernel(long long n, const double* __restrict__ x,
                                                            const double* __restrict__ y, const double* __restrict__ k,
                                                            const double* __restrict__ l, const double* __restrict__ a,
                                                            const double* __restrict__ om, const double* __restrict__ Om,
                                                            double* __restrict__ part) {
    double s_om = 0, s_Om = 0, mx = -1e300, mn = 1e300, nf = 0, s_a = 0, s_oa = 0;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double w = om[i], W = Om[i];
        const bool fin = isfinite(x[i]) && isfinite(y[i]) && isfinite(k[i]) && isfinite(l[i]);
        if (!fin) { nf += 1.0; continue; }
        const double am = a ? a[i] : 1.0;
        s_om += w; s_Om += W; s_a += am; s_oa += w * am;
        mx = fmax(mx, w); mn = fmin(mn, w);
    }
    __shared__ double sh[7][256];
    const int t = threadIdx.x;
    sh[0][t] = s_om; sh[1][t] = s_Om; sh[2][t] = mx; sh[3][t] = mn; sh[4][t] = nf; sh[5][t] = s_a; sh[6][t] = s_oa;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (t < s) {
            sh[0][t] += sh[0][t + s]; sh[1][t] += sh[1][t + s];
            sh[2][t] = fmax(sh[2][t], sh[2][t + s]); sh[3][t] = fmin(sh[3][t], sh[3][t + s]);
            sh[4][t] += sh[4][t + s]; sh[5][t] += sh[5][t + s]; sh[6][t] += sh[6][t + s];
        }
        __syncthreads();
    }
    if (t == 0)
        for (int q = 0; q < 7; q++) part[(size_t)blockIdx.x * 8 + q] = sh[q][0];
}
__global__ void diag_final_kernel(int nblocks, const double* __restrict__ part, long long n, double* __restrict__ out8) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double s_om = 0, s_Om = 0, mx = -1e300, mn = 1e300, nf = 0, s_a = 0, s_oa = 0;
    for (int b = 0; b < nblocks; b++) {
        const double* p = part + (size_t)b * 8;
        s_om += p[0]; s_Om += p[1]; mx = fmax(mx, p[2]); mn = fmin(mn, p[3]); nf += p[4]; s_a += p[5]; s_oa += p[6];
    }
    out8[0] = s_om; out8[1] = s_Om; out8[2] = mx; out8[3] = mn; out8[4] = nf; out8[5] = s_a; out8[6] = (double)n; out8[7] = s_oa;
}
// ---- Bogacki-Shampine 3(2) building blocks (MATLAB ode23, called by qgsw_raytrace.m:149) ----------
// stage state: yt = y + h*(b1 f1 + b2 f2 + b3 f3) for the four components x,y,k,l
__device__ __forceinline__ void bs23_stage_at(const Bs23Args& a, long long i, double hb1, double hb2, double hb3) {
#pragma unroll
    for (int c = 0; c < 4; c++) {
        // y + f*hB(:,j), hB = h*B, accumulated column by column with every product and sum rounded on its own
        double acc = __dmul_rn(a.f[0][c][i], hb1);
        if (hb2 != 0.0) acc = __dadd_rn(acc, __dmul_rn(a.f[1][c][i], hb2));
        if (hb3 != 0.0) acc = __dadd_rn(acc, __dmul_rn(a.f[2][c][i], hb3));
        a.yt[c][i] = __dadd_rn(a.y[c][i], acc);
    }
}
// hB(:,stage) with each product h*B rounded on its own: A = [1/2 3/4 1], B = [1/2 0 2/9; 0 3/4 1/3; 0 0 4/9; 0 0 0]
__device__ __forceinline__ void bs23_stage_h(const Bs23Args& a, long long i, int stage, double h) {
    if (stage == 0) bs23_stage_at(a, i, __dmul_rn(h, 0.5), 0.0, 0.0);
    else if (stage == 1) bs23_stage_at(a, i, 0.0, __dmul_rn(h, 0.75), 0.0);
    else bs23_stage_at(a, i, __dmul_rn(h, 2.0 / 9.0), __dmul_rn(h, 1.0 / 3.0), __dmul_rn(h, 4.0 / 9.0));
}
template <class View>
__global__ void bs23_stage_kernel(Bs23Args a, View v, int stage) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n || v.done() || v.idle(i)) return;
    bs23_stage_h(a, i, stage, v.h(i));
}
// err = max_i |(f*E)_i| / max(max(|y_i|,|ynew_i|), threshold)   (without the absh factor);
// mode 1: rh = max_i |f1_i| / max(|y_i|, threshold) for the initial step size
// packet i's four ratios folded into the running max m
__device__ __forceinline__ double bs23_norm_packet(const Bs23Args& a, long long i, int mode, double thr, double m) {
    const double E1 = -5.0 / 72.0, E2 = 1.0 / 12.0, E3 = 1.0 / 9.0, E4 = -1.0 / 8.0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        double num, den;
        if (mode == 1) { num = fabs(a.f[0][c][i]); den = fmax(fabs(a.y[c][i]), thr); }
        else {
            num = fabs(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.f[0][c][i], E1), __dmul_rn(a.f[1][c][i], E2)),
                                          __dmul_rn(a.f[2][c][i], E3)), __dmul_rn(a.f[3][c][i], E4)));
            den = fmax(fmax(fabs(a.y[c][i]), fabs(a.yt[c][i])), thr);
        }
        const double r = num / den;
        m = (r > m || r != r) ? r : m;              // NaN propagates (a blown-up packet fails the step)
    }
    return m;
}
__device__ __forceinline__ void bs23_norm_body(const Bs23Args& a, int mode, double thr, unsigned long long* out) {
    double m = 0.0;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride) m = bs23_norm_packet(a, i, mode, thr, m);
    __shared__ double sh[256];
    sh[threadIdx.x] = m;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) { double o = sh[threadIdx.x + s], v = sh[threadIdx.x]; sh[threadIdx.x] = (o > v || o != o) ? o : v; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double v = sh[0];
        if (v != v) v = __longlong_as_double(0x7ff0000000000000LL);     // NaN -> +inf so that the integer max orders it last
        atomicMax(out, (unsigned long long)__double_as_longlong(v));     // non-negative doubles order like their bit patterns
    }
}
// MODE a constant: a run-time mode keeps both ratios' registers live (54 instead of 32)
template <int MODE, class View>
__global__ void __launch_bounds__(256) bs23_norm_kernel(Bs23Args a, View v, double thr, unsigned long long* out) {
    if (v.done()) return;
    bs23_norm_body(a, MODE, thr, out);
}
// y <- ynew, f1 <- f4 (first same as last)
__device__ __forceinline__ void bs23_accept_at(const Bs23Args& a, long long i) {
#pragma unroll
    for (int c = 0; c < 4; c++) { a.y[c][i] = a.yt[c][i]; a.f[0][c][i] = a.f[3][c][i]; }
}
// predicated on the controller's decision
template <class View>
__global__ void bs23_accept_kernel(Bs23Args a, View v) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n || !v.accepted()) return;
    bs23_accept_at(a, i);
}
// ntrp23: out = y + (f1 w1 + f2 w2 + f3 w3 + f4 w4), w_j = hstep * (BI_j . [s s^2 s^3])
struct Bs23Interp { double w[4]; double* out[4]; };
__global__ void bs23_interp_kernel(Bs23Args a, Bs23Interp q) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
#pragma unroll
    for (int c = 0; c < 4; c++)
        q.out[c][i] = __dadd_rn(a.y[c][i], __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.f[0][c][i], q.w[0]), __dmul_rn(a.f[1][c][i], q.w[1])),
                                                               __dmul_rn(a.f[2][c][i], q.w[2])), __dmul_rn(a.f[3][c][i], q.w[3])));
}

// ---- swrt_ode23: the step-size controller of reference_api.ode23 in device memory ------------------------------------
// Every scalar operation is rounded on its own, in the host controller's order; Python's min / max are restated with their
// argument order (min(a, b) keeps a unless b < a), which decides what a NaN operand yields.
__device__ __forceinline__ double py_min(double a, double b) { return b < a ? b : a; }
__device__ __forceinline__ double py_max(double a, double b) { return b > a ? b : a; }
__device__ __forceinline__ double eps16(double t) {          // 16 * eps(t) = 16 * np.spacing(abs(t))
    t = fabs(t);
    return __dmul_rn(16.0, __dsub_rn(nextafter(t, __longlong_as_double(0x7ff0000000000000LL)), t));
}
__device__ __forceinline__ double ode23_alpha(const Ode23Ctl& c, double tt) { return c.tmax != 0.0 ? __ddiv_rn(tt, c.tmax) : 0.0; }
// The rules below act on one controller state: swrt_ode23's Ode23Ctl in device memory, or a packet's state loaded into a
// local Ode23Ctl by swrt_ode23_packets' kernels.  One copy of the rules keeps the two solves' decisions the same.
// the attempt from t with step h: tnew and the alphas of the three new RHS evaluations
__device__ __forceinline__ void ode23_set_attempt(Ode23Ctl& c) {
    c.tnew = c.last ? c.tfinal : __dadd_rn(c.t, c.h);
    c.al[0] = ode23_alpha(c, __dadd_rn(c.t, __dmul_rn(0.5, c.h)));
    c.al[1] = ode23_alpha(c, __dadd_rn(c.t, __dmul_rn(0.75, c.h)));
    c.al[2] = ode23_alpha(c, c.tnew);
}
// head of the host controller's outer loop: hmin, the MaxStep clamp and the 1.1 stretch onto tfinal.  Every step is
// h = tdir * absh (exact: tdir is +1 or -1).
__device__ __forceinline__ void ode23_new_step(Ode23Ctl& c) {
    c.hmin = eps16(c.t);
    c.absh = py_min(c.hmax, py_max(c.hmin, c.absh));
    c.h = __dmul_rn(c.tdir, c.absh);
    c.last = 0;
    if (__dmul_rn(1.1, c.absh) >= fabs(__dsub_rn(c.tfinal, c.t))) {
        c.h = __dsub_rn(c.tfinal, c.t);
        c.absh = fabs(c.h);
        c.last = 1;
    }
    c.nofailed = 1;
    ode23_set_attempt(c);
}
// after f1 and the scale norm: the initial step (rh, htspan rule, hmin) and the first attempt
__device__ __forceinline__ void ode23_init(Ode23Ctl& c, double nrm) {
    const double rh = __ddiv_rn(nrm, c.rh_den);
    c.nfevals = 1;
    c.hmin = eps16(c.t);
    double absh = py_min(c.hmax, c.htspan);
    if (__dmul_rn(absh, rh) > 1.0) absh = __ddiv_rn(1.0, rh);
    c.absh = py_max(absh, c.hmin);
    c.nxt = c.nxt_end = 1;
    ode23_new_step(c);
}
// after an attempt's norm: accept or reject, the next h and stage alphas; the dense rows [nxt, nxt_end) the accepted
// step passes
__device__ __forceinline__ void ode23_control(Ode23Ctl& c, double nrm) {
    c.accepted = 0;
    c.nxt = c.nxt_end;
    if (c.done || c.status) return;
    const double err = __dmul_rn(c.absh, nrm);
    c.err = err;
    c.nfevals += 3;
    if (!(err <= c.rtol)) {                    // also catches NaN
        c.nfailed++;
        if (c.absh <= c.hmin) { c.status = 1; return; }
        if (c.nofailed) {
            c.nofailed = 0;
            c.absh = isfinite(err) ? py_max(c.hmin, __dmul_rn(c.absh, py_max(0.5, __dmul_rn(0.8, pow_third(__ddiv_rn(c.rtol, err))))))
                                   : py_max(c.hmin, __dmul_rn(0.5, c.absh));
        } else {
            c.absh = py_max(c.hmin, __dmul_rn(0.5, c.absh));
        }
        c.h = __dmul_rn(c.tdir, c.absh);
        c.last = 0;
        ode23_set_attempt(c);
        return;
    }
    if (c.htrace && c.nsteps < c.hcap) c.htrace[c.nsteps] = c.h;
    c.nsteps++;
    c.accepted = 1;
    c.t_acc = c.t; c.h_acc = c.h;
    if (c.ntspan > 2) {
        int j = c.nxt;
        while (j < c.ntspan && __dmul_rn(c.tdir, __dsub_rn(c.tnew, c.tspan[j])) >= 0.0) j++;
        c.nxt_end = j;
    }
    if (c.nofailed) {
        const double temp = __dmul_rn(1.25, pow_third(__ddiv_rn(err, c.rtol)));
        c.absh = temp > 0.2 ? __ddiv_rn(c.absh, temp) : __dmul_rn(5.0, c.absh);
    }
    c.t = c.tnew;
    if (c.last) c.done = 1;
    else ode23_new_step(c);
}
__device__ __forceinline__ double take_norm(unsigned long long* norm) {
    const double v = __longlong_as_double((long long)*norm);
    *norm = 0ull;                              // ready for the next attempt's atomicMax
    return v;
}
// after f1 and the scale norm of swrt_bs23_begin
__global__ void ode23_init_kernel(Ode23Ctl* c, unsigned long long* norm) { ode23_init(*c, take_norm(norm)); }
__global__ void ode23_control_kernel(Ode23Ctl* c, unsigned long long* norm) { ode23_control(*c, take_norm(norm)); }
// the ntrp23 weights at s of a step of size h, as swrt_bs23_interp forms them
__device__ __forceinline__ void ntrp23_weights(double s, double h, double w[4]) {
    const double s2 = __dmul_rn(s, s), s3 = __dmul_rn(s2, s);
    w[0] = __dmul_rn(h, __dadd_rn(__dsub_rn(s, __dmul_rn(4.0 / 3.0, s2)), __dmul_rn(5.0 / 9.0, s3)));
    w[1] = __dmul_rn(h, __dsub_rn(s2, __dmul_rn(2.0 / 3.0, s3)));
    w[2] = __dmul_rn(h, __dsub_rn(__dmul_rn(4.0 / 3.0, s2), __dmul_rn(8.0 / 9.0, s3)));
    w[3] = __dmul_rn(h, __dadd_rn(-s2, s3));
}
// ntrp23 rows [c.nxt, c.nxt_end) of packet i after the accepted step: s == 1 gives ynew itself
__device__ __forceinline__ void bs23_rows_at(const Bs23Args& a, long long i, const Ode23Ctl& c) {
    const double t0 = c.t_acc, h = c.h_acc, tnew = c.t;
    for (int j = c.nxt; j < c.nxt_end; j++) {
        const double tj = c.tspan[j];
        const double s = tj == tnew ? 1.0 : __ddiv_rn(__dsub_rn(tj, t0), h);
        double* row = c.yout + (size_t)j * 4 * a.n;
        if (s == 1.0) {
#pragma unroll
            for (int c = 0; c < 4; c++) row[(size_t)c * a.n + i] = a.yt[c][i];
            continue;
        }
        double w[4];
        ntrp23_weights(s, h, w);
#pragma unroll
        for (int c = 0; c < 4; c++)
            row[(size_t)c * a.n + i] = __dadd_rn(a.y[c][i], __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.f[0][c][i], w[0]), __dmul_rn(a.f[1][c][i], w[1])),
                                                                             __dmul_rn(a.f[2][c][i], w[2])), __dmul_rn(a.f[3][c][i], w[3])));
    }
}
__global__ void bs23_interp_dev_kernel(Bs23Args a, const Ode23Ctl* ctl) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n || !ctl->accepted) return;
    bs23_rows_at(a, i, *ctl);
}
// ---- swrt_ode23_packets: the same rules, one controller per packet ---------------------------------------------------
__device__ __forceinline__ void pkt_load(const Ode23Pkt& s, long long i, long long n, Ode23Ctl& c) {
    c.t = s.t[i]; c.absh = s.absh[i]; c.h = s.h[i]; c.hmin = s.hmin[i]; c.tnew = s.tnew[i];
    c.t_acc = s.t_acc[i]; c.h_acc = s.h_acc[i];
#pragma unroll
    for (int q = 0; q < 3; q++) c.al[q] = s.al[q][i];
    const int fl = s.flags[i];
    c.last = (fl & kPktLast) != 0; c.nofailed = (fl & kPktNofailed) != 0; c.done = (fl & kPktDone) != 0;
    c.status = (fl & kPktStopped) != 0;
    c.nsteps = s.cnt[i]; c.nfailed = s.cnt[n + i];
    c.nxt = c.nxt_end = s.nxt[i];
}
__device__ __forceinline__ void pkt_store(const Ode23Pkt& s, long long i, long long n, const Ode23Ctl& c) {
    s.t[i] = c.t; s.absh[i] = c.absh; s.h[i] = c.h; s.hmin[i] = c.hmin; s.tnew[i] = c.tnew;
    s.t_acc[i] = c.t_acc; s.h_acc[i] = c.h_acc;
#pragma unroll
    for (int q = 0; q < 3; q++) s.al[q][i] = c.al[q];
    s.flags[i] = (c.last ? kPktLast : 0) | (c.nofailed ? kPktNofailed : 0) | (c.done ? kPktDone : 0) | (c.status ? kPktStopped : 0);
    s.cnt[i] = (int)c.nsteps; s.cnt[n + i] = (int)c.nfailed; s.cnt[2 * n + i] = c.status;
    s.nxt[i] = c.nxt_end;
}
// the error norm of packet i alone, as bs23_norm_body and its atomicMax deliver it for a one-packet ensemble
__device__ __forceinline__ double pkt_norm(const Bs23Args& a, long long i, int mode, double thr) {
    const double m = bs23_norm_packet(a, i, mode, thr, 0.0);
    return m != m ? __longlong_as_double(0x7ff0000000000000LL) : m;
}
// ---- events (swrt_ode23_packets_events): every operation rounded on its own (this file is compiled with FMA contraction) --
// g_j(x, y, k, l); OMEGA is omega_kernel's expression, so an event level and a histogram edge agree on a state's side
__device__ __forceinline__ double ev_g(int kind, double level, double f, double gH, const double v[4]) {
    const double kl = __dadd_rn(__dmul_rn(v[2], v[2]), __dmul_rn(v[3], v[3]));
    const double g = kind == SWRT_EVENT_X ? v[0] : kind == SWRT_EVENT_Y ? v[1] : kind == SWRT_EVENT_K ? v[2]
                   : kind == SWRT_EVENT_L ? v[3] : kind == SWRT_EVENT_KMAG ? __dsqrt_rn(kl)
                   : __dsqrt_rn(__dadd_rn(__dmul_rn(f, f), __dmul_rn(gH, kl)));
    return __dsub_rn(g, level);
}
// one accepted step of a packet: y, f1..f4 and ynew, from t0 with step h to tnew
struct EvStep { double y[4], f[4][4], yn[4]; double t0, h, tnew; };
// the step's ntrp23 interpolant at tau, exactly as bs23_rows_at writes a dense row (p(tnew) = ynew)
__device__ __forceinline__ void ev_point(const EvStep& q, double tau, double out[4]) {
    const double s = tau == q.tnew ? 1.0 : __ddiv_rn(__dsub_rn(tau, q.t0), q.h);
    if (s == 1.0) {
#pragma unroll
        for (int c = 0; c < 4; c++) out[c] = q.yn[c];
        return;
    }
    double w[4];
    ntrp23_weights(s, q.h, w);
#pragma unroll
    for (int c = 0; c < 4; c++)
        out[c] = __dadd_rn(q.y[c], __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(q.f[0][c], w[0]), __dmul_rn(q.f[1][c], w[1])),
                                                       __dmul_rn(q.f[2][c], w[2])), __dmul_rn(q.f[3][c], w[3])));
}
__device__ __forceinline__ double spacing(double t) {          // np.spacing(abs(t))
    t = fabs(t);
    return __dsub_rn(nextafter(t, __longlong_as_double(0x7ff0000000000000LL)), t);
}
// tdir*t: the time in integration order (t forward, -t backward, both exact), so that one set of comparisons and one
// bracket serve both directions.  Without SPANS every solve is forward and this is t itself.
template <bool SPANS> __device__ __forceinline__ double ev_key(bool fwd, double t) {
    if constexpr (SPANS) return fwd ? t : -t;
    else return t;
}
// the crossing of event j inside the step, g(t0) = vL and g(tnew) = vR of opposite signs: Illinois regula falsi on the
// interpolant over [tL, tR] = [t0, tnew] in integration order, so tR < tL backward (DESIGN.md section 11).  The backward
// locator is the forward one mirrored (t -> -t gives te bit for bit up to sign).  Returns te; g at p(te) is 0 or has vR's
// sign.
template <bool SPANS>
__device__ double ev_locate(const EvStep& q, bool fwd, int kind, double level, double f, double gH, double vL, double vR) {
    if (vR == 0.0) return q.tnew;
    double tL = q.t0, tR = q.tnew, gL = vL, gR = vR;
    const double tol = __dmul_rn(128.0, fmax(spacing(tL), spacing(tR))), half = __dmul_rn(0.5, tol);
    int moved = 0;                                               // the end that moved last: -1 left, +1 right
    // the forward bracket on tdir*t: tdir*(tR - tL) > tol, and tm kept half inside both ends
    for (int it = 0; it < 64 && __dsub_rn(ev_key<SPANS>(fwd, tR), ev_key<SPANS>(fwd, tL)) > tol; it++) {
        double tm = __dsub_rn(tR, __dmul_rn(gR, __ddiv_rn(__dsub_rn(tR, tL), __dsub_rn(gR, gL))));
        tm = ev_key<SPANS>(fwd, py_min(py_max(ev_key<SPANS>(fwd, tm), __dadd_rn(ev_key<SPANS>(fwd, tL), half)),
                                       __dsub_rn(ev_key<SPANS>(fwd, tR), half)));
        double v[4];
        ev_point(q, tm, v);
        const double gm = ev_g(kind, level, f, gH, v);
        if (gm == 0.0) { tR = tm; break; }
        if ((gm < 0.0) == (gL < 0.0)) {                          // the sign changes across [tm, tR]
            tL = tm; gL = gm;
            if (moved < 0) gR = __dmul_rn(0.5, gR);
            moved = -1;
        } else {                                                 // across [tL, tm]
            tR = tm; gR = gm;
            if (moved > 0) gL = __dmul_rn(0.5, gL);
            moved = 1;
        }
    }
    return tR;
}
// after packet i's accepted step (c.t = tnew): detect, locate and record its events in order of encounter (ascending
// tdir*te, then ie).  Returns true on a terminal stop, with its time and state in tstop / ystop; records after tstop are
// not kept.  SPANS: the direction is the packet's own c.tdir, else forward.
template <bool SPANS>
__device__ __forceinline__ bool pkt_events(const Bs23Args& a, long long i, const Ode23Ctl& c, const Ode23Ev& ev, double& tstop,
                                           double ystop[4]) {
    const long long n = a.n;
    const bool fwd = c.tdir > 0.0;
    EvStep q;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        q.y[k] = a.y[k][i]; q.yn[k] = a.yt[k][i];
#pragma unroll
        for (int j = 0; j < 4; j++) q.f[j][k] = a.f[j][k][i];
    }
    q.t0 = c.t_acc; q.h = c.h_acc; q.tnew = c.t;
    double te[kMaxEvents];
    unsigned fired = 0;
    bool stop = false;
#pragma unroll
    for (int j = 0; j < kMaxEvents; j++) {
        te[j] = 0.0;
        if (j >= ev.nev) continue;
        const double vL = ev.vl[j * n + i], vR = ev_g(ev.kind[j], ev.level[j], ev.f, ev.gH, q.yn);
        ev.vl[j * n + i] = vR;
        // vL != 0, no NaN, a sign change the direction allows (a zero at the left end is never an event)
        if ((vL < 0.0 && vR >= 0.0 && ev.dir[j] >= 0) || (vL > 0.0 && vR <= 0.0 && ev.dir[j] <= 0)) {
            te[j] = ev_locate<SPANS>(q, fwd, ev.kind[j], ev.level[j], ev.f, ev.gH, vL, vR);
            fired |= 1u << j;
            if (ev.term[j] && (!stop || ev_key<SPANS>(fwd, te[j]) < ev_key<SPANS>(fwd, tstop))) {
                tstop = te[j];
                stop = true;
            }
        }
    }
    if (!fired) return false;
#pragma unroll
    for (int j = 0; j < kMaxEvents; j++)
        if (stop && ev_key<SPANS>(fwd, te[j]) > ev_key<SPANS>(fwd, tstop)) fired &= ~(1u << j);
    int cnt = ev.ne[i];
    while (fired) {                                              // the first encountered (te, j) first
        int jm = -1;
        double tm = 0.0;
#pragma unroll
        for (int j = 0; j < kMaxEvents; j++)
            if (((fired >> j) & 1u) && (jm < 0 || ev_key<SPANS>(fwd, te[j]) < ev_key<SPANS>(fwd, tm))) {
                jm = j;
                tm = te[j];
            }
        fired &= ~(1u << jm);
        if (cnt < ev.cap) {
            double v[4];
            ev_point(q, tm, v);
            const long long r = (long long)cnt * n + i;
            ev.te[r] = tm; ev.ie[r] = jm + 1;
#pragma unroll
            for (int k = 0; k < 4; k++) ev.ye[((long long)cnt * 4 + k) * n + i] = v[k];
        }
        cnt++;
    }
    ev.ne[i] = cnt;
    if (stop) ev_point(q, tstop, ystop);
    return stop;
}

// swrt_ode23_packets_tspans: packet i's per-solve constants from its own tspan row, in ode23_consts' operation order (so
// bit for bit what the host forms for that row), kept in sp's arrays for the decide kernel
__device__ __forceinline__ void pkt_span_consts(const Ode23Spans& sp, long long i, Ode23Ctl& c) {
    const double* row = sp.tsp + i * sp.ntspan;
    const double t0 = row[0], tfinal = row[sp.ntspan - 1];
    c.tfinal = tfinal;
    c.tdir = tfinal >= t0 ? 1.0 : -1.0;
    const double span = fabs(__dsub_rn(tfinal, t0)), span10 = fabs(__dmul_rn(0.1, __dsub_rn(tfinal, t0)));
    c.hmax = span10 < span ? span10 : span;
    c.htspan = fabs(__dsub_rn(row[1], row[0]));
    c.t = t0;
    sp.tfinal[i] = c.tfinal; sp.hmax[i] = c.hmax; sp.tdir[i] = c.tdir;
}

// swrt_ode23_packets_tspans, before f1: the shard's tspan columns (col[j*n + i], as uploaded) laid out packet-contiguous in
// rows, every packet's alpha of its t0 into s.al[0] for the per-packet evaluation of f1, and no packet idle
__global__ void ode23_pkt_rows_kernel(long long n, int ntspan, const double* __restrict__ col, double* __restrict__ rows,
                                      Ode23Pkt s, double tmax) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int j = 0; j < ntspan; j++) rows[i * ntspan + j] = col[j * n + i];
    s.al[0][i] = tmax != 0.0 ? __ddiv_rn(col[i], tmax) : 0.0;
    s.flags[i] = 0;
}

template <bool EV, bool SPANS>
__global__ void ode23_pkt_begin_kernel(Bs23Args a, Ode23Pkt s, Ode23Ctl c, double thr, Ode23Ev ev, Ode23Spans sp) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    if constexpr (SPANS) pkt_span_consts(sp, i, c);
    ode23_init(c, pkt_norm(a, i, 1, thr));
    pkt_store(s, i, a.n, c);
    if constexpr (EV) {                                         // g_j(y0), and no records yet
        const long long n = a.n;
        const double v[4] = {a.y[0][i], a.y[1][i], a.y[2][i], a.y[3][i]};
#pragma unroll
        for (int j = 0; j < kMaxEvents; j++)
            if (j < ev.nev) ev.vl[j * n + i] = ev_g(ev.kind[j], ev.level[j], ev.f, ev.gH, v);
        const double nan = __longlong_as_double(0xffffffffffffffffLL);
        for (int r = 0; r < ev.cap; r++) {
            ev.te[(long long)r * n + i] = nan; ev.ie[(long long)r * n + i] = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) ev.ye[((long long)r * 4 + k) * n + i] = nan;
        }
        ev.ne[i] = 0;
    }
}
// after a round's three stages: each unfinished packet's norm, its controller, its dense rows and its predicated accept.
// Block-reduced into the report pair of this round: the packets still unfinished and the attempts the slowest of them
// needs; the other pair is cleared for the next round.  EV: the accepted step's events; a terminal one stops the packet
// at its te (status 2) with that record's state, and only the dense rows up to te are written.  SPANS: the packet's own
// tfinal, hmax, tdir and tspan row; with EV the events follow that packet's direction.
template <bool EV, bool SPANS>
__global__ void __launch_bounds__(256) ode23_pkt_decide_kernel(Bs23Args a, Ode23Pkt s, Ode23Ctl c, double thr, int round, Ode23Ev ev,
                                                               Ode23Spans sp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int open = 0, batch = 0;
    if (i < a.n && !ode23_pkt_idle(s, i)) {
        pkt_load(s, i, a.n, c);
        if constexpr (SPANS) {
            c.tfinal = sp.tfinal[i]; c.hmax = sp.hmax[i]; c.tdir = sp.tdir[i];
            c.tspan = sp.tsp + i * sp.ntspan;
        }
        ode23_control(c, pkt_norm(a, i, 0, thr));
        if (c.accepted) {
            bool stop = false;
            double tstop = 0.0, ystop[4];
            if constexpr (EV) {
                stop = pkt_events<SPANS>(a, i, c, ev, tstop, ystop);
                if (stop && c.ntspan > 2)
                    while (c.nxt_end > c.nxt &&
                           ev_key<SPANS>(c.tdir > 0.0, c.tspan[c.nxt_end - 1]) > ev_key<SPANS>(c.tdir > 0.0, tstop))
                        c.nxt_end--;
            }
            if (c.ntspan > 2) bs23_rows_at(a, i, c);
            bs23_accept_at(a, i);
            if (stop) {
#pragma unroll
                for (int k = 0; k < 4; k++) a.y[k][i] = ystop[k];
                c.t = tstop;
                c.status = 2;
            }
        }
        pkt_store(s, i, a.n, c);
        if (!c.done && !c.status) { open = 1; batch = ode23_batch_estimate(c.tfinal, c.t, c.absh, c.hmax); }
    }
    __shared__ int sh_open[8], sh_batch[8];
    for (int o = 16; o > 0; o >>= 1) {
        open += __shfl_xor_sync(0xffffffffu, open, o);
        batch = max(batch, __shfl_xor_sync(0xffffffffu, batch, o));
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { sh_open[w] = open; sh_batch[w] = batch; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 1; q < 8; q++) { open += sh_open[q]; batch = max(batch, sh_batch[q]); }
        int* rep = s.report + 2 * (round & 1);
        if (open) { atomicAdd(rep, open); atomicMax(rep + 1, batch); }
        if (blockIdx.x == 0) { int* nxt = s.report + 2 * ((round + 1) & 1); nxt[0] = 0; nxt[1] = 0; }
    }
}
}  // namespace

// x^p with p = 1/3 rounded to double, correctly rounded (ties aside), which is what glibc's pow returns in all but
// vanishingly rare cases: CUDA's pow (2 ulp) gives the candidates, and the one whose cube lies nearest to x^(3p) in
// double-double arithmetic wins.  3p = 1 - 2^-54 exactly, so x^(3p) = x - 2^-54 x ln(x) to far below an ulp.
__host__ __device__ double pow_third(double x) {
    const double r = pow(x, 1.0 / 3.0);
    if (!(x > 0.0) || !isfinite(x) || !isfinite(r) || r == 0.0) return r;
    const double Xl = -(x * log(x)) * 0x1p-54;
    double c = nextafter(nextafter(r, 0.0), 0.0), best = r, bestd = -1.0;
    for (int q = 0; q < 5; q++, c = nextafter(c, 2.0 * c)) {
        const double c2 = c * c, c2l = fma(c, c, -c2);
        const double c3 = c2 * c, c3l = fma(c2, c, -c3) + c2l * c;
        const double d = fabs((c3 - x) + (c3l - Xl));          // c3 - x is exact (Sterbenz)
        if (bestd < 0.0 || d < bestd) { bestd = d; best = c; }
    }
    return best;
}

void launch_bs23_interp(const Bs23Args& a, const double w[4], double* const out[4], cudaStream_t st) {
    Bs23Interp q;
    for (int j = 0; j < 4; j++) { q.w[j] = w[j]; q.out[j] = out[j]; }
    if (a.n > 0) bs23_interp_kernel<<<nblk(a.n, 256), 256, 0, st>>>(a, q);
}
template <class View> void launch_bs23_stage(const Bs23Args& a, const View& v, int stage, cudaStream_t st) {
    if (a.n > 0) bs23_stage_kernel<<<nblk(a.n, 256), 256, 0, st>>>(a, v, stage);
}
template <int MODE, class View>
void launch_bs23_norm(const Bs23Args& a, const View& v, double thr, unsigned long long* out, cudaStream_t st) {
    if (a.n <= 0) return;
    unsigned nb = nblk(a.n, 256 * 4);
    if (nb > 148 * 8) nb = 148 * 8;
    bs23_norm_kernel<MODE><<<nb, 256, 0, st>>>(a, v, thr, out);
}
template <class View> void launch_bs23_accept(const Bs23Args& a, const View& v, cudaStream_t st) {
    if (a.n > 0) bs23_accept_kernel<<<nblk(a.n, 256), 256, 0, st>>>(a, v);
}
template <class View>
void launch_rhs(const View& v, int stage, long long n, const double* k, const double* l, const double* const* e6,
                const double* const* e1, double f, double gH, double cgfac, double* const fj[4], cudaStream_t st) {
    E6 e, e2;
    for (int i = 0; i < 6; i++) { e.p[i] = e6[i]; e2.p[i] = e1 ? e1[i] : nullptr; }
    if (n > 0) rhs_kernel<<<nblk(n, 256), 256, 0, st>>>(v, stage, n, k, l, e, e2, e1 != nullptr, f, gH, cgfac, fj[0], fj[1], fj[2], fj[3]);
}
template void launch_bs23_stage(const Bs23Args&, const Ode23ValView&, int, cudaStream_t);
template void launch_bs23_stage(const Bs23Args&, const Ode23CtlView&, int, cudaStream_t);
template void launch_bs23_stage(const Bs23Args&, const Ode23PktView&, int, cudaStream_t);
template void launch_bs23_norm<0>(const Bs23Args&, const Ode23ValView&, double, unsigned long long*, cudaStream_t);
template void launch_bs23_norm<1>(const Bs23Args&, const Ode23ValView&, double, unsigned long long*, cudaStream_t);
template void launch_bs23_norm<0>(const Bs23Args&, const Ode23CtlView&, double, unsigned long long*, cudaStream_t);
template void launch_bs23_accept(const Bs23Args&, const Ode23ValView&, cudaStream_t);
template void launch_bs23_accept(const Bs23Args&, const Ode23CtlView&, cudaStream_t);
template void launch_rhs(const Ode23ValView&, int, long long, const double*, const double*, const double* const*, const double* const*,
                         double, double, double, double* const[4], cudaStream_t);
template void launch_rhs(const Ode23CtlView&, int, long long, const double*, const double*, const double* const*, const double* const*,
                         double, double, double, double* const[4], cudaStream_t);
template void launch_rhs(const Ode23PktView&, int, long long, const double*, const double*, const double* const*, const double* const*,
                         double, double, double, double* const[4], cudaStream_t);
void launch_ode23_init(Ode23Ctl* ctl, unsigned long long* norm, cudaStream_t st) { ode23_init_kernel<<<1, 1, 0, st>>>(ctl, norm); }
void launch_ode23_control(Ode23Ctl* ctl, unsigned long long* norm, cudaStream_t st) { ode23_control_kernel<<<1, 1, 0, st>>>(ctl, norm); }
void launch_bs23_interp_dev(const Bs23Args& a, const Ode23Ctl* ctl, cudaStream_t st) {
    if (a.n > 0) bs23_interp_dev_kernel<<<nblk(a.n, 256), 256, 0, st>>>(a, ctl);
}

void launch_ode23_pkt_rows(long long n, int ntspan, const double* col, double* rows, const Ode23Pkt& s, double tmax,
                           cudaStream_t st) {
    if (n > 0) ode23_pkt_rows_kernel<<<nblk(n, 256), 256, 0, st>>>(n, ntspan, col, rows, s, tmax);
}
void launch_ode23_pkt_begin(const Bs23Args& a, const Ode23Pkt& s, const Ode23Ctl& k, double thr, const Ode23Ev* ev,
                            const Ode23Spans* sp, cudaStream_t st) {
    if (a.n <= 0) return;
    const unsigned nb = nblk(a.n, 256);
    if (ev && sp) ode23_pkt_begin_kernel<true, true><<<nb, 256, 0, st>>>(a, s, k, thr, *ev, *sp);
    else if (ev) ode23_pkt_begin_kernel<true, false><<<nb, 256, 0, st>>>(a, s, k, thr, *ev, Ode23Spans{});
    else if (sp) ode23_pkt_begin_kernel<false, true><<<nb, 256, 0, st>>>(a, s, k, thr, Ode23Ev{}, *sp);
    else ode23_pkt_begin_kernel<false, false><<<nb, 256, 0, st>>>(a, s, k, thr, Ode23Ev{}, Ode23Spans{});
}
void launch_ode23_pkt_decide(const Bs23Args& a, const Ode23Pkt& s, const Ode23Ctl& k, double thr, int round, const Ode23Ev* ev,
                             const Ode23Spans* sp, cudaStream_t st) {
    if (a.n <= 0) return;
    const unsigned nb = nblk(a.n, 256);
    if (ev && sp) ode23_pkt_decide_kernel<true, true><<<nb, 256, 0, st>>>(a, s, k, thr, round, *ev, *sp);
    else if (ev) ode23_pkt_decide_kernel<true, false><<<nb, 256, 0, st>>>(a, s, k, thr, round, *ev, Ode23Spans{});
    else if (sp) ode23_pkt_decide_kernel<false, true><<<nb, 256, 0, st>>>(a, s, k, thr, round, Ode23Ev{}, *sp);
    else ode23_pkt_decide_kernel<false, false><<<nb, 256, 0, st>>>(a, s, k, thr, round, Ode23Ev{}, Ode23Spans{});
}

void launch_fill(double* p, double v, long long n, cudaStream_t st) {
    if (n > 0) fill_kernel<<<nblk(n, 256), 256, 0, st>>>(p, v, n);
}
void launch_omega(long long n, const double* k, const double* l, const double* u, const double* v, double f, double gH,
                  double* omega, double* Omega_abs, cudaStream_t st) {
    if (n > 0) omega_kernel<<<nblk(n, 256), 256, 0, st>>>(n, k, l, u, v, f, gH, omega, Omega_abs);
}
void launch_rk4_stage(const Rk4Args& a, cudaStream_t st) {
    if (a.n > 0) rk4_stage_kernel<<<nblk(a.n, 256), 256, 0, st>>>(a);
}
void launch_rk4_final(const Rk4Args& a, cudaStream_t st) {
    if (a.n > 0) rk4_final_kernel<<<nblk(a.n, 256), 256, 0, st>>>(a);
}
void launch_hist(long long n, const double* w, const double* edges_dev, int nedges, unsigned long long* counts_dev,
                 cudaStream_t st) {
    if (n <= 0) return;
    size_t smem = (size_t)nedges * 8 + (size_t)(nedges - 1) * 4;
    unsigned nb = nblk(n, 256 * 8);
    if (nb > 148 * 8) nb = 148 * 8;
    hist_kernel<<<nb, 256, smem, st>>>(n, w, edges_dev, nedges, counts_dev);
}
void launch_ideal_hist(long long npts, const double* u, const double* v, const double* kvx, const double* kvy, int nang,
                       double omega0, const double* edges_dev, int nedges, unsigned long long* counts_dev, cudaStream_t st) {
    if (npts <= 0) return;
    size_t smem = (size_t)nedges * 8 + (size_t)2 * nang * 8 + (size_t)(nedges - 1) * 4;
    unsigned nb = nblk(npts, 256);
    if (nb > 148 * 8) nb = 148 * 8;
    ideal_hist_kernel<<<nb, 256, smem, st>>>(npts, u, v, kvx, kvy, nang, omega0, edges_dev, nedges, counts_dev);
}
void launch_packet_quantity(long long n, int q, const PktQ& p, double* out, cudaStream_t st) {
    if (n > 0) packet_quantity_kernel<<<nblk(n, 256), 256, 0, st>>>(n, q, p, out);
}
cudaError_t launch_hist2(long long n, int qx, int qy, const PktQ& p, const double* edges_dev, int nxe, int nye,
                         unsigned long long* counts_dev, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    int dev = 0, optin = 0, nsm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    // the path is chosen by size alone: private counters when they fit beside the edges
    const size_t edge_bytes = (size_t)(nxe + nye) * 8;
    const size_t smem_path = edge_bytes + (size_t)(nxe - 1) * (nye - 1) * 4;
    const bool smem = smem_path <= (size_t)optin;
    const size_t bytes = smem ? smem_path : edge_bytes;
    auto kern = smem ? hist2_kernel<true> : hist2_kernel<false>;
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes)) != cudaSuccess) return e;
    // 1024 threads: the shared-memory path fits one CTA an SM, and the kernel is bound by latency, not bandwidth
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 1024, bytes)) != cudaSuccess) return e;
    // one wave of CTAs: each pays for zeroing and flushing its counters once
    unsigned nb = (unsigned)(per_sm > 0 ? per_sm : 1) * (unsigned)nsm;
    if (nb > nblk(n, 1024)) nb = nblk(n, 1024);
    kern<<<nb, 1024, bytes, st>>>(n, qx, qy, p, edges_dev, nxe, nye, counts_dev);
    return cudaGetLastError();
}
void launch_weight_scale(long long n, const WeightKinds& w, const PktQ& p, const double* a, int* exp_dev, cudaStream_t st) {
    if (n <= 0) return;
    unsigned nb = nblk(n, 256);
    if (nb > 148 * 8) nb = 148 * 8;
    weight_scale_kernel<<<nb, 256, 0, st>>>(n, w, p, a, exp_dev);
}
cudaError_t launch_hist2_sums(long long n, int qx, int qy, const PktQ& p, const double* a, const WeightKinds& w,
                              const int* exp_dev, const double* edges_dev, int nxe, int nye, long long* acc_dev,
                              unsigned long long* counts_dev, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    int dev = 0, nsm = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    // global counters only: the digits and non-finite count take 32 bytes per (bin, kind), so a private copy per CTA fits
    // shared memory only below ~7,000 bin-kinds, smaller than the spectra people plot
    const size_t bytes = (size_t)(nxe + nye) * 8;
    if ((e = cudaFuncSetAttribute(hist2_sums_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes)) != cudaSuccess) return e;
    int per_sm = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hist2_sums_kernel, 1024, bytes)) != cudaSuccess) return e;
    unsigned nb = (unsigned)(per_sm > 0 ? per_sm : 1) * (unsigned)nsm;
    if (nb > nblk(n, 1024)) nb = nblk(n, 1024);
    hist2_sums_kernel<<<nb, 1024, bytes, st>>>(n, qx, qy, p, a, w, exp_dev, edges_dev, nxe, nye, acc_dev, counts_dev);
    return cudaGetLastError();
}
void launch_diag(long long n, const double* x, const double* y, const double* k, const double* l, const double* a,
                 const double* omega, const double* Omega_abs, double* out8_dev, cudaStream_t st) {
    // out8_dev must have room for 8 + kDiagBlocks*8 doubles: results first, partials after
    double* part = out8_dev + 8;
    diag_partial_kernel<<<kDiagBlocks, 256, 0, st>>>(n, x, y, k, l, a, omega, Omega_abs, part);
    diag_final_kernel<<<1, 32, 0, st>>>(kDiagBlocks, part, n, out8_dev);
}


// ---------------------------------------------------------------------------------------------
// Gather-rate probe (the roofline denominator of the LAGRANGE6 / NUFFT modes).  Those kernels are bound by scattered
// reads of an L2-resident table through L1TEX, not by HBM: this kernel measures the rate the chip sustains for that access
// shape with nothing else in the way -- a quad of lanes reads one 64-byte segment (four 16-byte nodes) at a
// pseudo-random table offset, eight independent loads in flight per lane, table far larger than L1 and smaller than L2.
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) gather_probe_kernel(const double2* __restrict__ table, unsigned nseg_mask, int iters, double* __restrict__ sink) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned quad = t >> 2, q = t & 3;
    unsigned state = quad * 2654435761u + 12345u;
    double acc = 0.0;
    for (int it = 0; it < iters; it++) {
        double2 v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            state = state * 1664525u + 1013904223u;                 // one segment per quad per load: all four lanes agree
            const unsigned seg = (state >> 7) & nseg_mask;
            v[u] = __ldg(table + (size_t)seg * 4 + q);
        }
#pragma unroll
        for (int u = 0; u < 8; u++) acc += v[u].x + v[u].y;
    }
    if (acc == 123.456) sink[0] = acc;                              // keeps the loads alive
}
}  // namespace

// useful bytes gathered per second (GB/s) from a table of `table_bytes` (power of two); <0 on error
double gather_probe(size_t table_bytes, int iters, int reps, cudaStream_t st) {
    double2* table = nullptr; double* sink = nullptr;
    if (cudaMalloc(&table, table_bytes) != cudaSuccess || cudaMalloc(&sink, 8) != cudaSuccess) { cudaFree(table); return -1.0; }
    cudaMemsetAsync(table, 0, table_bytes, st);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const unsigned nseg = (unsigned)(table_bytes / 64);
    const int blocks = 148 * 8;
    gather_probe_kernel<<<blocks, 256, 0, st>>>(table, nseg - 1, iters, sink);      // warm-up (table into L2)
    double best = -1.0;
    for (int r = 0; r < reps; r++) {
        cudaEventRecord(e0, st);
        gather_probe_kernel<<<blocks, 256, 0, st>>>(table, nseg - 1, iters, sink);
        cudaEventRecord(e1, st);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double gbs = (double)blocks * 256 * iters * 8 * 16 / (ms * 1e-3) * 1e-9;
        if (gbs > best) best = gbs;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(table); cudaFree(sink);
    return cudaGetLastError() == cudaSuccess ? best : -1.0;
}

}  // namespace swrt
