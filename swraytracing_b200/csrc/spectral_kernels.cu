// spectral_kernels.cu -- SPECTRAL mode of libswrt: evaluate the flow planes at every packet by the
// exact Fourier-series sum, as a dense real-embedded complex contraction on the fp64 tensor pipe
// (DMMA m8n8k4), fused with the leapfrog stepper of ode_symplectic.m:13-21,33-37.
//
//   F_c(p) = sum_ky w_ky Re[ e^{i ky ty_p} * G_c(p,ky) ],   G_c(p,ky) = sum_kx C_c(kx,ky) e^{i kx tx_p}
//
// Stage 1 (G) is the GEMM:  M = packets, K = kx, N = (plane, ky).  The +kx / -kx halves are folded
// at pack time (S = C(+kx)+C(-kx), D = C(+kx)-C(-kx)), so K runs over kx >= 0 only:
//       Gr += Er*Sr - Ei*Di ,   Gi += Er*Si + Ei*Dr          (E = e^{i kx tx})
// which is the real GEMM  [Er Ei] (P x 2K)  x  [[Sr Si],[-Di Dr]] (2K x 2N).  A (the twiddles) is
// generated in registers by rotation recurrence; B (the packed stack) streams L2 -> shared memory
// with cp.async.bulk + mbarrier from one producer warp; stage 2 (the ky sum) is applied to the
// accumulator fragments in registers, followed by a quad shuffle reduction.
//
// Reference behaviour replaced: SpectralScheme.U / grad_U (SpectralScheme.m:45-68) + interpolate
// (interpolate.m:12-49) evaluated spectrally, and ode_symplectic's stage loop.
#include "swrt_internal.h"
#include "spectral_common.cuh"
#include <cstdio>
#include <cstdlib>
#include <cmath>

namespace swrt {

// ------------------------------------------------------------------------------------------------
// pack / setup kernels
// ------------------------------------------------------------------------------------------------
struct PlanePtrs { const double2* p[kNumSrcPlanes]; };

__device__ __forceinline__ double2 load_coef(const double2* pl, int kx, int ky, int kmax, int nkx) {
    // half-plane value with the ky=0 conjugate symmetrisation of fulspec.m:16 applied
    if (ky == 0) {
        if (kx < 0) { double2 v = pl[(-kx + kmax)]; v.y = -v.y; return v; }
        double2 v = pl[kx + kmax];
        if (kx == 0) v.y = 0.0;
        return v;
    }
    return pl[(size_t)ky * nkx + (kx + kmax)];
}

__global__ void pack_kernel(PackGeom g, PlanePtrs src, double* __restrict__ stack) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= g.total_doubles) return;
    int which = idx & 1;
    int lane = (idx >> 1) & 31;
    size_t rest = idx >> 6;
    int half_nt = g.NT / 2;
    int tp = rest % half_nt; rest /= half_nt;
    int s = rest % g.ksteps;
    int pass = rest / g.ksteps;
    int t = 2 * tp + which;
    int c = t / g.G, gg = t % g.G;
    int krow = lane & 3, ncol = lane >> 2;
    int kx = 2 * s + (krow >> 1), part_k = krow & 1;
    int j = ncol >> 1, part_n = ncol & 1;
    int ky = pass * 4 * g.G + 4 * gg + j;
    double val = 0.0;
    if (kx <= g.kmax && ky <= g.kmax) {
        const double2* pl = src.p[g.plane_ids[c]];
        double2 cp = load_coef(pl, kx, ky, g.kmax, g.nkx);
        double2 cm = make_double2(0.0, 0.0);
        double2 S, D;
        if (kx == 0) { S = cp; D = make_double2(0.0, 0.0); }
        else {
            cm = load_coef(pl, -kx, ky, g.kmax, g.nkx);
            S = make_double2(cp.x + cm.x, cp.y + cm.y);
            D = make_double2(cp.x - cm.x, cp.y - cm.y);
        }
        double w = (ky == 0) ? 1.0 : 2.0;
        if (part_k == 0) val = part_n == 0 ? S.x : S.y;
        else             val = part_n == 0 ? -D.y : D.x;
        val *= w;
    }
    stack[idx] = val;
}

void launch_pack(const PackGeom& g, const double2* const* planes_dev, double* stack_dev, cudaStream_t st) {
    PlanePtrs pp;
    for (int i = 0; i < kNumSrcPlanes; i++) pp.p[i] = planes_dev[i];
    size_t n = g.total_doubles;
    int bs = 256;
    pack_kernel<<<(unsigned)((n + bs - 1) / bs), bs, 0, st>>>(g, pp, stack_dev);
}

struct PlaneOut { double2* p[6]; };
// SpectralScheme.m:18-25 / grid_U.m:3-9 on the device: six planes from psi-hat.
__global__ void psi_to_planes_kernel(const double2* __restrict__ psik, PlaneOut out, int nkx, int nky,
                                     double kappa, double u_mean) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nkx * nky) return;
    int kmax = (nkx - 1) / 2;
    double kx = kappa * (double)((idx % nkx) - kmax);
    double ky = kappa * (double)(idx / nkx);
    double2 psi = psik[idx];
    // u = -i ky psi ; v = i kx psi
    double2 u = make_double2(ky * psi.y, -ky * psi.x);
    double2 v = make_double2(-kx * psi.y, kx * psi.x);
    // ux = i kx u, uy = i ky u, vx = i kx v, vy = i ky v
    double2 ux = make_double2(-kx * u.y, kx * u.x);
    double2 uy = make_double2(-ky * u.y, ky * u.x);
    double2 vx = make_double2(-kx * v.y, kx * v.x);
    double2 vy = make_double2(-ky * v.y, ky * v.x);
    if (idx == kmax) u.x += u_mean;   // (kx,ky) = (0,0): mean shear, grid_U.m:11
    out.p[0][idx] = u; out.p[1][idx] = v; out.p[2][idx] = ux; out.p[3][idx] = uy; out.p[4][idx] = vx; out.p[5][idx] = vy;
}

// psi-hat moment planes (spectra of REAL fields, so the ky = 0 symmetrisation of fulspec.m:16 applies):
//   N0 = psi, N1 = i kx psi, N2 = -kx^2 psi   with INTEGER kx
__global__ void psi_moments_kernel(const double2* __restrict__ psik, double2* n0, double2* n1, double2* n2, int nkx, int nky) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nkx * nky) return;
    const int kmax = (nkx - 1) / 2;
    const double kx = (double)((idx % nkx) - kmax);
    const double2 psi = psik[idx];
    n0[idx] = psi;
    n1[idx] = make_double2(-kx * psi.y, kx * psi.x);
    n2[idx] = make_double2(-kx * kx * psi.x, -kx * kx * psi.y);
}
void launch_psi_moments(const double2* psik, double2* n0, double2* n1, double2* n2, int nkx, int nky, cudaStream_t st) {
    int n = nkx * nky;
    psi_moments_kernel<<<(n + 255) / 256, 256, 0, st>>>(psik, n0, n1, n2, nkx, nky);
}

void launch_psi_to_planes(const double2* psik, double2* const* planes, int nkx, int nky, double kappa,
                          double u_mean, cudaStream_t st) {
    PlaneOut po;
    for (int i = 0; i < 6; i++) po.p[i] = planes[i];
    int n = nkx * nky;
    psi_to_planes_kernel<<<(n + 255) / 256, 256, 0, st>>>(psik, po, nkx, nky, kappa, u_mean);
}

// out = wa*a + wb*b : the on-device frame blend of interpolate_U.m:19-23 applied to the
// coefficient stack (linear, so identical to blending the evaluated fields).
// (the expression is pinned -- one rounded product, one fma -- so that the single blend and the multi-blend kernel below
// produce the same doubles: a fused run of m time-dependent steps equals m single-step launches bit for bit)
__global__ void axpby_kernel(double* __restrict__ out, const double* __restrict__ a, const double* __restrict__ b,
                             double wa, double wb, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = fma(wa, a[i], __dmul_rn(wb, b[i]));
}
// out[j][i] = (1 - al_j)*a[i] + al_j*b[i] for the m steps of a fused run, al_j = alpha0 + (j0 + j)*dalpha (the host's
// expression for step j0 + j of swrt_step): every operand is read once for all m blends
__global__ void axpby_multi_kernel(double* __restrict__ out, const double* __restrict__ a, const double* __restrict__ b,
                                   double alpha0, double dalpha, int j0, int m, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const double av = a[i], bv = b[i];
        for (int j = 0; j < m; j++) {
            const double al = __dadd_rn(alpha0, __dmul_rn((double)(j0 + j), dalpha));      // un-fused: the host's alpha0 + j*dalpha
            out[(size_t)j * n + i] = fma(__dsub_rn(1.0, al), av, __dmul_rn(al, bv));
        }
    }
}
void launch_axpby_multi(double* out, const double* a, const double* b, double alpha0, double dalpha, int j0, int m, size_t n,
                        cudaStream_t st) {
    int bs = 256;
    size_t nb = (n + bs - 1) / bs;
    if (nb > 148 * 16) nb = 148 * 16;
    axpby_multi_kernel<<<(unsigned)nb, bs, 0, st>>>(out, a, b, alpha0, dalpha, j0, m, n);
}
// the blend above at the ode23 controller's alpha (weights 1 - al, al as the host forms them); alpha 0 and 1 read a frame
// directly (as active_stack does), so nothing is blended then, nor once the solve is done
__global__ void axpby_dev_kernel(double* __restrict__ out, const double* __restrict__ a, const double* __restrict__ b,
                                 const Ode23Ctl* ctl, int stage, size_t n) {
    if (ode23_idle(ctl)) return;
    const double al = ctl->al[stage];
    if (al == 0.0 || al == 1.0) return;
    const double wa = __dsub_rn(1.0, al);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = fma(wa, a[i], __dmul_rn(al, b[i]));
}
void launch_axpby_dev(double* out, const double* a, const double* b, const Ode23Ctl* ctl, int stage, size_t n, cudaStream_t st) {
    int bs = 256;
    size_t nb = (n + bs - 1) / bs;
    if (nb > 148 * 16) nb = 148 * 16;
    axpby_dev_kernel<<<(unsigned)nb, bs, 0, st>>>(out, a, b, ctl, stage, n);
}
void launch_axpby(double* out, const double* a, const double* b, double wa, double wb, size_t n, cudaStream_t st) {
    int bs = 256;
    size_t nb = (n + bs - 1) / bs;
    if (nb > 148 * 16) nb = 148 * 16;
    axpby_kernel<<<(unsigned)nb, bs, 0, st>>>(out, a, b, wa, wb, n);
}

PackGeom make_geom(int nx, int npl, const int* plane_ids, int mtiles, int twiddle_pref) {
    PackGeom g{};
    g.nx = nx; g.nkx = nx - 1; g.nky = nx / 2; g.kmax = nx / 2 - 1;
    g.npl = npl;
    // accumulator budget: MT * NT * 2 doubles per thread = 96..112 registers-pairs -> NT*MT ~ 24
    int nt_target = 24 / mtiles;
    int G = nt_target / npl; if (G < 1) G = 1;
    if ((npl * G) & 1) G += 1;            // NT must be even (n-tiles are fetched in pairs)
    // supported instantiations (see launch_spectral): keep in sync
    g.G = G; g.NT = npl * G;
    int kyp = 4 * G;
    g.npass = (g.nky + kyp - 1) / kyp;
    // ~48 KB chunks (kc k-steps of NT*256 bytes), kc a multiple of the k-loop unroll
    int kc0 = 192 / g.NT;
    kc0 = kc0 >= 16 ? 16 : (kc0 >= 8 ? 8 : 4);
    const int ks = (g.kmax + 1 + 1) / 2;
    auto layout = [&](int kc) {
        if (kc % kKUnroll) kc = ((kc + kKUnroll - 1) / kKUnroll) * kKUnroll;
        g.kc = kc;
        g.ksteps = ((ks + kc - 1) / kc) * kc;
        g.chunks_per_eval = g.npass * (g.ksteps / kc);
        g.chunk_doubles = (size_t)kc * g.NT * 32;
        g.total_doubles = (size_t)g.npass * g.ksteps * g.NT * 32;
    };
    // Twiddle table: one double per lane per k-step per warp (the A fragments of a whole step), written and read back
    // by the same lane.  With it the k-loop holds no fp64 instruction but the DMMAs (tools/dmma_lds_bench.cu: 36.3
    // against 34.9 TFLOP/s for the loop with the 4-DFMA rotation per k-step).  It needs ksteps * 2 KB of shared memory
    // next to a ring of at least three chunks: 48 KB chunks up to nx = 128, 24 KB chunks at nx = 256 (measured there:
    // 33.0 TFLOP/s rotating in registers with 48 KB chunks, 32.0 with 24 KB chunks, 33.7 with 24 KB chunks and the table);
    // larger grids rotate in registers.
    constexpr size_t kSmemBudget = 216 * 1024;
    auto atab_fits = [&]() { return (size_t)g.ksteps * 32 * 8 * kConsumerWarps + 3 * g.chunk_doubles * 8 <= kSmemBudget; };
    // twiddle_pref: 0 = automatic (shared-memory table when it fits beside a ring of full-size chunks, else the global / L2
    // table), 1 = rotate in registers, 2 = global table wherever a table is possible, 3 = shared-memory table even with
    // shrunk chunks (the round-1 layout at 256^2), else the global one.  Measured (profiles/README.md, TFLOP/s, rotation /
    // shared / global): 128^2 31.1 / 32.2 / 31.6; 256^2 32.9 / 33.9 (24 KB chunks) / 34.2; 512^2 33.4 / does not fit / 34.8.
    bool want_atab = mtiles == 1 && kCtasPerSm == 1 && twiddle_pref != 1 && twiddle_pref != 2;
    const bool want_global = mtiles == 1 && kCtasPerSm == 1 && twiddle_pref != 1;
    const bool shrink_for_table = twiddle_pref == 3;
    int kc_forced = 0;
#ifdef SWRT_DEV_TUNING      // developer experiments only: the shipped library reads no environment variables
    if (const char* e = getenv("SWRT_ATAB")) want_atab = want_atab && atoi(e) != 0;
    if (const char* e = getenv("SWRT_KC")) { kc_forced = atoi(e); if (kc_forced < kKUnroll) kc_forced = kKUnroll; }
#endif
    if (kc_forced) {
        layout(kc_forced);
        g.atab = want_atab && atab_fits();
    } else {
        layout(kc0);
        g.atab = want_atab && atab_fits();
        if (want_atab && !g.atab && kc0 > 4 && shrink_for_table) {
            layout(4);
            g.atab = atab_fits();
            if (!g.atab) layout(kc0);
        }
    }
    if (!g.atab && want_global) g.atab = 2;       // table in the per-CTA global scratch: full-size chunks, full-size ring
    const size_t chunk_bytes = g.chunk_doubles * 8;
    const size_t ring_budget = g.atab == 1 ? (kSmemBudget - (size_t)g.ksteps * 32 * 8 * kConsumerWarps) : (size_t)(200 * 1024 / kCtasPerSm);
    g.nstages = (int)(ring_budget / chunk_bytes);
    if (g.nstages > 8) g.nstages = 8;
    if (g.nstages < 3) g.nstages = 3;
    // Warps 4..7 (the second warp of every SM sub-partition) start ~1.5 chunks after warps 0..3, so
    // that one group's non-MMA phases (chunk hand-over, per-pass stage 2, per-step twiddle seeds)
    // run under the other group's DMMAs instead of leaving the fp64 pipe idle.  A stage is
    // refilled `lag` chunks after its issuing warp left it, which must exceed the skew.
    g.lag = g.nstages - 1;
    if (g.lag > 4) g.lag = 4;
    g.desync_ns = (int)((g.lag >= 3 ? 1.5 : 0.6) * g.kc * g.NT * 16 / 1.9);
#ifdef SWRT_DEV_TUNING
    if (const char* e = getenv("SWRT_LAG")) g.lag = atoi(e);
    if (const char* e = getenv("SWRT_DESYNC_NS")) g.desync_ns = atoi(e);
    if (const char* e = getenv("SWRT_NSTAGES")) { g.nstages = atoi(e); if (g.nstages < 2) g.nstages = 2; }
#endif
    if (g.lag >= g.nstages) g.lag = g.nstages - 1;
    if (g.lag < 1) g.lag = 1;
    for (int i = 0; i < kMaxPlanes; i++) g.plane_ids[i] = i < npl ? plane_ids[i] : 0;
    return g;
}

size_t spectral_smem_bytes(const PackGeom& g) {
    // ring | full/empty barriers (padded to 128 bytes) | twiddle table
    return (size_t)g.nstages * g.chunk_doubles * 8 + 128 + (g.atab == 1 ? (size_t)g.ksteps * 32 * 8 * kConsumerWarps : 0);
}

// ------------------------------------------------------------------------------------------------
// per-row epilogue pieces shared by the dense kernel and the anchored step kernel (same arithmetic in both)
// ------------------------------------------------------------------------------------------------
// stage 2 of one pass: F_c += Re[e^{i ky ty} G_c(ky)] for this lane's ky of every group, then advance the y twiddles
template <int NPL, int G, bool PSI, int NF>
__device__ __forceinline__ void stage2_pass(const double (&acc)[NPL * G][2], Cplx (&ytw)[G], const Cplx yrot, double& kyd,
                                            double (&F)[NF]) {
#pragma unroll
    for (int gg = 0; gg < G; gg++) {
        const double cy = ytw[gg].re, sy = ytw[gg].im;
        if constexpr (PSI) {
            const double ky = kyd + (double)(4 * gg);
            const double g0r = acc[0 * G + gg][0], g0i = acc[0 * G + gg][1];
            const double g1r = acc[1 * G + gg][0], g1i = acc[1 * G + gg][1];
            const double g2r = acc[2 * G + gg][0], g2i = acc[2 * G + gg][1];
            const double a0 = fma(g0r, cy, -g0i * sy), b0 = fma(g0i, cy, g0r * sy);
            const double a1 = fma(g1r, cy, -g1i * sy), b1 = fma(g1i, cy, g1r * sy);
            const double a2 = fma(g2r, cy, -g2i * sy);
            F[0] = fma(ky, b0, F[0]);          // u  / kap
            F[1] += a1;                        // v  / kap
            F[2] = fma(ky, b1, F[2]);          // ux / kap^2
            F[3] = fma(ky * ky, a0, F[3]);     // uy / kap^2
            F[4] += a2;                        // vx / kap^2
        } else {
#pragma unroll
            for (int c = 0; c < NPL; c++) {
                F[c] = fma(acc[c * G + gg][0], cy, F[c]);
                F[c] = fma(-acc[c * G + gg][1], sy, F[c]);
            }
        }
        ytw[gg] = cmul(ytw[gg], yrot);
    }
    kyd += (double)(4 * G);
}

// quad reduction (the 4 lanes of a quad hold 4 interleaved ky subsets) and, for psi-hat stacks, the six planes
template <bool PSI, int NPL, int NF, bool DEV = false>
__device__ __forceinline__ void finish_planes(double (&F)[NF], const SpecArgs& a, int ev) {
#pragma unroll
    for (int c = 0; c < (PSI ? 5 : NPL); c++) {
        double v = F[c];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        F[c] = v;
    }
    if constexpr (PSI) {
        const double kap = a.kappa, kap2 = a.kappa * a.kappa;
        // mean shear of the blended frame (grid_U.m:11; interpolate_U.m:19-23), every rounding pinned
        const double al = DEV ? a.sel.ctl->al[a.sel.stage] : __dadd_rn(a.alpha0, __dmul_rn((double)(a.j0 + ev), a.dalpha));
        const double um = __dadd_rn(__dmul_rn(__dsub_rn(1.0, al), a.u_mean0), __dmul_rn(al, a.u_mean1));
        F[0] = fma(kap, F[0], um);
        F[1] = kap * F[1];
        F[2] = kap2 * F[2];
        F[3] = kap2 * F[3];
        F[4] = kap2 * F[4];
        F[5] = -F[2];
    }
}

// phi2(dt): x += dt*U(x1); k -= dt*(grad U)^T k with the OLD k (ode_symplectic.m:18-21); then phi1(dt/2) with the new k
template <int NF>
__device__ __forceinline__ void leapfrog_kick(const double (&F)[NF], const SpecArgs& a, double& px, double& py, double& pk,
                                              double& pl, double& hcx, double& hcy) {
    const double u = F[0], v = F[1], ux = F[2], uy = F[3], vx = F[4], vy = F[5];
    px = px + a.dt * u;
    py = py + a.dt * v;
    const double k0 = pk, l0 = pl;
    pk = k0 - a.dt * (ux * k0 + vx * l0);
    pl = l0 - a.dt * (uy * k0 + vy * l0);
    // (explicit un-fused mul/add so that a fused run of n steps and n single-step
    // launches produce bit-identical states)
    half_drift(pk, pl, a.f2, a.gH, __dmul_rn(__dmul_rn(0.5, a.dt), a.gH), hcx, hcy);
    px = __dadd_rn(px, hcx);
    py = __dadd_rn(py, hcy);
}

// ------------------------------------------------------------------------------------------------
// the contraction kernel
// ------------------------------------------------------------------------------------------------
// PSI = true: the stack holds the three psi-hat moment planes N0 = psi, N1 = i kx psi, N2 = -kx^2 psi
// (integer kx); the six velocity/gradient planes of SpectralScheme.m:18-25 are assembled in stage 2:
//   u = kap ky Im[T G0], v = kap Re[T G1], ux = kap^2 ky Im[T G1], uy = kap^2 ky^2 Re[T G0],
//   vx = kap^2 Re[T G2], vy = -ux   (T = e^{i ky ty}),  which halves the DMMA work (6 nx^2 flops).
// ATAB: 0 = x twiddles rotated in registers inside the k-loop; 1 = tabulated once per step in shared memory; 2 = tabulated
// once per step in a per-CTA global scratch (L2-resident; grids whose table does not fit in shared memory), read back
// with plain loads one unrolled body ahead -- in both table forms the k-loop holds no fp64 instruction but the DMMAs.
template <int NPL, int G, int MT, int MODE, bool PSI, int ATAB>
__global__ void __launch_bounds__(kSpecThreads, kCtasPerSm) spectral_kernel(const SpecArgs a) {
    static_assert(!ATAB || MT == 1, "the twiddle table is laid out for one m-tile per warp");
    constexpr int NT = NPL * G;
    constexpr int NF = PSI ? 6 : NPL;          // planes produced per packet
    static_assert(!PSI || NPL == 3, "psi mode contracts exactly three moment planes");
    constexpr int HALF_NT = NT / 2;
    constexpr int TILE_P = kConsumerWarps * 8 * MT;
    static_assert(NT % 2 == 0, "n-tiles are fetched in pairs");

    extern __shared__ __align__(128) unsigned char smem_raw[];
    const PackGeom& g = a.g;
    const int nstages = g.nstages;
    const uint32_t chunk_bytes = (uint32_t)(g.chunk_doubles * 8);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_raw + (size_t)nstages * chunk_bytes);
    uint64_t* empty_bar = full_bar + nstages;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // this lane's column of the warp's twiddle table: sA[s * 32] = A element of k-step s (written and read by this lane only)
    double* sA;
    if constexpr (ATAB == 2) sA = a.twid + ((size_t)blockIdx.x * kConsumerWarps + warp) * g.ksteps * 32 + lane;
    else sA = reinterpret_cast<double*>(smem_raw + (size_t)nstages * chunk_bytes + 128) + (size_t)warp * g.ksteps * 32 + lane;
    const long long ntiles = (a.n + TILE_P - 1) / TILE_P;
    const int nevals = (MODE == SPEC_LEAPFROG) ? a.nsteps : 1;
    // SPEC_EVAL_DEV (swrt_ode23): the stack the host would pick for the controller's alpha; nothing to do once it is done
    const double* stack = a.stack;
    if constexpr (MODE == SPEC_EVAL_DEV) {
        if (ode23_idle(a.sel.ctl)) return;
        const double al = a.sel.ctl->al[a.sel.stage];
        if (al == 1.0 && a.sel.frame1) stack = static_cast<const double*>(a.sel.frame1);
        else if (al != 0.0 && a.sel.blend) stack = static_cast<const double*>(a.sel.blend);
    }

    if (threadIdx.x == 0) {
        for (int s = 0; s < nstages; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kConsumerWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    long long my_tiles = 0;
    if ((long long)blockIdx.x < ntiles) my_tiles = (ntiles - 1 - blockIdx.x) / gridDim.x + 1;
    const long long total_chunks = my_tiles * nevals * (long long)g.chunks_per_eval;
    // The packed stack streams through a ring of nstages smem buffers with cp.async.bulk; chunk j
    // lives in stage j % nstages.  Producer duty rotates over the warps (lane 0 of warp j % 8 issues
    // chunk j) so that no single warp paces the CTA.  Chunk j is issued when its warp STARTS chunk
    // j - D (D = nstages - lag): the stage it refills was left `lag` chunks ago by that warp, and lag
    // exceeds the deliberate skew between the two warp groups, so the empty-barrier wait inside is
    // (almost) never a stall.  No deadlock: the issue of chunk j happens before its warp waits on the
    // full barrier of chunk j - D, and only needs chunks < j - D, which were issued earlier.
    const int D = nstages - g.lag;
    // This warp issues the chunks pj = warp, warp + 8, warp + 16, ...; the ring stage, the ring iteration and the source
    // chunk of pj are carried incrementally (64-bit divisions by run-time values in the issue path cost the issuing
    // warp ~700 cycles per turn, i.e. once per step at C2).
    // a fused run on a time-dependent flow reads one pre-blended stack per step: the nstack stacks are contiguous, so the
    // source chunk index simply wraps after chunks_per_eval * nstack (every tile walks its evaluations 0..nevals-1 in order)
    const int src_period = g.chunks_per_eval * ((MODE == SPEC_LEAPFROG && a.nstack > 1) ? a.nstack : 1);
    long long pj = warp;
    int p_st = warp % nstages, p_src = warp % src_period;
    long long p_it = warp / nstages;
    auto producer_issue = [&]() {          // lane 0 only; issues chunk pj
        if (p_it > 0) mbar_wait(&empty_bar[p_st], (uint32_t)((p_it - 1) & 1));
        mbar_expect_tx(&full_bar[p_st], chunk_bytes);
        bulk_g2s(smem_raw + (size_t)p_st * chunk_bytes, stack + (size_t)p_src * g.chunk_doubles, chunk_bytes, &full_bar[p_st]);
    };
    auto producer_advance = [&]() {        // all lanes (uniform): pj += kConsumerWarps
        pj += kConsumerWarps;
        p_st += kConsumerWarps;
        while (p_st >= nstages) { p_st -= nstages; p_it++; }
        p_src += kConsumerWarps;
        while (p_src >= src_period) p_src -= src_period;
    };
    static_assert(kConsumerWarps >= 8, "the prologue assumes at most one chunk per warp (D < kConsumerWarps)");
    if (pj < D && pj < total_chunks) {
        if (lane == 0) producer_issue();
        producer_advance();
    }

    if (warp >= kConsumerWarps / 2 && g.desync_ns > 0 && kCtasPerSm == 1) {
        // __nanosleep returns far too early for this purpose (measured ~250 cycles for 2000 ns): spin on
        // the SM clock instead (desync_ns is converted with the nominal 1.9 GHz it was computed for)
        const long long until = clock64() + (long long)(g.desync_ns * 1.9);
        while (clock64() < until) {}
    }

    // ===== consumer warps =====
    const int quad_row = lane >> 2;       // packet row inside an m-tile
    const int jq = lane & 3;              // complex column inside an n-tile (C fragment) / k row (A fragment)
    const int kx0 = jq >> 1;              // first kx handled by this lane's A element (0 or 1)
    const bool odd = lane & 1;            // A element is Ei (odd) or Er (even)
    const int chunks_per_pass = g.ksteps / g.kc;
    const int kyp_passes = g.npass;

    int stage = 0; uint32_t phase = 0;
    long long ci = 0;        // chunks consumed so far by this warp
    bool ready = false;      // next chunk's full barrier already observed complete
#ifdef SWRT_TRACE
    int trace_n = 0;
#define SWRT_TRACE_EV(id)                                                                      \
    do {                                                                                       \
        if (a.trace && blockIdx.x == 3 && lane == 0 && trace_n < 4 * 160)                      \
            a.trace[(size_t)warp * 4 * 160 + trace_n++] = (unsigned long long)clock64();       \
    } while (0)
#else
#define SWRT_TRACE_EV(id) do {} while (0)
#endif

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        long long prow[MT];
        double px[MT], py[MT], pk[MT], pl[MT];
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
            long long r = tile * TILE_P + (long long)warp * 8 * MT + mt * 8 + quad_row;
            prow[mt] = r;
            long long rc = r < a.n ? r : a.n - 1;
            if (MODE == SPEC_LEAPFROG) { px[mt] = a.x[rc]; py[mt] = a.y[rc]; pk[mt] = a.k[rc]; pl[mt] = a.l[rc]; }
            else { px[mt] = a.xin[rc]; py[mt] = a.yin[rc]; pk[mt] = 0; pl[mt] = 0; }
        }

        // half-drift displacement dt/2 * gH*k/omega(k): k only changes in the kick, so the value computed
        // after a kick serves the second half drift of that step AND the first half drift of the next
        double hcx[MT], hcy[MT];
        if (MODE == SPEC_LEAPFROG) {
#pragma unroll
            for (int mt = 0; mt < MT; mt++) {
                half_drift(pk[mt], pl[mt], a.f2, a.gH, __dmul_rn(__dmul_rn(0.5, a.dt), a.gH), hcx[mt], hcy[mt]);
            }
        }

        for (int ev = 0; ev < nevals; ev++) {
            if (MODE == SPEC_LEAPFROG) {
                // phi1(dt/2): x += dt/2 * gH*k/omega(k)   (ode_symplectic.m:13-16,34)
#pragma unroll
                for (int mt = 0; mt < MT; mt++) { px[mt] = __dadd_rn(px[mt], hcx[mt]); py[mt] = __dadd_rn(py[mt], hcy[mt]); }
            }
            // ---- twiddle seeds -------------------------------------------------------------
            double tp_[MT], tq_[MT];            // x twiddle in (p,q) form: p = this lane's A element
            double ep0[MT], eq0[MT];            // value at the start of every pass
            double xdc[MT], xds[MT];            // rotation by e^{i 4 tx} minus one (two k-steps), sign-adjusted
            double ep1[MT], eq1[MT];            // second chain: value at k-step 1 of every pass
            double tpB[MT], tqB[MT];
            Cplx ytw[MT][G];                    // e^{i ky ty} for this lane's ky of each group
            Cplx yrot[MT];                      // e^{i 4G ty}
            double F[MT][NF];
            double kyd[MT];                     // PSI: this lane's ky of group 0 in the current pass (as double)
#pragma unroll
            for (int mt = 0; mt < MT; mt++) {
                double s1, c1;
                sincospi(reduced_turns(px[mt], a.dx, a.nxd, a.inv_nx), &s1, &c1);
                double er = kx0 ? c1 : 1.0, ei = kx0 ? s1 : 0.0;
                ep0[mt] = odd ? ei : er;
                eq0[mt] = odd ? er : ei;
                xdc[mt] = -2.0 * s1 * s1;
                double ds = 2.0 * s1 * c1;
                xds[mt] = odd ? ds : -ds;
                // two interleaved recurrences (even / odd k-steps), each advancing by e^{i 4 tx}: half the dependent
                // chain length per k-step; ep1 = ep0 rotated once by e^{i 2 tx}
                ep1[mt] = fma(ep0[mt], xdc[mt], fma(eq0[mt], xds[mt], ep0[mt]));
                eq1[mt] = fma(eq0[mt], xdc[mt], fma(-ep0[mt], xds[mt], eq0[mt]));
                {
                    const double s2 = ds, c2 = fma(-2.0 * s1, s1, 1.0);     // sin 2tx, cos 2tx
                    xdc[mt] = -2.0 * s2 * s2;
                    const double ds2 = 2.0 * s2 * c2;
                    xds[mt] = odd ? ds2 : -ds2;
                }
                double sy, cy;
                sincospi(reduced_turns(py[mt], a.dx, a.nxd, a.inv_nx), &sy, &cy);
                Cplx e1{cy, sy};
                Cplx e2 = cmul(e1, e1);
                Cplx e3 = cmul(e2, e1);
                Cplx e4 = cmul(e2, e2);
                Cplx cur = jq == 0 ? Cplx{1.0, 0.0} : (jq == 1 ? e1 : (jq == 2 ? e2 : e3));
#pragma unroll
                for (int gg = 0; gg < G; gg++) {
                    ytw[mt][gg] = cur;
                    cur = cmul(cur, e4);
                }
                yrot[mt] = cpow<G>(e4);
#pragma unroll
                for (int c = 0; c < NF; c++) F[mt][c] = 0.0;
                kyd[mt] = (double)jq;
            }

            if constexpr (ATAB) {
                // the same two recurrences the in-loop rotation runs, tabulated once per step for all passes
                double ap = ep0[0], aq = eq0[0], bp = ep1[0], bq = eq1[0];
                for (int s = 0; s < g.ksteps; s += 2) {
                    sA[s * 32] = ap; sA[(s + 1) * 32] = bp;
                    const double nap = fma(ap, xdc[0], fma(aq, xds[0], ap)), naq = fma(aq, xdc[0], fma(-ap, xds[0], aq));
                    const double nbp = fma(bp, xdc[0], fma(bq, xds[0], bp)), nbq = fma(bq, xdc[0], fma(-bp, xds[0], bq));
                    ap = nap; aq = naq; bp = nbp; bq = nbq;
                }
            }
            double apf[kKUnroll];                  // ATAB 2: the A elements of the next unrolled body, in flight from L2
            if constexpr (ATAB == 2) {
#pragma unroll
                for (int su = 0; su < kKUnroll; su++) apf[su] = sA[su * 32];
            }
            // ---- passes over ky blocks -----------------------------------------------------
            for (int pass = 0; pass < kyp_passes; pass++) {
                double acc[MT][NT][2];
#pragma unroll
                for (int mt = 0; mt < MT; mt++) {
#pragma unroll
                    for (int t = 0; t < NT; t++) { acc[mt][t][0] = 0.0; acc[mt][t][1] = 0.0; }
                    if constexpr (!ATAB) {
                        tp_[mt] = ep0[mt]; tq_[mt] = eq0[mt];
                        tpB[mt] = ep1[mt]; tqB[mt] = eq1[mt];
                    }
                }
                for (int ch = 0; ch < chunks_per_pass; ch++) {
                    SWRT_TRACE_EV(0);
                    {   // producer duty for chunk ci + D (one warp in eight, lane 0 only)
                        if (ci + D == pj && pj < total_chunks) {
                            if (lane == 0) producer_issue();
                            producer_advance();
                        }
                    }
                    SWRT_TRACE_EV(1);
                    if (!ready) mbar_wait(&full_bar[stage], phase);
                    SWRT_TRACE_EV(2);
                    const double2* sB = reinterpret_cast<const double2*>(smem_raw + (size_t)stage * chunk_bytes) + lane;
                    const double* sAc = sA + (size_t)ch * g.kc * 32;
                    int nstage = stage + 1; uint32_t nphase = phase;
                    if (nstage == nstages) { nstage = 0; nphase ^= 1; }
                    for (int s0 = 0; s0 < g.kc; s0 += kKUnroll) {
                        // probe the NEXT chunk's full barrier while this chunk's last k-steps run, so the
                        // hand-over at the chunk boundary does not wait on the barrier round trip
                        if (s0 + kKUnroll >= g.kc) ready = mbar_test(&full_bar[nstage], nphase);
                        double acur[kKUnroll];
                        if constexpr (ATAB == 2) {
                            int nb = ch * g.kc + s0 + kKUnroll;          // next body of this pass; the table serves every pass
                            if (nb >= g.ksteps) nb = 0;
#pragma unroll
                            for (int su = 0; su < kKUnroll; su++) { acur[su] = apf[su]; apf[su] = sA[(nb + su) * 32]; }
                        }
#pragma unroll
                        for (int su = 0; su < kKUnroll; su++) {
                            const int s = s0 + su;
                            if constexpr (ATAB == 1) tp_[0] = sAc[s * 32];
                            if constexpr (ATAB == 2) tp_[0] = acur[su];
#pragma unroll
                            for (int tp = 0; tp < HALF_NT; tp++) {
                                double2 b = sB[(s * HALF_NT + tp) * 32];
#pragma unroll
                                for (int mt = 0; mt < MT; mt++) {
                                    dmma884(acc[mt][2 * tp][0], acc[mt][2 * tp][1], tp_[mt], b.x);
                                    dmma884(acc[mt][2 * tp + 1][0], acc[mt][2 * tp + 1][1], tp_[mt], b.y);
                                }
                            }
#pragma unroll
                            for (int mt = 0; mt < (ATAB ? 0 : MT); mt++) {
                                // this chain's next value (two k-steps ahead): E <- E + E*(e^{i 4 tx} - 1); then swap chains
                                double np = fma(tp_[mt], xdc[mt], fma(tq_[mt], xds[mt], tp_[mt]));
                                double nq = fma(tq_[mt], xdc[mt], fma(-tp_[mt], xds[mt], tq_[mt]));
                                tp_[mt] = tpB[mt]; tq_[mt] = tqB[mt];
                                tpB[mt] = np; tqB[mt] = nq;
                            }
                        }
                    }
                    SWRT_TRACE_EV(3);
                    // every lane's LDS of this stage has been consumed by the DMMAs above (mma.sync is
                    // warp-convergent), so lane 0 may hand the stage back
                    if (lane == 0) mbar_arrive(&empty_bar[stage]);
                    stage = nstage; phase = nphase;
                    ++ci;
                }
                // ---- stage 2: F_c += Gr*cos(ky ty) - Gi*sin(ky ty) for this lane's ky ----------
#pragma unroll
                for (int mt = 0; mt < MT; mt++) stage2_pass<NPL, G, PSI, NF>(acc[mt], ytw[mt], yrot[mt], kyd[mt], F[mt]);
            }
            // ---- quad reduction: the 4 lanes of a quad hold 4 interleaved ky subsets ----------
#pragma unroll
            for (int mt = 0; mt < MT; mt++) finish_planes<PSI, NPL, NF, MODE == SPEC_EVAL_DEV>(F[mt], a, ev);
            if (MODE == SPEC_LEAPFROG) {
                if constexpr (NF >= 6) {
#pragma unroll
                    for (int mt = 0; mt < MT; mt++) leapfrog_kick<NF>(F[mt], a, px[mt], py[mt], pk[mt], pl[mt], hcx[mt], hcy[mt]);
                }
            } else {
                if (jq == 0) {
#pragma unroll
                    for (int mt = 0; mt < MT; mt++) {
                        if (prow[mt] < a.n) {
#pragma unroll
                            for (int c = 0; c < NF; c++)
                                if (a.out[c]) a.out[c][prow[mt]] = F[mt][c];
                        }
                    }
                }
            }
        }
        if (MODE == SPEC_LEAPFROG) {
            if (jq == 0) {
#pragma unroll
                for (int mt = 0; mt < MT; mt++) {
                    if (prow[mt] < a.n) {
                        a.x[prow[mt]] = px[mt]; a.y[prow[mt]] = py[mt];
                        a.k[prow[mt]] = pk[mt]; a.l[prow[mt]] = pl[mt];
                    }
                }
            }
        }
    }
}

template <int NPL, int G, int MT, int MODE, bool PSI, int ATAB>
static cudaError_t launch_inst2(const SpecArgs& a, int num_sms, cudaStream_t st) {
    constexpr int TILE_P = kConsumerWarps * 8 * MT;
    size_t smem = spectral_smem_bytes(a.g);
    auto kern = spectral_kernel<NPL, G, MT, MODE, PSI, ATAB>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long ntiles = (a.n + TILE_P - 1) / TILE_P;
    int grid = (int)(ntiles < (long long)num_sms * kCtasPerSm ? ntiles : (long long)num_sms * kCtasPerSm);
    if (grid < 1) grid = 1;
    kern<<<grid, kSpecThreads, smem, st>>>(a);
    return cudaGetLastError();
}

template <int NPL, int G, int MT, int MODE, bool PSI>
static cudaError_t launch_inst(const SpecArgs& a, int num_sms, cudaStream_t st) {
    if constexpr (MT == 1) {
        if (a.g.atab == 1) return launch_inst2<NPL, G, MT, MODE, PSI, 1>(a, num_sms, st);
        if (a.g.atab == 2 && a.twid) return launch_inst2<NPL, G, MT, MODE, PSI, 2>(a, num_sms, st);
    }
    return launch_inst2<NPL, G, MT, MODE, PSI, 0>(a, num_sms, st);
}

template <int NPL, int G, int MT>
static cudaError_t dispatch_mode(const SpecArgs& a, int mode, int num_sms, cudaStream_t st) {
    if (a.psi) {
        if constexpr (NPL == 3) {
            if (mode == SPEC_LEAPFROG) return launch_inst<NPL, G, MT, SPEC_LEAPFROG, true>(a, num_sms, st);
            return launch_inst<NPL, G, MT, SPEC_EVAL, true>(a, num_sms, st);
        } else return cudaErrorInvalidValue;
    }
    if (mode == SPEC_LEAPFROG) {
        if constexpr (NPL == 6) return launch_inst<NPL, G, MT, SPEC_LEAPFROG, false>(a, num_sms, st);
        else return cudaErrorInvalidValue;
    }
    return launch_inst<NPL, G, MT, SPEC_EVAL, false>(a, num_sms, st);
}

// swrt_ode23's evaluations: the six planes (or the psi-hat moment planes) with one m-tile, alpha from the controller
cudaError_t launch_spectral_eval_dev(const SpecArgs& a, int num_sms, cudaStream_t st) {
    if (a.psi && a.g.npl == 3 && a.g.G == 8) return launch_inst<3, 8, 1, SPEC_EVAL_DEV, true>(a, num_sms, st);
    if (!a.psi && a.g.npl == 6 && a.g.G == 4) return launch_inst<6, 4, 1, SPEC_EVAL_DEV, false>(a, num_sms, st);
    return cudaErrorInvalidValue;
}

cudaError_t launch_spectral(const SpecArgs& a, int mode, int mtiles, int num_sms, cudaStream_t st) {
    const int npl = a.g.npl, G = a.g.G;
#define SWRT_INST(NPL_, G_, MT_) \
    if (npl == NPL_ && G == G_ && mtiles == MT_) return dispatch_mode<NPL_, G_, MT_>(a, mode, num_sms, st);
    SWRT_INST(6, 4, 1) SWRT_INST(6, 2, 2)
    SWRT_INST(7, 4, 1) SWRT_INST(7, 2, 2)
    SWRT_INST(2, 12, 1) SWRT_INST(2, 6, 2)
    SWRT_INST(3, 8, 1) SWRT_INST(3, 4, 2)
    SWRT_INST(4, 6, 1) SWRT_INST(4, 3, 2)
    SWRT_INST(1, 24, 1) SWRT_INST(1, 12, 2)
#undef SWRT_INST
    return cudaErrorInvalidValue;
}

// ================================================================================================
// anchored leapfrog (DESIGN.md section 3e): per sub-step  drift + key -> counting sort -> K1 (anchor_transform_kernel) -> K2
// ================================================================================================
// Anchor cells of 2^-m turns, m the smallest with (pi kmax 2^-m)^R / R! <= 2^-53 (the truncation bound of the expansion
// relative to sum |B|).  Grids 256^2 and 512^2 (the transforms K1 is instantiated for): below, the dense kernel's cost per
// packet is small enough that the anchored sub-step's fixed cost does not pay; above, an anchor's H' block (npass * 12 KB)
// no longer fits two K2 CTAs per SM.
int anchor_log2_cells(int nx) {
    if (nx < 256 || nx > 512 || (nx & (nx - 1))) return 0;
    const double kmax = nx / 2 - 1;
    double fact = 1.0;
    for (int i = 2; i <= kAnchorOrders; i++) fact *= i;
    for (int m = 8; m < 30; m++)
        if (std::pow(M_PI * kmax * std::ldexp(1.0, -m), kAnchorOrders) / fact <= std::ldexp(1.0, -53)) return m;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// K1: the expansion blocks of every anchor cell by a fused fp64 FFT (anchor_transform_kernel)
// ------------------------------------------------------------------------------------------------
// For anchor cell c of N = 64 M cells (M = nx = 2 (kmax + 1)), order r < 8 and every stack column (plane, ky):
//   H~_r(c) = sum_{kx=-kmax..kmax} (kx/kmax)^r C(kx) e^{i pi kx t_c},   t_c = (2c + 1) / N,
// and K2 reads H'_r = i^r / r! * H~_r.  With c = 64 q + s the sum splits into a pre-twiddle and an M-point transform:
//   H~_r(64 q + s) = sum_{k mod M} [ (kx/kmax)^r C(kx) e^{i pi kx (2s + 1) / N} ] e^{2 pi i k q / M},   kx = k or k - M,
// the residue kmax + 1 being zero.  C(+-kx) = (S +- D) / 2 undoes the stack's fold (C(0) = S).  The transform is a
// Stockham radix-8 FFT (last pass radix 4 at M = 256) in shared memory; pre-twiddles and FFT twiddles are sincospi of exact
// dyadic arguments, so no error is carried across s or across passes.
//
// A work item is (pass, tp, ky column j, k-step ks, s): 8 transforms (2 n-tiles x the 4 orders r = 4 ks + 0..3) whose
// outputs at q form one 128-byte line of K2's B layout in cell 64 q + s, hexp[c][pass][ks][tp][lane = col*4 + r%4][which].
// Items run in (column, s) order and are split evenly over a persistent grid; a CTA re-reads the input columns only when
// (pass, tp, j) changes.  Every cell is written whatever the occupancy, so H' depends on the flow and the sub-step only.
constexpr int kAtThreads = 256;
constexpr int kAtTr = 8;                // transforms per work item
constexpr int kAtS = 64;                // N / M: pre-twiddle phases s

__device__ __forceinline__ Cplx cadd(Cplx a, Cplx b) { return Cplx{a.re + b.re, a.im + b.im}; }
__device__ __forceinline__ Cplx csub(Cplx a, Cplx b) { return Cplx{a.re - b.re, a.im - b.im}; }
__device__ __forceinline__ Cplx cmul_i(Cplx a) { return Cplx{-a.im, a.re}; }

// in-place DFT with the positive exponent, v_m <- sum_i v_i e^{2 pi i i m / R}
__device__ __forceinline__ void dft4(Cplx& v0, Cplx& v1, Cplx& v2, Cplx& v3) {
    const Cplx t0 = cadd(v0, v2), t1 = csub(v0, v2), t2 = cadd(v1, v3), t3 = cmul_i(csub(v1, v3));
    v0 = cadd(t0, t2); v2 = csub(t0, t2); v1 = cadd(t1, t3); v3 = csub(t1, t3);
}
template <int R>
__device__ __forceinline__ void dft(Cplx (&v)[R]) {
    if constexpr (R == 4) {
        dft4(v[0], v[1], v[2], v[3]);
    } else {
        static_assert(R == 8, "radix 4 or 8");
        constexpr double h = 0.70710678118654752440;        // sqrt(1/2)
        dft4(v[0], v[2], v[4], v[6]);
        dft4(v[1], v[3], v[5], v[7]);
        const Cplx o1{(v[3].re - v[3].im) * h, (v[3].re + v[3].im) * h};     // e^{i pi/4} O_1
        const Cplx o2 = cmul_i(v[5]);                                         // e^{i pi/2} O_2
        const Cplx o3{(-v[7].re - v[7].im) * h, (v[7].re - v[7].im) * h};    // e^{3 i pi/4} O_3
        const Cplx e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6], o0 = v[1];
        v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
        v[1] = cadd(e1, o1); v[5] = csub(e1, o1);
        v[2] = cadd(e2, o2); v[6] = csub(e2, o2);
        v[3] = cadd(e3, o3); v[7] = csub(e3, o3);
    }
}

template <int M> struct AtSmem {
    static constexpr int kPad = M + M / 8;                   // transform stride in the work buffer (padded, bank spread)
    static constexpr size_t kBuf = (size_t)kAtTr * kPad;     // complex; also holds the 16-double output lines of M cells
    static constexpr size_t kBytes = (kBuf + 2 * M + M + M) * sizeof(Cplx);    // buffer | input (2 n-tiles) | twiddles | pre-twiddles
};
__device__ __forceinline__ int at_pad(int k) { return k + (k >> 3); }

// One Stockham pass of radix R over the 8 transforms of an item, stride L (the product of the earlier radices).
// KIND 0: the first pass, input = weighted, pre-twiddled columns; 1: work buffer in place; 2: the last pass, writes
// H' = i^r / r! * X into the output lines (q-major, 16 doubles per cell, XOR-swizzled by q).
template <int M, int R, int L, int KIND>
__device__ __forceinline__ void at_pass(Cplx* buf, const Cplx* xin, const Cplx* tw, const Cplx* pre, int ks, int kmax) {
    constexpr int BPT = M / R;                                   // butterflies per transform
    constexpr int CNT = kAtTr * BPT / kAtThreads;                 // per thread
    static_assert(CNT >= 1 && kAtTr * BPT % kAtThreads == 0, "butterflies must tile the CTA");
    constexpr int P = AtSmem<M>::kPad;
    auto load = [&](int c, Cplx (&v)[R]) {
        const int u = threadIdx.x + c * kAtThreads, tr = u / BPT, b = u % BPT;
#pragma unroll
        for (int i = 0; i < R; i++) {
            const int k = b + i * BPT;
            if constexpr (KIND == 0) {
                const int kx = k < M / 2 ? k : k - M;
                const double w = (double)kx / (double)kmax;
                const int r = 4 * ks + (tr & 3);
                double wr = 1.0;
                for (int e = 0; e < r; e++) wr *= w;
                const Cplx y = cmul(xin[(tr >> 2) * M + k], pre[k]);
                v[i] = Cplx{wr * y.re, wr * y.im};
            } else {
                v[i] = buf[tr * P + at_pad(k)];
            }
            if constexpr (L > 1) {
                if (i > 0) v[i] = cmul(v[i], tw[(i * (b % L)) * (M / (L * R))]);
            }
        }
        dft<R>(v);
    };
    auto store = [&](int c, const Cplx (&v)[R]) {
        const int u = threadIdx.x + c * kAtThreads, tr = u / BPT, b = u % BPT;
        const int q0 = (b / L) * L * R + b % L;
        if constexpr (KIND < 2) {
#pragma unroll
            for (int m = 0; m < R; m++) buf[tr * P + at_pad(q0 + m * L)] = v[m];
        } else {
            const int krow = tr & 3, r = 4 * ks + krow, which = tr >> 2;
            double fact = 1.0;
            for (int e = 2; e <= r; e++) fact *= (double)e;
            double* line = reinterpret_cast<double*>(buf);
#pragma unroll
            for (int m = 0; m < R; m++) {
                const int q = q0 + m * L;
                const double re = v[m].re / fact, im = v[m].im / fact;
                const double hr = krow == 0 ? re : (krow == 1 ? -im : (krow == 2 ? -re : im));
                const double hi = krow == 0 ? im : (krow == 1 ? re : (krow == 2 ? -im : -re));
                const int p = krow * 2 + which;                   // line position of the real part; imaginary at + 8
                line[q * 16 + (p ^ (q & 15))] = hr;
                line[q * 16 + ((p + 8) ^ (q & 15))] = hi;
            }
        }
    };
    if constexpr (KIND == 1) {
        // thread group c touches only transforms [c * 8 / CNT, (c + 1) * 8 / CNT): in place one group at a time
#pragma unroll
        for (int c = 0; c < CNT; c++) {
            Cplx v[R];
            load(c, v);
            __syncthreads();
            store(c, v);
        }
    } else {
        // the first pass reads the inputs, not the buffer; the last one writes lines that span every transform's region
        Cplx v[CNT][R];
#pragma unroll
        for (int c = 0; c < CNT; c++) load(c, v[c]);
        if constexpr (KIND == 2) __syncthreads();
#pragma unroll
        for (int c = 0; c < CNT; c++) store(c, v[c]);
    }
    __syncthreads();
}

template <int LOGM>
__global__ void __launch_bounds__(kAtThreads, 2) anchor_transform_kernel(const SpecArgs a) {
    constexpr int M = 1 << LOGM, N = kAtS * M;
    constexpr int NT = 24, HALF_NT = NT / 2;                     // psi-hat stack: 3 planes x G = 8
    constexpr size_t P = AtSmem<M>::kBuf;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Cplx* buf = reinterpret_cast<Cplx*>(smem_raw);
    Cplx* xin = buf + P;                     // [which][k]: the item's two input columns, unfolded, residues mod M
    Cplx* tw = xin + 2 * M;                  // e^{2 pi i m / M}
    Cplx* pre = tw + M;                      // e^{i pi kx (2s + 1) / N}
    const int kmax = a.g.kmax;
    const int ncols = a.g.npass * HALF_NT * 4 * 2;
    const long long items = (long long)ncols * kAtS;
    const long long lo = items * blockIdx.x / gridDim.x, hi = items * (blockIdx.x + 1) / gridDim.x;
    for (int m = threadIdx.x; m < M; m += kAtThreads) {
        double sn, cs;
        sincospi((double)m * (2.0 / M), &sn, &cs);
        tw[m] = Cplx{cs, sn};
    }
    int cached = -1;
    for (long long it = lo; it < hi; it++) {
        const int col = (int)(it / kAtS), s = (int)(it % kAtS);
        const int ks = col & 1, j = (col >> 1) & 3, tp = (col >> 3) % HALF_NT, pass = (col >> 3) / HALF_NT;
        if ((col >> 1) != cached) {          // unfold the stack's S/D columns of (pass, tp, j) for both n-tiles
            cached = col >> 1;
            for (int e = threadIdx.x; e < 2 * M; e += kAtThreads) {
                const int which = e / M, kx = e % M;
                if (kx > kmax) {
                    if (kx == kmax + 1) xin[which * M + kx] = Cplx{0.0, 0.0};
                    continue;
                }
                // lane = krow + 4 * ncol, krow = 2 (kx & 1) + part_k, ncol = 2 j + part_n: v[part_k][part_n]
                const double* src = a.stack + ((size_t)(pass * a.g.ksteps + (kx >> 1)) * HALF_NT + tp) * 64 + which;
                const int l0 = 2 * (kx & 1) + 8 * j;
                const double v00 = src[(l0) * 2], v01 = src[(l0 + 4) * 2], v10 = src[(l0 + 1) * 2], v11 = src[(l0 + 5) * 2];
                // S = (v00, v01), D = (v11, -v10)
                if (kx == 0) {
                    xin[which * M] = Cplx{v00, v01};
                } else {
                    xin[which * M + kx] = Cplx{0.5 * (v00 + v11), 0.5 * (v01 - v10)};
                    xin[which * M + M - kx] = Cplx{0.5 * (v00 - v11), 0.5 * (v01 + v10)};
                }
            }
        }
        for (int k = threadIdx.x; k < M; k += kAtThreads) {
            const int kx = k < M / 2 ? k : k - M;
            double sn, cs;
            sincospi((double)(kx * (2 * s + 1)) * (1.0 / N), &sn, &cs);
            pre[k] = Cplx{cs, sn};
        }
        __syncthreads();                     // inputs ready; the previous item's lines have been written out
        at_pass<M, 8, 1, 0>(buf, xin, tw, pre, ks, kmax);
        if constexpr (LOGM == 9) {
            at_pass<M, 8, 8, 1>(buf, xin, tw, pre, ks, kmax);
            at_pass<M, 8, 64, 2>(buf, xin, tw, pre, ks, kmax);
        } else {
            static_assert(LOGM == 8, "M = 256 or 512");
            at_pass<M, 8, 8, 1>(buf, xin, tw, pre, ks, kmax);
            at_pass<M, 4, 64, 2>(buf, xin, tw, pre, ks, kmax);
        }
        // the M output lines of this item: 128 contiguous bytes in each cell 64 q + s
        const double* line = reinterpret_cast<const double*>(buf);
        double* dst = a.hexp + (size_t)s * a.anc_block + ((size_t)(pass * 2 + ks) * HALF_NT + tp) * 64 + j * 16;
        for (int e = threadIdx.x; e < M * 16; e += kAtThreads) {
            const int q = e >> 4, p = e & 15;
            dst[(size_t)q * kAtS * a.anc_block + p] = line[q * 16 + (p ^ (q & 15))];
        }
    }
}

double anchor_transform_flops(const PackGeom& g) {
    // per transform point: complex product by the pre-twiddle (6) and the order weight (2) in the first pass, 1/r! (2) in
    // the last; per radix-8 butterfly 56 (two 4-point DFTs of 16, the e^{i pi/4} rotations 8, the combination 16), per
    // radix-4 one 16; a complex twiddle (6) on all but the first input of every butterfly after the first pass
    const int M = g.nx;
    const double bf8 = 56.0 + 7 * 6.0, bf4 = 16.0 + 3 * 6.0;
    double per = 10.0 * M + 56.0 * (M / 8) + bf8 * (M / 8) + (M == 512 ? bf8 * (M / 8) : bf4 * (M / 4));
    return per * (double)g.npass * g.NT * 4 * kAnchorOrders * kAtS;
}

cudaError_t launch_anchor_transform(const SpecArgs& a, int nanchors, int num_sms, cudaStream_t st) {
    if (a.g.npl != 3 || a.g.G != 8 || !a.psi || 2 * (a.g.kmax + 1) != a.g.nx || nanchors != kAtS * a.g.nx)
        return cudaErrorInvalidValue;
    auto run = [&](auto kern, size_t smem) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kAtThreads, smem);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) per_sm = 1;
        const long long items = (long long)a.g.npass * 12 * 4 * 2 * kAtS;
        const long long grid = (long long)num_sms * per_sm < items ? (long long)num_sms * per_sm : items;
        kern<<<(unsigned)grid, kAtThreads, smem, st>>>(a);
        return cudaGetLastError();
    };
    if (a.g.nx == 512) return run(anchor_transform_kernel<9>, AtSmem<512>::kBytes);
    if (a.g.nx == 256) return run(anchor_transform_kernel<8>, AtSmem<256>::kBytes);
    return cudaErrorInvalidValue;
}

// first half drift (the dense kernel's arithmetic) and the anchor key; rank = position inside the anchor (atomic order:
// results do not depend on it)
__global__ void anchor_key_kernel(double* __restrict__ x, double* __restrict__ y, const double* __restrict__ k,
                                  const double* __restrict__ l, long long n, double dx, double nxd, double inv_nx, double f2,
                                  double gH, double dt, double inv_h, int nanchors, unsigned long long* __restrict__ cnt,
                                  int* __restrict__ key, unsigned long long* __restrict__ rank) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double hx, hy;
    half_drift(k[i], l[i], f2, gH, __dmul_rn(__dmul_rn(0.5, dt), gH), hx, hy);
    const double xi = __dadd_rn(x[i], hx);
    x[i] = xi;
    y[i] = __dadd_rn(y[i], hy);
    int c = (int)floor(reduced_turns(xi, dx, nxd, inv_nx) * inv_h);
    c = c < 0 ? 0 : (c >= nanchors ? nanchors - 1 : c);
    key[i] = c;
    rank[i] = atomicAdd(&cnt[c], 1ULL);
}
void launch_anchor_key(double* x, double* y, const double* k, const double* l, long long n, double dx, double nxd, double inv_nx,
                       double f2, double gH, double dt, double inv_h, int nanchors, unsigned long long* cnt, int* key,
                       unsigned long long* rank, cudaStream_t st) {
    anchor_key_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, y, k, l, n, dx, nxd, inv_nx, f2, gH, dt, inv_h, nanchors, cnt,
                                                                  key, rank);
}

// exclusive scan of the anchor counts (one CTA; at most 2^15 anchors)
__global__ void __launch_bounds__(1024) anchor_scan_kernel(const unsigned long long* __restrict__ cnt, unsigned long long* __restrict__ off,
                                                           int nanchors) {
    __shared__ unsigned long long sc[1024];
    const int t = threadIdx.x;
    const int per = (nanchors + 1023) / 1024;
    const int lo = t * per, hi = (lo + per < nanchors) ? lo + per : nanchors;
    unsigned long long c = 0;
    for (int i = lo; i < hi; i++) c += cnt[i];
    sc[t] = c;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const unsigned long long vc = t >= d ? sc[t - d] : 0;
        __syncthreads();
        sc[t] += vc;
        __syncthreads();
    }
    unsigned long long base = t ? sc[t - 1] : 0;
    for (int i = lo; i < hi; i++) {
        off[i] = base;
        base += cnt[i];
    }
}
void launch_anchor_scan(const unsigned long long* cnt, unsigned long long* off, int nanchors, cudaStream_t st) {
    anchor_scan_kernel<<<1, 1024, 0, st>>>(cnt, off, nanchors);
}

__global__ void anchor_scatter_kernel(const int* __restrict__ key, const unsigned long long* __restrict__ rank,
                                      const unsigned long long* __restrict__ off, long long* __restrict__ perm, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) perm[off[key[i]] + rank[i]] = i;
}
void launch_anchor_scatter(const int* key, const unsigned long long* rank, const unsigned long long* off, long long* perm, long long n,
                           cudaStream_t st) {
    anchor_scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(key, rank, off, perm, n);
}

// K2: one CTA per anchor.  The anchor's H' block (8 orders x 2 nky x 3 planes, in K2's B-fragment order) is bulk-copied into
// shared memory; each warp takes 8-packet groups of the anchor: A = [z^0 .. z^7] of its 8 packets (two k-steps of m8n8k4),
// per ky pass 2 x NT DMMAs give G = sum_r z^r H'_r, then the dense kernel's stage 2, quad reduction, kick and half drift.
// A packet's result depends on its own state and its anchor's H' only: grouping, order and padding do not change a bit.
template <int G>
__global__ void __launch_bounds__(kAncWarps * 32, 2) anchored_step_kernel(const SpecArgs a) {
    constexpr int NPL = 3, NT = NPL * G, HALF_NT = NT / 2, NF = 6;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int anc = blockIdx.x;
    const unsigned long long cnt = a.anc_cnt[anc];
    if (cnt == 0) return;
    const unsigned long long off = a.anc_off[anc];
    const uint32_t block_bytes = (uint32_t)(a.anc_block * 8);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + block_bytes);
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, block_bytes);
        const unsigned char* src = reinterpret_cast<const unsigned char*>(a.hexp + (size_t)anc * a.anc_block);
        for (uint32_t o = 0; o < block_bytes; o += 32768) {
            const uint32_t b = block_bytes - o < 32768 ? block_bytes - o : 32768;
            bulk_g2s(smem_raw + o, src + o, b, bar);
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int quad_row = lane >> 2, jq = lane & 3;
    const double ta = ((double)anc + 0.5) * a.anc_h;
    const long long ngroups = (long long)((cnt + 7) / 8);
    bool waited = false;
    for (long long gi = warp; gi < ngroups; gi += kAncWarps) {
        long long row = gi * 8 + quad_row;
        const bool valid = row < (long long)cnt;
        if (!valid) row = (long long)cnt - 1;
        const long long p = a.anc_perm[off + row];
        double px = a.x[p], py = a.y[p], pk = a.k[p], pl = a.l[p];     // x, y after the first half drift
        // A fragments: z^jq (k-step 0) and z^(4 + jq) (k-step 1)
        const double z = a.zscale * (reduced_turns(px, a.dx, a.nxd, a.inv_nx) - ta);
        const double z2 = z * z;
        const double zj = jq == 0 ? 1.0 : (jq == 1 ? z : (jq == 2 ? z2 : z2 * z));
        const double a0 = zj, a1 = zj * (z2 * z2);
        // y twiddles exactly as the dense kernel forms them
        Cplx ytw[G], yrot;
        double F[NF], kyd;
        {
            double sy, cy;
            sincospi(reduced_turns(py, a.dx, a.nxd, a.inv_nx), &sy, &cy);
            Cplx e1{cy, sy};
            Cplx e2 = cmul(e1, e1);
            Cplx e3 = cmul(e2, e1);
            Cplx e4 = cmul(e2, e2);
            Cplx cur = jq == 0 ? Cplx{1.0, 0.0} : (jq == 1 ? e1 : (jq == 2 ? e2 : e3));
#pragma unroll
            for (int gg = 0; gg < G; gg++) {
                ytw[gg] = cur;
                cur = cmul(cur, e4);
            }
            yrot = cpow<G>(e4);
#pragma unroll
            for (int c = 0; c < NF; c++) F[c] = 0.0;
            kyd = (double)jq;
        }
        if (!waited) { mbar_wait(bar, 0); waited = true; }
        for (int pass = 0; pass < a.g.npass; pass++) {
            double acc[NT][2];
#pragma unroll
            for (int t = 0; t < NT; t++) { acc[t][0] = 0.0; acc[t][1] = 0.0; }
            const double2* sB = reinterpret_cast<const double2*>(smem_raw) + (size_t)pass * 2 * HALF_NT * 32 + lane;
#pragma unroll
            for (int ks = 0; ks < 2; ks++) {
                const double av = ks ? a1 : a0;
#pragma unroll
                for (int tp = 0; tp < HALF_NT; tp++) {
                    const double2 b = sB[(ks * HALF_NT + tp) * 32];
                    dmma884(acc[2 * tp][0], acc[2 * tp][1], av, b.x);
                    dmma884(acc[2 * tp + 1][0], acc[2 * tp + 1][1], av, b.y);
                }
            }
            stage2_pass<NPL, G, true, NF>(acc, ytw, yrot, kyd, F);
        }
        finish_planes<true, NPL, NF>(F, a, a.ev);
        double hcx, hcy;
        leapfrog_kick<NF>(F, a, px, py, pk, pl, hcx, hcy);
        if (valid && jq == 0) { a.x[p] = px; a.y[p] = py; a.k[p] = pk; a.l[p] = pl; }
    }
    if (!waited) mbar_wait(bar, 0);       // the bulk copy must land before the CTA exits
}

cudaError_t launch_anchored_step(const SpecArgs& a, int nanchors, cudaStream_t st) {
    if (a.g.npl != 3 || a.g.G != 8 || !a.psi) return cudaErrorInvalidValue;
    const size_t smem = a.anc_block * 8 + 16;
    auto kern = anchored_step_kernel<8>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<nanchors, kAncWarps * 32, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace swrt
