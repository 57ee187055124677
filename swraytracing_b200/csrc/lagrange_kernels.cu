// lagrange_kernels.cu -- LAGRANGE6 mode of libswrt: the reference's own field evaluation, the
// 6x6-point (Iord = 2) periodic Lagrange stencil of ray_trace_sw/interpolate.m:12-49 (a quad of lanes
// per packet in the eval / leapfrog kernels, one thread per packet in the RK4 ones), fused with the
// integrators that call it (ode_symplectic.m:33-37, step_packet.m:37-78, step_packet_xka.m:38-91 +
// cg_sw.m:15-31).
//
// Data layout: the gridded planes are node-interleaved, grid[(ix*nx + iy)*NPL + c], so the six
// (seven) values of one stencil node are one contiguous 48 (56) byte record and one stencil row is a
// contiguous run; the whole grid (12.6 MB at 512^2) stays L2-resident.  The kernels are gather /
// L2-bound: 36 nodes * NPL * 8 bytes per evaluation.
#include "swrt_internal.h"

namespace swrt {

namespace {

constexpr int IORD = 2;
constexpr int NW = 2 * (IORD + 1);   // 6 weights per axis

struct Stencil {
    int ig[NW], jg[NW];
    double wx[NW], wy[NW];
};

__device__ __forceinline__ double matlab_mod(double a, double m) {
    double r = fmod(a, m);
    if (r < 0.0) r += m;
    return r;
}

// interpolate.m:33-41, operation for operation:  w_i = 1; for j ~= i (ascending):  w_i = w_i*(a - j + bump)/(j - i)
// -- multiply by the numerator factor, then divide by the integer (j - i), five times per weight.  This translation
// unit is compiled with -fmad=false (Makefile / __graft_entry__.py) so that no product is fused into a following
// add: with IEEE division, sqrt, floor and fmod the LAGRANGE6 kernels then reproduce the reference's double
// arithmetic bit for bit (tests/test_gpu_parity.py::test_lagrange_mode_is_bit_identical_to_the_restatement).
__device__ __forceinline__ void lagrange_weights(double a, double bump, double* w) {
    double t[NW];
#pragma unroll
    for (int j = 0; j < NW; j++) t[j] = a - (double)(j - IORD) + bump;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        double p = 1.0;
#pragma unroll
        for (int j = 0; j < NW; j++)
            if (j != i) p = p * t[j] / (double)(j - i);
        w[i] = p;
    }
}

__device__ __forceinline__ void make_stencil(double x, double y, double dx, double dy, int nx, int ny,
                                             double bump, Stencil& s) {
    // interpolate.m:21-31
    double xl = matlab_mod(x / dx, (double)nx);
    double yl = matlab_mod(y / dy, (double)ny);
    double fx = floor(xl), fy = floor(yl);
    double ax = 1.0 + xl - (1.0 + fx);
    double ay = 1.0 + yl - (1.0 + fy);
    lagrange_weights(ax, bump, s.wx);
    lagrange_weights(ay, bump, s.wy);
    int i0 = (int)fx, j0 = (int)fy;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        // reference: ig = 1 + mod(i0 + i - 1, nx), jg = 1 + mod(j0 + j - 1, nx)  (both wrap with nx)
        int a = (i0 + i - IORD) % nx; if (a < 0) a += nx;
        int b = (j0 + i - IORD) % nx; if (b < 0) b += nx;
        s.ig[i] = a; s.jg[i] = b;
    }
}

// sum_i sum_j (wx_i*wy_j) * node(ig,jg), i outer, j inner -- interpolate.m:43-49
template <int NPL>
__device__ __forceinline__ void gather_planes(const double* __restrict__ grid, int nx, const Stencil& s, double* F) {
#pragma unroll
    for (int c = 0; c < NPL; c++) F[c] = 0.0;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        const double* row = grid + (size_t)s.ig[i] * nx * NPL;
#pragma unroll
        for (int j = 0; j < NW; j++) {
            const double w = s.wx[i] * s.wy[j];
            const double* node = row + (size_t)s.jg[j] * NPL;
            if constexpr (NPL % 2 == 0) {
                const double2* n2 = reinterpret_cast<const double2*>(node);
#pragma unroll
                for (int c = 0; c < NPL / 2; c++) {
                    double2 v = __ldg(n2 + c);
                    F[2 * c] = F[2 * c] + w * v.x;
                    F[2 * c + 1] = F[2 * c + 1] + w * v.y;
                }
            } else {
#pragma unroll
                for (int c = 0; c < NPL; c++) F[c] = F[c] + w * __ldg(node + c);
            }
        }
    }
}

// ---- quad-per-packet evaluation (eval + leapfrog kernels) ----------------------------------------------------------
// Four lanes share one packet: lane q gathers the plane pair (2q, 2q+1) of every stencil node, so the quad's loads of a
// node are 48 (56) contiguous bytes instead of three instructions that each scatter over 32 different lines -- the
// thread-per-packet version is bound by L1 data-pipe wavefronts.  Each lane evaluates three of the twelve 1-D weights
// (the divisions are the expensive part) and the quad exchanges them by shuffle; every plane is still accumulated by
// ONE lane in the reference's order (i outer, j inner, interpolate.m:43-49), so the results stay bit-identical.
__device__ __forceinline__ void lagrange_weights3(double a, double bump, int i_lo, double* w3) {
    double t[NW];
#pragma unroll
    for (int j = 0; j < NW; j++) t[j] = a - (double)(j - IORD) + bump;
#pragma unroll
    for (int m = 0; m < 3; m++) {
        const int i = i_lo + m;
        double p = 1.0;
#pragma unroll
        for (int j = 0; j < NW; j++)
            if (j != i) p = p * t[j] / (double)(j - i);
        w3[m] = p;
    }
}

__device__ __forceinline__ void make_stencil_quad(double x, double y, double dx, int nx, double bump, int q, int quad_base,
                                                  Stencil& s) {
    // interpolate.m:21-31 (every lane of the quad computes the same reduced coordinates)
    const double xl = matlab_mod(x / dx, (double)nx);
    const double yl = matlab_mod(y / dx, (double)nx);
    const double fx = floor(xl), fy = floor(yl);
    const double ax = 1.0 + xl - (1.0 + fx);
    const double ay = 1.0 + yl - (1.0 + fy);
    double mine[3];
    // lanes 0,1: wx[0..2], wx[3..5];  lanes 2,3: wy[0..2], wy[3..5]
    lagrange_weights3(q < 2 ? ax : ay, bump, (q & 1) * 3, mine);
#pragma unroll
    for (int i = 0; i < NW; i++) {
        s.wx[i] = __shfl_sync(0xffffffffu, mine[i % 3], quad_base + i / 3);
        s.wy[i] = __shfl_sync(0xffffffffu, mine[i % 3], quad_base + 2 + i / 3);
    }
    const int i0 = (int)fx, j0 = (int)fy;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        int a = (i0 + i - IORD) % nx; if (a < 0) a += nx;
        int b = (j0 + i - IORD) % nx; if (b < 0) b += nx;
        s.ig[i] = a; s.jg[i] = b;
    }
}

// lane q accumulates planes c0 = 2q and c1 = 2q+1 (those below NPL) over the 36 nodes
template <int NPL>
__device__ __forceinline__ void gather_pair(const double* __restrict__ grid, int nx, const Stencil& s, int q, double& F0, double& F1) {
    F0 = 0.0; F1 = 0.0;
    const int c0 = 2 * q;
    const bool on0 = c0 < NPL, on1 = c0 + 1 < NPL;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        const double* row = grid + (size_t)s.ig[i] * nx * NPL;
#pragma unroll
        for (int j = 0; j < NW; j++) {
            const double w = s.wx[i] * s.wy[j];
            const double* node = row + (size_t)s.jg[j] * NPL + c0;
            double v0 = 0.0, v1 = 0.0;
            if constexpr (NPL % 2 == 0) {
                if (on0) { const double2 v = __ldg(reinterpret_cast<const double2*>(node)); v0 = v.x; v1 = v.y; }
            } else {
                if (on0) v0 = __ldg(node);
                if (on1) v1 = __ldg(node + 1);
            }
            F0 = F0 + w * v0;
            F1 = F1 + w * v1;
        }
    }
}

// both frames of interpolate_U.m:5-17 in one sweep over the 36 nodes: the weight product is formed once per node and the
// two frames' loads are issued together; each frame's plane is still accumulated by one lane in the reference's order
template <int NPL>
__device__ __forceinline__ void gather_pair2(const double* __restrict__ grid, const double* __restrict__ grid2, int nx,
                                             const Stencil& s, int q, double& F0, double& F1, double& G0, double& G1) {
    F0 = 0.0; F1 = 0.0; G0 = 0.0; G1 = 0.0;
    const int c0 = 2 * q;
    const bool on0 = c0 < NPL, on1 = c0 + 1 < NPL;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        const size_t rowoff = (size_t)s.ig[i] * nx * NPL;
#pragma unroll
        for (int j = 0; j < NW; j++) {
            const double w = s.wx[i] * s.wy[j];
            const size_t off = rowoff + (size_t)s.jg[j] * NPL + c0;
            double v0 = 0.0, v1 = 0.0, g0 = 0.0, g1 = 0.0;
            if constexpr (NPL % 2 == 0) {
                if (on0) {
                    const double2 v = __ldg(reinterpret_cast<const double2*>(grid + off));
                    const double2 g = __ldg(reinterpret_cast<const double2*>(grid2 + off));
                    v0 = v.x; v1 = v.y; g0 = g.x; g1 = g.y;
                }
            } else {
                if (on0) { v0 = __ldg(grid + off); g0 = __ldg(grid2 + off); }
                if (on1) { v1 = __ldg(grid + off + 1); g1 = __ldg(grid2 + off + 1); }
            }
            F0 = F0 + w * v0;
            F1 = F1 + w * v1;
            G0 = G0 + w * g0;
            G1 = G1 + w * g1;
        }
    }
}

// TWO = a second frame is gathered with the same weights (interpolate_U.m).  The steady instantiation must not carry the
// second gather: with a run-time branch ptxas hoists both frames' 72 loads and the kernel lands at 252 registers
// (2 blocks per SM instead of 5; 0.27 -> 0.43 ms at C2).
#ifndef SWRT_LAG_TWO_MINB
#define SWRT_LAG_TWO_MINB 4     /* two-frame kernels: 128 registers; 0 / 1 / 3 / 4 give 2.20 / 1.56 / 2.23 / 2.62e9 packet-steps/s at C3 */
#endif
#ifndef SWRT_LAG_MINB
#define SWRT_LAG_MINB 0     /* 0 = unspecified: ptxas then settles at 96 (leapfrog) / 64 (eval) registers */
#endif
template <int NPL, bool TWO>
__global__ void __launch_bounds__(128, TWO ? SWRT_LAG_TWO_MINB : SWRT_LAG_MINB) lagrange_eval_kernel(const LagArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> 2;
    const int lane = threadIdx.x & 31, q = lane & 3, qb = lane & ~3;
    const long long pc = p < a.n ? p : a.n - 1;          // idle quads of the last warp still take part in the shuffles
    Stencil s;
    make_stencil_quad(a.xin[pc], a.yin[pc], a.dx, a.nx, a.bump, q, qb, s);
    double F0, F1;
    if constexpr (TWO) {   // interpolate_U.m:19-23: interpolate BOTH frames, then (1 - alpha)*F1 + alpha*F2
        double G0, G1;
        gather_pair2<NPL>(a.grid, a.grid2, a.nx, s, q, F0, F1, G0, G1);
        F0 = (1.0 - a.alpha) * F0 + a.alpha * G0;
        F1 = (1.0 - a.alpha) * F1 + a.alpha * G1;
    } else {
        gather_pair<NPL>(a.grid, a.nx, s, q, F0, F1);
    }
    if (p < a.n) {
        if (2 * q < NPL && a.out[2 * q]) a.out[2 * q][p] = F0;
        if (2 * q + 1 < NPL && a.out[2 * q + 1]) a.out[2 * q + 1][p] = F1;
    }
}

// swrt_ode23 / swrt_ode23_packets' evaluation at the view's alpha of `stage`: the frames lag_frames picks for that alpha
// (one grid at alpha 0 or 1, else both blended as above), per packet.  gather_pair / gather_pair2 do no shuffles, so the
// quads of a warp may take different branches; idle packets join make_stencil_quad and store nothing.
template <int NPL, class View>
__global__ void __launch_bounds__(128, SWRT_LAG_TWO_MINB) lagrange_eval_ode23_kernel(const LagArgs a, const View v, int stage) {
    if (v.done()) return;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> 2;
    const int lane = threadIdx.x & 31, q = lane & 3, qb = lane & ~3;
    const long long pc = p < a.n ? p : a.n - 1;
    const double al = a.grid2 ? v.alpha(stage, pc) : 0.0;
    Stencil st;
    make_stencil_quad(a.xin[pc], a.yin[pc], a.dx, a.nx, a.bump, q, qb, st);
    if (v.idle(pc)) return;
    double F0, F1;
    if (al == 0.0 || al == 1.0) {
        gather_pair<NPL>(al == 0.0 ? a.grid : a.grid2, a.nx, st, q, F0, F1);
    } else {
        double G0, G1;
        gather_pair2<NPL>(a.grid, a.grid2, a.nx, st, q, F0, F1, G0, G1);
        F0 = (1.0 - al) * F0 + al * G0;
        F1 = (1.0 - al) * F1 + al * G1;
    }
    if (p < a.n) {
        if (2 * q < NPL && a.out[2 * q]) a.out[2 * q][p] = F0;
        if (2 * q + 1 < NPL && a.out[2 * q + 1]) a.out[2 * q + 1][p] = F1;
    }
}

// ode_symplectic.m:13-21,33-37 with scheme.U / grad_U = six Lagrange interpolations at x1
template <int NPL, bool TWO>
__global__ void __launch_bounds__(128, TWO ? SWRT_LAG_TWO_MINB : SWRT_LAG_MINB) lagrange_leapfrog_kernel(const LagArgs a) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long p = t >> 2;
    const int lane = threadIdx.x & 31, q = lane & 3, qb = lane & ~3;
    const long long pc = p < a.n ? p : a.n - 1;
    double x = a.x[pc], y = a.y[pc], k = a.k[pc], l = a.l[pc];
    const double f2 = a.f * a.f, h = 0.5 * a.dt;
    for (int st = 0; st < a.nsteps; st++) {
        double om = sqrt(f2 + a.gH * (k * k + l * l));
        x = x + h * (a.gH * k / om);
        y = y + h * (a.gH * l / om);
        Stencil s;
        make_stencil_quad(x, y, a.dx, a.nx, a.bump, q, qb, s);
        double F0, F1;
        if constexpr (TWO) {
            double G0, G1;
            const double al = a.alpha + (double)(a.j0 + st) * a.dalpha;     // the host's alpha0 + j*dalpha, same doubles
            gather_pair2<NPL>(a.grid, a.grid2, a.nx, s, q, F0, F1, G0, G1);
            F0 = (1.0 - al) * F0 + al * G0;
            F1 = (1.0 - al) * F1 + al * G1;
        } else {
            gather_pair<NPL>(a.grid + (size_t)st * a.gstride, a.nx, s, q, F0, F1);
        }
        // every lane needs all six planes for the kick: lane 0 holds (u,v), lane 1 (ux,uy), lane 2 (vx,vy)
        double F[6];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            F[2 * c] = __shfl_sync(0xffffffffu, F0, qb + c);
            F[2 * c + 1] = __shfl_sync(0xffffffffu, F1, qb + c);
        }
        x = x + a.dt * F[0];
        y = y + a.dt * F[1];
        const double k0 = k, l0 = l;
        k = k0 - a.dt * (F[2] * k0 + F[4] * l0);
        l = l0 - a.dt * (F[3] * k0 + F[5] * l0);
        om = sqrt(f2 + a.gH * (k * k + l * l));
        x = x + h * (a.gH * k / om);
        y = y + h * (a.gH * l / om);
    }
    if (p < a.n && q == 0) { a.x[p] = x; a.y[p] = y; a.k[p] = k; a.l[p] = l; }
}

// One RK4 position stage of step_packet(.m:41-51) / step_packet_xka(.m:42-52): interpolate the
// node-wise fields  U.u + C.x  and  U.v + C.y.  Without H the group velocity is a per-packet scalar
// added at every node (step_packet.m:37,41); with H it is a field (cg_sw.m:15-26).
template <int NPL, bool XKA>
__device__ __forceinline__ void velocity_stage(const double* __restrict__ grid, int nx, const Stencil& s, double k,
                                               double l, double K2, double C02, double f2, double Cx, double Cy,
                                               double& vx, double& vy) {
    vx = 0.0; vy = 0.0;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        const double* row = grid + (size_t)s.ig[i] * nx * NPL;
#pragma unroll
        for (int j = 0; j < NW; j++) {
            const double w = s.wx[i] * s.wy[j];
            const double* node = row + (size_t)s.jg[j] * NPL;
            double u = __ldg(node), v = __ldg(node + 1);
            if constexpr (XKA) {
                double gH = C02 * __ldg(node + 6);
                double om = sqrt(f2 + gH * K2);
                vx = vx + w * (u + gH * k / om);
                vy = vy + w * (v + gH * l / om);
            } else {
                vx = vx + w * (u + Cx);
                vy = vy + w * (v + Cy);
            }
        }
    }
}

template <int NPL, bool XKA>
__global__ void __launch_bounds__(128) lagrange_rk4_kernel(const LagArgs a) {
    long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.n) return;
    double x = a.x[p], y = a.y[p], k = a.k[p], l = a.l[p];
    double amp = XKA ? a.a[p] : 0.0;
    const double f = a.f, f2 = f * f, C02 = a.C0 * a.C0, dt = a.dt;
    for (int st = 0; st < a.nsteps; st++) {
        const double* __restrict__ grid = a.grid + (size_t)st * a.gstride;    // fused run on pre-blended frames
        const double K2 = k * k + l * l;
        double Cx = 0.0, Cy = 0.0;
        if (!XKA) {   // cg_sw.m:19-26 with scalar gH
            double om = sqrt(f2 + C02 * K2);
            Cx = C02 * k / om; Cy = C02 * l / om;
        }
        Stencil s;
        double vx, vy;
        make_stencil(x, y, a.dx, a.dx, a.nx, a.nx, a.bump, s);
        // gradients at the OLD position for step_packet (step_packet.m:58-61)
        double g[4] = {0, 0, 0, 0};
        if (!XKA) {
            double F[NPL];
            gather_planes<NPL>(grid, a.nx, s, F);
            g[0] = F[2]; g[1] = F[3]; g[2] = F[4]; g[3] = F[5];
        }
        velocity_stage<NPL, XKA>(grid, a.nx, s, k, l, K2, C02, f2, Cx, Cy, vx, vy);
        const double x1 = dt * vx, y1 = dt * vy;
        make_stencil(x + x1 / 2, y + y1 / 2, a.dx, a.dx, a.nx, a.nx, a.bump, s);
        velocity_stage<NPL, XKA>(grid, a.nx, s, k, l, K2, C02, f2, Cx, Cy, vx, vy);
        const double x2 = dt * vx, y2 = dt * vy;
        make_stencil(x + x2 / 2, y + y2 / 2, a.dx, a.dx, a.nx, a.nx, a.bump, s);
        velocity_stage<NPL, XKA>(grid, a.nx, s, k, l, K2, C02, f2, Cx, Cy, vx, vy);
        const double x3 = dt * vx, y3 = dt * vy;
        make_stencil(x + x3, y + y3, a.dx, a.dx, a.nx, a.nx, a.bump, s);
        velocity_stage<NPL, XKA>(grid, a.nx, s, k, l, K2, C02, f2, Cx, Cy, vx, vy);
        const double x4 = dt * vx, y4 = dt * vy;
        const double xn = x + (x1 + 2 * x2 + 2 * x3 + x4) / 6;
        const double yn = y + (y1 + 2 * y2 + 2 * y3 + y4) / 6;
        double oxi = 0.0, oyi = 0.0, dci = 0.0;
        if (XKA) {
            // gradients, grad(omega), div C at the NEW position (step_packet_xka.m:59-65),
            // composed node-wise exactly as cg_sw.m:22-31 forms them on the grid
            make_stencil(xn, yn, a.dx, a.dx, a.nx, a.nx, a.bump, s);
#pragma unroll
            for (int i = 0; i < NW; i++) {
                const double* row = grid + (size_t)s.ig[i] * a.nx * NPL;
#pragma unroll
                for (int j = 0; j < NW; j++) {
                    const double w = s.wx[i] * s.wy[j];
                    const double* node = row + (size_t)s.jg[j] * NPL;
                    const double u = __ldg(node), v = __ldg(node + 1);
                    g[0] = g[0] + w * __ldg(node + 2);
                    g[1] = g[1] + w * __ldg(node + 3);
                    g[2] = g[2] + w * __ldg(node + 4);
                    g[3] = g[3] + w * __ldg(node + 5);
                    const double gH = C02 * __ldg(node + (NPL > 6 ? 6 : 0));
                    const double om = sqrt(f2 + gH * K2);
                    const double cx = gH * k / om, cy = gH * l / om;
                    oxi = oxi + w * (f * K2 * v / (2 * om));
                    oyi = oyi + w * (-f * K2 * u / (2 * om));
                    dci = dci + w * ((k * f * v - l * f * u - cx * cx - cy * cy) / om);
                }
            }
        }
        // RK4 on (k,l) with the frozen matrix (step_packet.m:65-78, step_packet_xka.m:69-82)
        const double k1 = dt * (-g[0] * k - g[2] * l - oxi);
        const double l1 = dt * (-g[1] * k - g[3] * l - oyi);
        const double k2 = dt * (-g[0] * (k + k1 / 2) - g[2] * (l + l1 / 2) - oxi);
        const double l2 = dt * (-g[1] * (k + k1 / 2) - g[3] * (l + l1 / 2) - oyi);
        const double k3 = dt * (-g[0] * (k + k2 / 2) - g[2] * (l + l2 / 2) - oxi);
        const double l3 = dt * (-g[1] * (k + k2 / 2) - g[3] * (l + l2 / 2) - oyi);
        const double k4 = dt * (-g[0] * (k + k3) - g[2] * (l + l3) - oxi);
        const double l4 = dt * (-g[1] * (k + k3) - g[3] * (l + l3) - oyi);
        k = k + (k1 + 2 * k2 + 2 * k3 + k4) / 6;
        l = l + (l1 + 2 * l2 + 2 * l3 + l4) / 6;
        if (XKA) {   // wave action, step_packet_xka.m:86-91
            const double a1 = dt * (-amp * dci);
            const double a2 = dt * (-(amp + a1 / 2) * dci);
            const double a3 = dt * (-(amp + a2 / 2) * dci);
            const double a4 = dt * (-(amp + a3) * dci);
            amp = amp + (a1 + 2 * a2 + 2 * a3 + a4) / 6;
        }
        x = xn; y = yn;
    }
    a.x[p] = x; a.y[p] = y; a.k[p] = k; a.l[p] = l;
    if (XKA) a.a[p] = amp;
}

// standalone FI = interpolate(x,y,F,dx,dy): F is the caller's column-major nx x ny grid (x fastest)
__global__ void __launch_bounds__(128) interpolate_single_kernel(const double* __restrict__ F, int nx, int ny,
                                                                  const double* __restrict__ x,
                                                                  const double* __restrict__ y, long long n, double dx,
                                                                  double dy, double bump, double* __restrict__ out) {
    long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    Stencil s;
    make_stencil(x[p], y[p], dx, dy, nx, ny, bump, s);
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < NW; i++)
#pragma unroll
        for (int j = 0; j < NW; j++) acc = acc + (s.wx[i] * s.wy[j]) * __ldg(F + (size_t)s.jg[j] * nx + s.ig[i]);
    out[p] = acc;
}

struct GridPtrs { const double* p[kMaxPlanes]; };
// caller planes are column-major (x fastest): plane[ix + nx*iy]  ->  grid[(ix*nx + iy)*npl + c]
__global__ void interleave_kernel(GridPtrs src, int npl, int nx, double* __restrict__ grid) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)nx * nx * npl;
    if (idx >= total) return;
    int c = idx % npl;
    size_t node = idx / npl;
    int iy = node % nx, ix = node / nx;
    grid[idx] = src.p[c][(size_t)iy * nx + ix];
}

inline unsigned blocks_for(long long n, int bs) { return (unsigned)((n + bs - 1) / bs); }

}  // namespace

void launch_interleave_grid(const double* const* planes_dev, int npl, int nx, double* grid, cudaStream_t st) {
    GridPtrs gp{};
    for (int i = 0; i < npl; i++) gp.p[i] = planes_dev[i];
    size_t total = (size_t)nx * nx * npl;
    interleave_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(gp, npl, nx, grid);
}

cudaError_t launch_lagrange_eval(const LagArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    const unsigned nb = blocks_for(4 * a.n, 128);
    if (a.npl == 6) { if (a.grid2) lagrange_eval_kernel<6, true><<<nb, 128, 0, st>>>(a); else lagrange_eval_kernel<6, false><<<nb, 128, 0, st>>>(a); }
    else if (a.npl == 7) { if (a.grid2) lagrange_eval_kernel<7, true><<<nb, 128, 0, st>>>(a); else lagrange_eval_kernel<7, false><<<nb, 128, 0, st>>>(a); }
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

template <class View> cudaError_t launch_lagrange_eval_ode23(const LagArgs& a, const View& v, int stage, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    const unsigned nb = blocks_for(4 * a.n, 128);
    if (a.npl == 6) lagrange_eval_ode23_kernel<6><<<nb, 128, 0, st>>>(a, v, stage);
    else if (a.npl == 7) lagrange_eval_ode23_kernel<7><<<nb, 128, 0, st>>>(a, v, stage);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
template cudaError_t launch_lagrange_eval_ode23(const LagArgs&, const Ode23CtlView&, int, cudaStream_t);
template cudaError_t launch_lagrange_eval_ode23(const LagArgs&, const Ode23PktView&, int, cudaStream_t);

cudaError_t launch_lagrange_leapfrog(const LagArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    const unsigned nb = blocks_for(4 * a.n, 128);
    if (a.npl == 6) { if (a.grid2) lagrange_leapfrog_kernel<6, true><<<nb, 128, 0, st>>>(a); else lagrange_leapfrog_kernel<6, false><<<nb, 128, 0, st>>>(a); }
    else if (a.npl == 7) { if (a.grid2) lagrange_leapfrog_kernel<7, true><<<nb, 128, 0, st>>>(a); else lagrange_leapfrog_kernel<7, false><<<nb, 128, 0, st>>>(a); }
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}

cudaError_t launch_lagrange_rk4(const LagArgs& a, bool xka, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    if (xka) {
        if (a.npl != 7) return cudaErrorInvalidValue;
        lagrange_rk4_kernel<7, true><<<blocks_for(a.n, 128), 128, 0, st>>>(a);
    } else {
        if (a.npl == 6) lagrange_rk4_kernel<6, false><<<blocks_for(a.n, 128), 128, 0, st>>>(a);
        else if (a.npl == 7) lagrange_rk4_kernel<7, false><<<blocks_for(a.n, 128), 128, 0, st>>>(a);
        else return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_interpolate_single(const double* F, int nx, int ny, const double* x, const double* y, long long n,
                                      double dx, double dy, double bump, double* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    interpolate_single_kernel<<<blocks_for(n, 128), 128, 0, st>>>(F, nx, ny, x, y, n, dx, dy, bump, out);
    return cudaGetLastError();
}

}  // namespace swrt
