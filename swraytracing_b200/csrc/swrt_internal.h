// swrt_internal.h -- shared declarations between the kernels and the C-ABI layer of libswrt.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>

namespace swrt {

constexpr int kMaxPlanes = 7;          // u,v,ux,uy,vx,vy,H
constexpr int kNumSrcPlanes = 10;      // + the three psi-hat moment planes N0,N1,N2 (ids 7,8,9)
#ifndef SWRT_CONSUMER_WARPS
#define SWRT_CONSUMER_WARPS 8
#endif
constexpr int kConsumerWarps = SWRT_CONSUMER_WARPS;      // MMA warps per CTA in the spectral kernel
#ifndef SWRT_CTAS_PER_SM
#define SWRT_CTAS_PER_SM 1
#endif
constexpr int kCtasPerSm = SWRT_CTAS_PER_SM;             // independent CTAs per SM (each with its own smem ring)
constexpr int kSpecThreads = kConsumerWarps * 32;         // warp 0 lane 0 also issues the bulk copies

// ---------------------------------------------------------------------------------------------
// Packed coefficient stack ("B operand") geometry.  See DESIGN.md section 3.
//   A pass covers KYP = 4*G consecutive ky for all NPL planes: NT = NPL*G n-tiles of 8 real
//   columns (4 complex (re,im) column pairs).  One k-step covers two kx>=0 wavenumbers
//   (rows Er(kx),Ei(kx),Er(kx+1),Ei(kx+1)).  Storage order (doubles):
//       [pass][kstep][tile pair tp][lane 0..31][2]
//   so that lane reads ONE 16-byte word per pair of n-tiles and a whole chunk of KC k-steps is
//   one contiguous block that a single cp.async.bulk moves into shared memory.
// ---------------------------------------------------------------------------------------------
struct PackGeom {
    int nx, nkx, nky, kmax;
    int npl, G, NT;
    int npass;            // ceil(nky / (4G))
    int ksteps;           // k-steps per pass, padded to a multiple of kc
    int kc;               // k-steps per chunk (pipeline stage)
    int chunks_per_eval;  // npass * ksteps / kc
    int nstages;
    int lag;              // a stage is refilled `lag` chunks after warp 0 released it
    int desync_ns;        // start-up skew of warps 4..7 (0 = none)
    int atab;             // x twiddles of a step: 0 = rotated in registers inside the k-loop, 1 = tabulated in shared memory
                          //    (A fragments by LDS.64), 2 = tabulated in a per-CTA global scratch (L2), prefetched by LDG
    size_t chunk_doubles; // kc * NT * 32
    size_t total_doubles; // npass * ksteps * NT * 32
    int plane_ids[kMaxPlanes];   // which of the 7 source planes each stack plane is
};

// ---------------------------------------------------------------------------------------------
// swrt_ode23: a whole ode23 solve with the step-size controller in device memory (DESIGN.md section 11).  The stage,
// evaluation, norm, interp and accept kernels of an attempt read h, the stage alphas and `done` from here; a single-thread
// controller kernel after each attempt's norm makes reference_api.ode23's decisions.  Queued attempts after the last
// one (or after a failure) exit at once.
// ---------------------------------------------------------------------------------------------
struct Ode23Ctl {
    // per solve (set by the host before the first attempt)
    double tfinal, rtol, hmax, tmax, rh_den, htspan;   // rh_den = 0.8 * rtol^(1/3); htspan = |tspan(2) - tspan(1)|
    const double* tspan; int ntspan;                   // device copy of tspan (dense output when ntspan > 2)
    double* yout;                                      // ntspan x 4 x n rows (dense output) or null
    double* htrace; int hcap;                          // accepted step sizes (optional)
    // controller state
    double t, absh, h, tnew, hmin, err;
    double al[3];                                      // RHS alphas of stages 2..4 (t + h/2, t + 3h/4, tnew)
    double t_acc, h_acc;                               // t and h of the attempt just accepted (dense output)
    int last;                                          // this attempt lands on tfinal (the host controller's `done`)
    int nofailed;
    int accepted;                                      // the attempt just decided was accepted: interp and accept run
    int done;                                          // the solve is complete
    int status;                                        // 0, or 1 = step size below hmin (t holds where)
    int nxt, nxt_end;                                  // dense rows [nxt, nxt_end) are written after this attempt
    long long nsteps, nfailed, nfevals;
    // per solve, appended so that the fields above keep their offsets
    double tdir;                                       // +1 (tfinal >= t0) or -1 (a decreasing tspan: backward in time)
};
// a pointer-argument evaluation: the frame is chosen on the device from ctl->al[stage] as the host picks it for a value
// alpha (alpha == 0: frame 0, alpha == 1: frame 1, else the blend); frame1 / blend may be null for a steady flow
struct Ode23Sel {
    const Ode23Ctl* ctl;
    int stage;
    const void* frame1;
    const void* blend;
};
__device__ __forceinline__ bool ode23_idle(const Ode23Ctl* c) { return c->done || c->status; }
// attempts to queue before the host looks at the state again: the steps left if every step grew five-fold up to hmax
// (the most the controller allows, so a lower bound) plus a margin for rejections and slower growth
__host__ __device__ inline int ode23_batch_estimate(double tfinal, double t, double absh, double hmax) {
    double left = fabs(tfinal - t), hh = absh;
    int est = 0;
    while (left > 0.0 && est < 1024) { left -= hh < hmax ? hh : hmax; hh *= 5.0; est++; }
    const int b = est + 2 + est / 4;
    return b < 256 ? b : 256;
}

// swrt_ode23_packets: every packet under its own controller.  The state of Ode23Ctl's controller section, one entry per
// packet (SoA, n each); a kernel loads a packet's entries into a local Ode23Ctl that also carries the per-solve
// constants, applies swrt_ode23's rules to it and stores it back.
constexpr int kPktLast = 1, kPktNofailed = 2, kPktDone = 4, kPktStopped = 8;
struct Ode23Pkt {
    double *t, *absh, *h, *hmin, *tnew, *al[3], *t_acc, *h_acc;
    int* flags;                    // kPkt* bits
    int* cnt;                      // 3 x n: accepted steps, rejected steps, status (1 = stopped: step size below hmin)
    int* nxt;                      // next dense row to write
    int* report;                   // 2 x {unfinished packets, attempts to queue}: decide kernel of round r writes pair r & 1
};
__device__ __forceinline__ bool ode23_pkt_idle(const Ode23Pkt& s, long long i) { return s.flags[i] & (kPktDone | kPktStopped); }
// swrt_ode23_packets_events: up to kMaxEvents level crossings of a function of the packet state, located on each accepted
// step's ntrp23 cubic by the decide kernel (DESIGN.md section 11).  Passed by value; the arrays are per-packet SoA buffers
// of the handle (n entries per row).
constexpr int kMaxEvents = 8;
struct Ode23Ev {
    int nev, cap;                                        // events, records kept per packet
    int kind[kMaxEvents], dir[kMaxEvents], term[kMaxEvents];
    double level[kMaxEvents];
    double f, gH;                                        // SWRT_EVENT_OMEGA: omega = sqrt(f^2 + gH (k^2 + l^2))
    double* vl;                                          // nev x n: g_j at the last accepted state
    double* te;                                          // cap x n (NaN when unused)
    double* ye;                                          // cap x 4 x n (NaN when unused)
    int* ie;                                             // cap x n: 1-based event index (0 when unused)
    int* ne;                                             // n: events found (may exceed cap)
};
// swrt_ode23_packets_tspans: every packet's own tspan row, packet-contiguous (row i at tsp + i*ntspan), and the per-solve
// constants of Ode23Ctl that then differ per packet (SoA, n each), formed by the begin kernel and loaded by the decide
// kernel.  Passed by value; all null when the packets share one tspan.
struct Ode23Spans {
    const double* tsp; int ntspan;
    double *tfinal, *hmax, *tdir;
};
// the alphas of `stage` (selected, not indexed: a run-time index would move the kernel argument to local memory)
__device__ __forceinline__ const double* ode23_pkt_alpha(const Ode23Pkt& s, int stage) {
    return stage == 0 ? s.al[0] : stage == 1 ? s.al[1] : s.al[2];
}

// The controller an attempt kernel (stage, RHS, norm, accept, LAGRANGE6 evaluation) reads, one view per solve:
//   done()           nothing is left in this launch (uniform: the kernel returns at its top)
//   idle(i)          packet i is finished and writes nothing
//   h(i)             packet i's step size
//   alpha(stage, i)  packet i's flow alpha of the RHS evaluation of `stage`
//   accepted()       the accept kernel's predicate
// The host controller (swrt_bs23_*, swrt_rhs): h and the alphas as values, never idle.
struct Ode23ValView {
    double hv, al[3];
    __device__ bool done() const { return false; }
    __device__ bool idle(long long) const { return false; }
    __device__ double h(long long) const { return hv; }
    __device__ double alpha(int stage, long long) const { return stage == 0 ? al[0] : stage == 1 ? al[1] : al[2]; }
    __device__ bool accepted() const { return true; }
};
// swrt_ode23: one controller in device memory for the whole launch
struct Ode23CtlView {
    const Ode23Ctl* ctl;
    __device__ bool done() const { return ode23_idle(ctl); }
    __device__ bool idle(long long) const { return false; }
    __device__ double h(long long) const { return ctl->h; }
    __device__ double alpha(int stage, long long) const { return ctl->al[stage]; }
    __device__ bool accepted() const { return ctl->accepted; }
};
// swrt_ode23_packets: one controller per packet (its norm and accept are part of the decide kernel)
struct Ode23PktView {
    Ode23Pkt s;
    __device__ bool done() const { return false; }
    __device__ bool idle(long long i) const { return ode23_pkt_idle(s, i); }
    __device__ double h(long long i) const { return s.h[i]; }
    __device__ double alpha(int stage, long long i) const { return ode23_pkt_alpha(s, stage)[i]; }
};

PackGeom make_geom(int nx, int npl, const int* plane_ids, int mtiles, int twiddle_pref = 0);

// one source slot: complex planes on the device, [plane][ky][kx+kmax] as double2 (kx fastest)
void launch_pack(const PackGeom& g, const double2* const* planes_dev /*[kNumSrcPlanes] device ptrs (host array)*/,
                 double* stack_dev, cudaStream_t st);
void launch_psi_moments(const double2* psik, double2* n0, double2* n1, double2* n2, int nkx, int nky, cudaStream_t st);
void launch_psi_to_planes(const double2* psik, double2* const* planes /*host array of 6 dev ptrs*/,
                          int nkx, int nky, double kappa, double u_mean, cudaStream_t st);
void launch_axpby(double* out, const double* a, const double* b, double wa, double wb, size_t n,
                  cudaStream_t st);
// m blends in one launch: out[j*n + i] = (1 - al_j)*a[i] + al_j*b[i], al_j = alpha0 + (j0 + j)*dalpha, j < m
void launch_axpby_multi(double* out, const double* a, const double* b, double alpha0, double dalpha, int j0, int m, size_t n,
                        cudaStream_t st);

struct SpecArgs {
    const double* stack;
    PackGeom g;
    long long n;            // packets
    const double* xin; const double* yin;    // EVAL: positions
    double* x; double* y; double* k; double* l;   // LEAPFROG: state (in/out)
    double* out[kMaxPlanes];                  // EVAL: outputs per stack plane (may be null)
    double dx, nxd;         // grid spacing and nx as double
    double inv_nx;          // 1/nx when nx is a power of two (exact), else 0
    double f2, gH, dt;
    int nsteps;
    bool psi;               // stack = psi-hat moment planes; assemble the six planes in stage 2
    double kappa;           // psi mode: 2*pi/L
    double u_mean0, u_mean1;   // psi mode: mean shear of the two flow slots; evaluation j adds (1-al_j)*u_mean0 + al_j*u_mean1
    double alpha0, dalpha;  //   with al_j = alpha0 + (j0 + j)*dalpha (EVAL: j = 0)
    int j0;
    int nstack;             // LEAPFROG: `stack` holds nstack (= nsteps) consecutive stacks, one per fused step (a
                            //   time-dependent flow pre-blended at al_j for every step of the launch); 0/1 = one stack
    double* twid;           // atab == 2: per-CTA twiddle scratch, gridDim.x * 8 warps * ksteps * 32 doubles
    unsigned long long* trace;   // developer timeline buffer (only read when built with -DSWRT_TRACE)
    // anchored leapfrog (DESIGN.md section 3e).  anchor_transform_kernel writes the expansion blocks of every anchor cell;
    // anchored_step_kernel expands them to the packets of each anchor and steps them.
    const unsigned long long* anc_cnt;    // packets per anchor id
    const unsigned long long* anc_off;    // first entry of each anchor in anc_perm
    const long long* anc_perm;            // packet indices grouped by anchor
    double* hexp;                         // H' blocks (K2's B fragments), anc_block doubles per anchor id
    size_t anc_block;                     // npass * 2 k-steps * NT * 32
    double anc_h;                         // anchor cell width in the reduced coordinate t of reduced_turns (t in [0, 2))
    double zscale;                        // pi * kmax: z = zscale * (t - t_anchor)
    int ev;                               // anchored_step_kernel: sub-step index j of the run (mean-shear blend weight)
    Ode23Sel sel;                         // SPEC_EVAL_DEV: stack and alpha chosen from the ode23 controller
};

enum SpecMode { SPEC_EVAL = 0, SPEC_LEAPFROG = 1, SPEC_EVAL_DEV = 3 };

// anchored leapfrog: expansion order, anchor geometry and its kernels (K1 = anchor_transform_kernel, K2 = anchored_step_kernel)
constexpr int kAnchorOrders = 8;        // R: Taylor orders of e^{i kx delta} kept per anchor (two DMMA k-steps)
constexpr int kAncWarps = 4;            // warps per CTA of anchored_step_kernel (two CTAs per SM)
// anchor cell width in turns 2^-m for an nx grid, or 0 when this grid keeps the dense kernel
int anchor_log2_cells(int nx);
// H' blocks of all nanchors = 64 nx cells from the stack a.stack (one sub-step) into a.hexp
cudaError_t launch_anchor_transform(const SpecArgs& a, int nanchors, int num_sms, cudaStream_t st);
// fp64 flops one launch of it executes (pre-twiddles and weights, butterflies, pass twiddles, output scaling)
double anchor_transform_flops(const PackGeom& g);
cudaError_t launch_anchored_step(const SpecArgs& a, int nanchors, cudaStream_t st);
void launch_anchor_key(double* x, double* y, const double* k, const double* l, long long n, double dx, double nxd, double inv_nx,
                       double f2, double gH, double dt, double inv_h, int nanchors, unsigned long long* cnt, int* key,
                       unsigned long long* rank, cudaStream_t st);
void launch_anchor_scan(const unsigned long long* cnt, unsigned long long* off, int nanchors, cudaStream_t st);
void launch_anchor_scatter(const int* key, const unsigned long long* rank, const unsigned long long* off, long long* perm, long long n,
                           cudaStream_t st);

// fused step_packet / step_packet_xka in SPECTRAL mode (spectral_rk4_kernels.cu): two packed stacks share one chunk ring
struct SpecRk4Args {
    const double* stackA;   // stage evaluations: (u,v) or (u,v,H)
    const double* stackB;   // the big evaluation: six planes / the psi-hat moment planes (old position) or seven planes (new position)
    PackGeom gA, gB;
    int nstages, lag, atab, tab_ksteps;      // joint ring geometry (filled by spectral_rk4_geometry)
    uint32_t stage_bytes;
    long long n;
    double *x, *y, *k, *l, *a;
    double dx, nxd, inv_nx;
    double f, C0, dt;
    int nsteps;
    int nstack;             // > 1: one pre-blended pair of stacks per step (time-dependent flow), stored back to back
    bool psiB;              // stackB = psi-hat moment planes
    double* twid;           // per-CTA global twiddle scratch (atab == 2): gridDim.x * 8 warps * tab_ksteps * 32 doubles
    double kappa, u_mean0, u_mean1, alpha0, dalpha;
    int j0;
};
bool spectral_rk4_geometry(SpecRk4Args& a, size_t* smem_bytes);
cudaError_t launch_spectral_rk4(const SpecRk4Args& a, bool xka, int num_sms, cudaStream_t st);

// returns cudaError; grid is sized to the SM count (persistent CTAs)
cudaError_t launch_spectral(const SpecArgs& a, int mode, int mtiles, int num_sms, cudaStream_t st);
size_t spectral_smem_bytes(const PackGeom& g);

// ---------------------------------------------------------------------------------------------
// Lagrange (reference-semantics) kernels.  Grid planes are node-interleaved: F[ix][iy][NPL].
// ---------------------------------------------------------------------------------------------
struct LagArgs {
    const double* grid;     // [nx][nx][npl] doubles
    const double* grid2;    // second frame for the exact two-frame blend (eval / leapfrog kernels), else null
    double alpha;           // blend weight of grid2 (step j of a fused run: alpha + (j0 + j)*dalpha)
    double dalpha; int j0;
    size_t gstride;         // fused runs on pre-blended grids: step j reads grid + j*gstride (doubles); 0 = one grid
    int nx, npl;            // npl = 6 or 7 (7th = H)
    long long n;
    const double* xin; const double* yin;
    double* x; double* y; double* k; double* l; double* a;
    double* out[kMaxPlanes];
    double dx, bump;
    double f, gH, C0, dt;
    int nsteps;
};
void launch_interleave_grid(const double* const* planes_dev, int npl, int nx, double* grid, cudaStream_t st);
cudaError_t launch_lagrange_eval(const LagArgs& a, cudaStream_t st);
cudaError_t launch_lagrange_leapfrog(const LagArgs& a, cudaStream_t st);
cudaError_t launch_lagrange_rk4(const LagArgs& a, bool xka, cudaStream_t st);
cudaError_t launch_interpolate_single(const double* F, int nx, int ny, const double* x, const double* y,
                                      long long n, double dx, double dy, double bump, double* out, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// Elementwise / diagnostics kernels
// ---------------------------------------------------------------------------------------------
struct Rk4Args {   // spectral-mode RK4 glue (point-wise composition), all device SoA arrays
    long long n;
    double *x, *y, *k, *l, *a;
    double *xs, *ys;                 // stage positions
    double *ax, *ay;                 // accumulated (x1+2x2+2x3+x4)
    const double *u, *v, *H;         // evaluated at stage position
    const double *ux, *uy, *vx, *vy; // final evaluation
    double dt, f, C0;
    int stage; bool xka;
};
void launch_rk4_stage(const Rk4Args& a, cudaStream_t st);
void launch_rk4_final(const Rk4Args& a, cudaStream_t st);
// RHS of the planes e6 at (k, l) into fj[0..3], skipped for the view's idle packets.  With e1 set (swrt_ode23_packets,
// SPECTRAL, two frames) e6 holds the planes at alpha 0 and e1 at alpha 1, and each packet blends them at its alpha of
// `stage`, in place in e6.
template <class View>
void launch_rhs(const View& v, int stage, long long n, const double* k, const double* l, const double* const* e6,
                const double* const* e1, double f, double gH, double cgfac, double* const fj[4], cudaStream_t st);
void launch_omega(long long n, const double* k, const double* l, const double* u, const double* v,
                  double f, double gH, double* omega, double* Omega_abs, cudaStream_t st);
void launch_hist(long long n, const double* w, const double* edges_dev, int nedges,
                 unsigned long long* counts_dev, cudaStream_t st);
void launch_ideal_hist(long long npts, const double* u, const double* v, const double* kvx, const double* kvy, int nang,
                       double omega0, const double* edges_dev, int nedges, unsigned long long* counts_dev, cudaStream_t st);
// swrt_packet_quantity / swrt_hist2: the packet arrays a quantity SWRT_Q_* is computed from (om / Om as compute_omega
// filled them; only the arrays the requested quantities read need be set)
struct PktQ { const double *x, *y, *k, *l, *om, *Om; double L; };
void launch_packet_quantity(long long n, int q, const PktQ& p, double* out, cudaStream_t st);
// histcounts2 of (qx, qy) into counts_dev ((nxe-1)*(nye-1) u64, column-major, added to); edges_dev = xedges then yedges.
// Per-CTA shared-memory counters when they fit the opt-in shared memory, else global atomics.  Returns the launch error.
cudaError_t launch_hist2(long long n, int qx, int qy, const PktQ& p, const double* edges_dev, int nxe, int nye,
                         unsigned long long* counts_dev, cudaStream_t st);
// swrt_weight_scale / swrt_hist2_sums: the weight kinds SWRT_W_* of one call, computed from PktQ's k, l, om and a.  The
// scale exponents live on the device as E + kScaleBias (0: no finite non-zero weight, E = 0) so that a zeroed word is the
// identity of the int32 MAX the kernel and a multi-device all-reduce apply.
struct WeightKinds { int n; int kind[4]; };            // 4 = SWRT_MAX_WEIGHTS
constexpr int kScaleBias = 1100;
// atomicMax of every kind's biased exponent into exp_dev[0..nw) (zeroed by the caller)
void launch_weight_scale(long long n, const WeightKinds& w, const PktQ& p, const double* a, int* exp_dev, cudaStream_t st);
// the fixed-point digits of each kind's weights, per bin of (qx, qy), added to acc_dev (4 int64 per (bin, kind), layout of
// swrt_hist2_sums' acc) with the exponents exp_dev; counts_dev (may be null) gets swrt_hist2's counts.  Global atomics only.
cudaError_t launch_hist2_sums(long long n, int qx, int qy, const PktQ& p, const double* a, const WeightKinds& w,
                              const int* exp_dev, const double* edges_dev, int nxe, int nye, long long* acc_dev,
                              unsigned long long* counts_dev, cudaStream_t st);
void launch_diag(long long n, const double* x, const double* y, const double* k, const double* l, const double* a,
                 const double* omega, const double* Omega_abs, double* out8_dev, cudaStream_t st);
void launch_fill(double* p, double v, long long n, cudaStream_t st);
double gather_probe(size_t table_bytes, int iters, int reps, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// NUFFT mode (type-2 non-uniform FFT evaluation of the same Fourier series; nufft_kernels.cu)
// ---------------------------------------------------------------------------------------------
constexpr int kNufftW = 18;             // ES-kernel width in fine-grid points (16 gives 2e-12 on the gradients at 512^2, 18 gives 1.4e-13)
constexpr double kNufftSigma = 2.0;     // oversampling: nf = 2 nx
constexpr double kNufftBeta = 2.30 * kNufftW;
struct NufftArgs {
    const double2* grid;    // (u,v) fine grid, [iy*nf + ix]
    const double* hgrid;    // optional (u,v,H,0) fine grid, 4 doubles per node, same indexing (flows that carry H)
    size_t gstride, hstride;   // fused runs on pre-blended fine grids: step j reads grid + j*gstride (double2) /
                               // hgrid + j*hstride (doubles); 0 = one grid for every step
    int nf;
    long long n;
    const double* xin; const double* yin;
    double* x; double* y; double* k; double* l; double* a;
    double* out[7];
    double dx, nxd, beta, dscale;       // dscale = -sigma / (dx * w/2): d/dx of the kernel argument
    double f2, gH, dt;
    double f, C0;                       // RK4 steppers (step_packet / step_packet_xka)
    int nsteps;
};
void launch_nufft_spread(const double2* half, int nx, int nf, const double* invphi_dev, double2* full, cudaStream_t st);
void launch_nufft_store(const double2* full, int nf, int c, int stride, double* grid2, cudaStream_t st);
cudaError_t launch_nufft_eval(const NufftArgs& a, cudaStream_t st);
cudaError_t launch_nufft_leapfrog(const NufftArgs& a, cudaStream_t st);
cudaError_t launch_nufft_rk4(const NufftArgs& a, bool xka, cudaStream_t st);

struct Bs23Args {          // ode23 work arrays, component order x,y,k,l
    long long n;
    double* y[4];          // the packet state itself
    double* yt[4];         // stage state / ynew
    double* f[4][4];       // f1..f4
};
// the attempt kernels for the views of the host controller (Ode23ValView), swrt_ode23 (Ode23CtlView) and, for the stage,
// RHS and LAGRANGE6 evaluation, swrt_ode23_packets (Ode23PktView)
template <class View> void launch_bs23_stage(const Bs23Args& a, const View& v, int stage, cudaStream_t st);
// atomicMax of the error norm into `out`, which the caller has zeroed; MODE 1: the scale norm of the initial step
template <int MODE, class View>
void launch_bs23_norm(const Bs23Args& a, const View& v, double thr, unsigned long long* out, cudaStream_t st);
template <class View> void launch_bs23_accept(const Bs23Args& a, const View& v, cudaStream_t st);
template <class View> cudaError_t launch_lagrange_eval_ode23(const LagArgs& a, const View& v, int stage, cudaStream_t st);
void launch_bs23_interp(const Bs23Args& a, const double w[4], double* const out[4], cudaStream_t st);

void launch_ode23_init(Ode23Ctl* ctl, unsigned long long* norm, cudaStream_t st);
void launch_ode23_control(Ode23Ctl* ctl, unsigned long long* norm, cudaStream_t st);
void launch_bs23_interp_dev(const Bs23Args& a, const Ode23Ctl* ctl, cudaStream_t st);
// out = (1 - al)*a + al*b with al = ctl->al[stage], skipped when al is 0 or 1 (the evaluation then reads a frame itself)
void launch_axpby_dev(double* out, const double* a, const double* b, const Ode23Ctl* ctl, int stage, size_t n, cudaStream_t st);
cudaError_t launch_spectral_eval_dev(const SpecArgs& a, int num_sms, cudaStream_t st);     // a.sel set
cudaError_t launch_nufft_eval_dev(const NufftArgs& a, const Ode23Sel& sel, cudaStream_t st);
// swrt_ode23_packets: `k` holds the per-solve constants (controller section zero, t = t0).  begin: the rh norm and the
// initial step of every packet from f1; decide: each packet's norm, controller, dense rows and accept, as swrt_ode23's
// kernels with the packet's own state.  With ev set, begin also seeds the event values and clears the records, and decide
// locates and records the events of every accepted step and applies a terminal stop.  With sp set (no events), every
// packet's tfinal, tdir, hmax, htspan, t0 and tspan come from its own row of sp.tsp instead of k.
// swrt_ode23_packets_tspans: col (n x ntspan column-major) to packet-contiguous rows, s.al[0] = t0/tmax, flags cleared
void launch_ode23_pkt_rows(long long n, int ntspan, const double* col, double* rows, const Ode23Pkt& s, double tmax,
                           cudaStream_t st);
void launch_ode23_pkt_begin(const Bs23Args& a, const Ode23Pkt& s, const Ode23Ctl& k, double thr, const Ode23Ev* ev,
                            const Ode23Spans* sp, cudaStream_t st);
void launch_ode23_pkt_decide(const Bs23Args& a, const Ode23Pkt& s, const Ode23Ctl& k, double thr, int round, const Ode23Ev* ev,
                             const Ode23Spans* sp, cudaStream_t st);
cudaError_t launch_nufft_eval_pkt(const NufftArgs& a, const double2* grid1, const Ode23Pkt& s, int stage, cudaStream_t st);
// (rtol/err)^(1/3) as glibc's correctly rounded-in-practice pow gives it (host and device, misc_kernels.cu)
__host__ __device__ double pow_third(double x);

}  // namespace swrt
