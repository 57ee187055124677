/* swrt.h -- C ABI of libswrt.so: B200-native engine for SWRaytracing's packet hot path.
 *
 * The reference (ndefilippis/SWRaytracing) is MATLAB and has no FFI; its callers are MATLAB
 * scripts that invoke a handful of functions by name.  Each entry point below replaces one of
 * those function-level interfaces (cited as file:line relative to the reference tree); the MEX
 * gateway (matlab/swrt_mex.c) and the Python ctypes mirror (swraytracing_b200/engine.py) bind
 * exactly these symbols.  See INTEGRATION.md for the reference-side stubs.
 *
 * Conventions
 *   - all arrays are caller-owned HOST pointers unless the name says _dev; fp64; MATLAB
 *     column-major; complex data as separate real/imag arrays (Octave's MEX API is
 *     non-interleaved);
 *   - every function returns 0 on success, <0 on error; swrt_last_error() gives the message;
 *     nothing throws or longjmps; no caller pointer is kept after return;
 *   - one host thread drives a handle; a handle owns swrt_params.ngpu CUDA devices (default 1) and the
 *     device-resident SoA packet state (x,y,k,l,a) plus the flow-coefficient stacks.  With ngpu > 1 the
 *     packets are sharded in contiguous index ranges over the devices device .. device+ngpu-1, the flow
 *     is replicated on each, every call below keeps its meaning for the WHOLE ensemble, and the only
 *     exchanges are NCCL all-reduces (single-process ncclCommInitAll communicator) of the u64 histogram
 *     counts, the diagnostic scalars and the ode23 error norm.  The caller is one MATLAB / Octave /
 *     Python process (qgsw_raytrace.m:121-150 runs the whole loop in one interpreter);
 *   - there is NO CPU fallback: without a CUDA device every call fails with SWRT_ERR_CUDA.
 */
#ifndef SWRT_H
#define SWRT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWRT_VERSION 200

/* error codes */
#define SWRT_OK            0
#define SWRT_ERR_ARG      -1   /* bad argument (null pointer, size mismatch, bad enum) */
#define SWRT_ERR_STATE    -2   /* call order (no flow set, no packets set, wrong mode) */
#define SWRT_ERR_CUDA     -3   /* CUDA runtime / no device */
#define SWRT_ERR_ALLOC    -4   /* out of device or host memory */
#define SWRT_ERR_NCCL     -5

/* field-evaluation mode */
#define SWRT_MODE_SPECTRAL  0  /* exact Fourier-series sum (dense DMMA contraction)            */
#define SWRT_MODE_LAGRANGE6 1  /* the reference's 6x6 Lagrange stencil, interpolate.m:12-49     */
#define SWRT_MODE_NUFFT     2  /* the SAME exact Fourier series as SPECTRAL (<= 1e-12 of max|plane|), evaluated as a
                                  type-2 non-uniform FFT: oversampled cuFFT grid of u,v per frame (setup) + an 18x18
                                  kernel gather per evaluation, gradients from the kernel's analytic derivative (= the
                                  spectral derivatives of SpectralScheme.m:20-23 / grid_U.m:6-9).  Cost independent of
                                  nx.  An H plane (step_packet_xka) rides on a second fine grid.  The ux,uy,vx,vy planes
                                  handed to swrt_set_flow_planes_spectral / swrt_set_flow_grid are NOT used in this mode:
                                  the gradients are always the spectral derivatives of the u and v supplied.      */

/* integrator */
#define SWRT_SCHEME_LEAPFROG   0  /* ode_symplectic.m:13-21,33-37                               */
#define SWRT_SCHEME_RK4_PACKET 1  /* ray_trace_sw/step_packet.m:37-78                           */
#define SWRT_SCHEME_RK4_XKA    2  /* ray_trace_sw/step_packet_xka.m:38-91 (+ cg_sw.m:15-31)     */

/* swrt_params.flags */
#define SWRT_FLAG_RHS_GH    1  /* odefun group velocity gH*k/omega (SW_zero_background_raytracing.m:182-184,
                                  initialize_raytracing :134-145) instead of Cg*k/omega (qgsw_raytrace.m:262) */

/* histogram kind */
#define SWRT_HIST_INTRINSIC 0  /* omega = sqrt(f^2 + gH K^2), analysis/load_data.m:33           */
#define SWRT_HIST_ABSOLUTE  1  /* Omega = omega + U.k, symplectic_full_fourier.m:41,55          */

typedef struct swrt_handle swrt_handle;

typedef struct swrt_params {
    int32_t nx;        /* grid size (even); spectral arrays are (nx-1) x (nx/2), g2k.m:5-9      */
    int32_t mode;      /* SWRT_MODE_*                                                           */
    int32_t device;    /* CUDA device ordinal                                                   */
    int32_t flags;     /* SWRT_FLAG_* bits (0 = the qgsw_raytrace.m conventions)                  */
    double  L;         /* domain side; dx = L/nx (qgsw_raytrace.m:13-14)                        */
    double  f;         /* Coriolis parameter                                                    */
    double  gH;        /* Cg^2 = C0^2 (ode_symplectic.m:10-11)                                  */
    double  bump;      /* Lagrange "bump": 1e-13 (ray_trace_sw/interpolate.m:13) or 1e-10 (qg_flow_ray_trace/interpolate.m:13 -- the
                          copy interpolate_U.m and the QG drivers' odefun run beside -- and interpolate_par.m:13) */
    int32_t ngpu;      /* devices device .. device+ngpu-1 share the packets (0 or 1 = one device)  */
    int32_t reserved;  /* must be 0                                                             */
} swrt_params;

/* ---- lifetime ----------------------------------------------------------------------------- */
int  swrt_version(void);
int  swrt_device_count(void);
int  swrt_create(const swrt_params* p, swrt_handle** h);
int  swrt_destroy(swrt_handle* h);
/* message of the last failure on this handle (h may be NULL: last failure of swrt_create) */
const char* swrt_last_error(const swrt_handle* h);

/* ---- background flow (slots 0 and 1 = the two time frames of interpolate_U.m:5-17) --------- */
/* psi-hat in g2k layout; builds u,v,ux,uy,vx,vy = SpectralScheme.m:18-25 / grid_U.m:3-9 with
 * wavenumbers kappa*kx, kappa*ky (kappa = 2*pi/L) and adds u_mean to u (grid_U.m:11).          */
int swrt_set_flow_spectral(swrt_handle* h, int slot, const double* psik_re, const double* psik_im,
                           int nkx, int nky, double u_mean);
/* caller-supplied coefficient planes in the order u,v,ux,uy,vx,vy[,H]; nplanes = 6 or 7.
 * Plane 7 holds the coefficients of H = 1 + eta_g (raytrace_sw.m:44-45), mean included.        */
int swrt_set_flow_planes_spectral(swrt_handle* h, int slot, const double* const* planes_re,
                                  const double* const* planes_im, int nplanes, int nkx, int nky);
/* gridded planes nx x nx (column-major, x fastest) = grid_U.m:11-17 output / SpectralScheme
 * fields; H may be NULL.  In SPECTRAL mode the grids are transformed with g2k on the device.   */
int swrt_set_flow_grid(swrt_handle* h, int slot, const double* u, const double* v,
                       const double* ux, const double* uy, const double* vx, const double* vy,
                       const double* H, int nx);

/* ---- packets ------------------------------------------------------------------------------ */
int swrt_set_packets(swrt_handle* h, int64_t n, const double* x, const double* y,
                     const double* k, const double* l, const double* a /* may be NULL -> 1 */);
int swrt_get_packets(swrt_handle* h, double* x, double* y, double* k, double* l,
                     double* a /* may be NULL */);
int64_t swrt_num_packets(const swrt_handle* h);
/* devices behind the handle, and shard i's device ordinal and packet range [lo, lo+n) (any pointer may be NULL) */
int swrt_num_devices(const swrt_handle* h);
int swrt_shard_info(const swrt_handle* h, int i, int* device, int64_t* lo, int64_t* n);
/* device-resident SoA buffers (for callers that already live on the GPU, e.g. torch) */
int swrt_packets_alloc_dev(swrt_handle* h, int64_t n);
int swrt_packets_dev(swrt_handle* h, double** x, double** y, double** k, double** l, double** a);

/* ---- evaluation --------------------------------------------------------------------------- */
/* U,V,Ux,Uy,Vx,Vy at the current packet positions, flow = (1-alpha)*slot0 + alpha*slot1
 * (interpolate_U.m:19-23; SpectralScheme.U / grad_U, SpectralScheme.m:45-68).  Any output
 * pointer may be NULL.  If slot 1 is unset alpha must be 0.                                    */
int swrt_eval(swrt_handle* h, double alpha, double* U, double* V, double* Ux, double* Uy,
              double* Vx, double* Vy);
/* the same at caller-given positions (n host doubles each); does not touch the packet state.  */
int swrt_eval_at(swrt_handle* h, double alpha, int64_t n, const double* x, const double* y,
                 double* U, double* V, double* Ux, double* Uy, double* Vx, double* Vy, double* H);
/* odefun of qgsw_raytrace.m:259-265: dx/dt = U + Cg k/omega, dk/dt = -(grad U)^T k             */
int swrt_rhs(swrt_handle* h, double alpha, double* dxdt, double* dydt, double* dkdt, double* dldt);
/* standalone FI = interpolate(x,y,F,dx,dy) (interpolate.m:1-50): one nx x ny grid, n points.   */
int swrt_interpolate(int device, const double* x, const double* y, int64_t n, const double* F,
                     int nx, int ny, double dx, double dy, double bump, double* FI);

/* ---- stepping ----------------------------------------------------------------------------- */
/* nsteps fused steps of the chosen scheme; step j evaluates the flow at alpha0 + j*dalpha.    */
int swrt_step(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha);
/* the same launches without the host wait (swrt_step returns when the kernels are done; this returns when they are
 * queued): host work of the previous diagnostic interval overlaps the kernel.  swrt_synchronize completes it.   */
int swrt_step_async(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha);
/* The reference's integrators take HOST arrays and return HOST arrays (ode_symplectic.m:1-4: x0,k0 in, x,k out;
 * step_packet.m:1 / step_packet_xka.m:1: P in, Pout out).  swrt_step_host is that call shape in one entry point:
 * swrt_set_packets(n, x,y,k,l,a) + swrt_step(scheme, dt, nsteps, alpha0, dalpha) + swrt_get_packets(xo,yo,ko,lo,ao),
 * with identical results, but pipelined over packet chunks: the buffers may be ordinary pageable memory, they are
 * staged through an internal pinned ring by helper threads, and chunk i computes while chunk i+1 uploads and chunk
 * i-1 downloads.  Output pointers may alias the inputs; a / ao may be NULL (a = 1).  The device keeps the final
 * packets, as after swrt_set_packets + swrt_step.                                                            */
int swrt_step_host(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha, int64_t n,
                   const double* x, const double* y, const double* k, const double* l, const double* a,
                   double* xo, double* yo, double* ko, double* lo, double* ao);

/* ---- ode23 (Bogacki-Shampine 3(2), MATLAB builtin called by qgsw_raytrace.m:149 and
 * qg2layersw_raytrace.m:195 on y = [x;y;k;l]) -- device building blocks.  The HOST owns the step-size
 * controller (swraytracing_b200/reference_api.py: ode23) so that a multi-GPU host can MAX-all-reduce
 * the error norm, which in the reference couples all packets.  alpha = t/tmax per stage.
 *   begin:   f1 = odefun(alpha, y); rh = max_i |f1_i| / max(|y_i|, threshold)
 *   attempt: stages 2,3, ynew, f4; err = max_i |(f*E)_i| / max(|y_i|, |ynew_i|, threshold)
 *   accept:  y <- ynew, f1 <- f4 (first-same-as-last)                                           */
int swrt_bs23_begin(swrt_handle* h, double alpha, double threshold, double* rh_norm);
int swrt_bs23_attempt(swrt_handle* h, double hstep, const double alpha[3], double threshold, double* err_norm);
int swrt_bs23_accept(swrt_handle* h);
/* dense output of the LAST attempted step (MATLAB ntrp23, used by ode23 when tspan lists output times:
 * SW_zero_background_raytracing.m:73-78): y(t + s*hstep) = y + hstep * [f1 f2 f3 f4] * BI * [s; s^2; s^3],
 * BI = [1 -4/3 5/9; 0 1 -2/3; 0 4/3 -8/9; 0 -1 1].  Call between attempt and accept; s in (0, 1].     */
int swrt_bs23_interp(swrt_handle* h, double hstep, double s, double* x, double* y, double* k, double* l);
/* [~, Y] = ode23(odefun, tspan, [x;y;k;l]) on the resident packets (qgsw_raytrace.m:143-150,
 * SW_zero_background_raytracing.m:73-78) in one call, the step-size controller on the device: the decisions of
 * reference_api.ode23 (MATLAB's ode23 with MaxStep 0.1*|tf - t0|).  alpha = t/tmax (tmax = 0: steady flow, slot 0).
 * ntspan >= 2; when ntspan > 2, Y (ntspan x 4 x n, host, may be NULL) receives the state at every tspan entry (ntrp23
 * dense output).  A decreasing tspan (tspan[end] < tspan[0]) integrates backward in time, as MATLAB's ode23 does: every
 * step is h = -absh; an entry that steps against the direction from tspan[0] to tspan[end] is SWRT_ERR_ARG (equal
 * neighbours are allowed).  stats[0..3] = accepted steps, rejected steps, RHS evaluations, host waits.  h_trace (may be
 * NULL) receives up to h_cap accepted step sizes, signed (negative when integrating backward).  SWRT_ERR_STATE when the step size falls below 16*eps(t) (a packet blew
 * up; the message names t); the packets are then those of the last accepted step.                               */
int swrt_ode23(swrt_handle* h, const double* tspan, int ntspan, double tmax, double rtol, double atol, double* Y,
               int64_t stats[4], double* h_trace, int h_cap);
/* [~, Y] = ode23(odefun_i, tspan, y_i) for every packet i on its own: packet i advances exactly as swrt_ode23 advances an
 * ensemble holding packet i alone (its own error norm, initial step, rejections and dense output), so a packet's result
 * does not depend on the other packets, their number or the sharding.  tspan as in swrt_ode23 (a decreasing tspan
 * integrates backward in time).  Y as in swrt_ode23 (ntspan x 4 x n, may be NULL; the rows after a stopped packet's
 * t_end are NaN).
 * pstat (may be NULL): n x 3 int32, column-major = accepted steps, rejected steps, status (0 reached tfinal, 1 step size
 * fell below 16*eps(t)); t_end (may be NULL): tfinal, or the t at which the packet stopped (it keeps its last accepted
 * state).  stats[0..4] = accepted steps, rejected steps and RHS evaluations summed over packets, packets that stopped,
 * host waits.  A stopped packet is not an error: SWRT_OK is returned.                                               */
int swrt_ode23_packets(swrt_handle* h, const double* tspan, int ntspan, double tmax, double rtol, double atol, double* Y,
                       int32_t* pstat, double* t_end, int64_t stats[5]);
/* for i = 1:n, [~, Y] = ode23(odefun_i, tspan(:, i), y_i); end -- swrt_ode23_packets with a tspan of its own for every
 * packet: staggered observation or release times, and forward and backward packets in one call.  tspan is n x ntspan,
 * column-major: entry j of packet i is tspan[j*n + i] (ntspan >= 2, shared).  Packet i advances exactly as swrt_ode23
 * advances a handle holding packet i alone with the tspan of its row: its own direction (+1 when its last entry is >= its
 * first, else -1), initial step, MaxStep, stop and dense rows.  A row whose entries are all equal takes one step of size 0
 * and keeps its state.  tmax is shared (alpha = t/tmax for every packet).  Y (ntspan x 4 x n, may be NULL) row j of
 * packet i is the state at tspan[j*n + i]; Y, pstat, t_end and stats[0..4] as in swrt_ode23_packets.  SWRT_ERR_ARG, with
 * the packets untouched, when an entry is not finite or steps against its own row's direction (the message names the
 * packet and the entry; equal neighbours are allowed).  With events: swrt_ode23_packets_tspans_events.               */
int swrt_ode23_packets_tspans(swrt_handle* h, const double* tspan /* n x ntspan, column-major */, int ntspan,
                              double tmax, double rtol, double atol, double* Y, int32_t* pstat, double* t_end,
                              int64_t stats[5]);

/* [t, Y, te, ye, ie] = ode23(odefun_i, tspan, y_i, odeset('Events', ...)) for every packet i on its own: event j is a level
 * crossing of g_j(x, y, k, l), a function of the packet state alone.  omega is swrt_hist_omega's intrinsic frequency
 * sqrt(f^2 + gH (k^2 + l^2)) (analysis/load_data.m:33); every operation is rounded on its own.                       */
#define SWRT_EVENT_X      0   /* g = x - level (unwrapped) */
#define SWRT_EVENT_Y      1   /* g = y - level             */
#define SWRT_EVENT_K      2   /* g = k - level             */
#define SWRT_EVENT_L      3   /* g = l - level             */
#define SWRT_EVENT_KMAG   4   /* g = sqrt(k^2 + l^2) - level */
#define SWRT_EVENT_OMEGA  5   /* g = omega - level         */
#define SWRT_MAX_EVENTS   8
typedef struct swrt_event {
    int32_t kind;        /* SWRT_EVENT_* */
    int32_t direction;   /* 0 any crossing, +1 rising only (g: < 0 to >= 0), -1 falling only (g: > 0 to <= 0) */
    int32_t terminal;    /* 1: the packet stops at the event */
    int32_t reserved;    /* 0 */
    double level;        /* finite */
} swrt_event;
/* The solve of swrt_ode23_packets; tspan must be strictly increasing.  After every accepted step from t to tnew, event j
 * fires when g_j at the previous accepted state (y0 at the start) is non-zero, neither value is NaN, the sign changes and
 * the direction allows it; a zero at the left end is never an event (none at t0).  It is located on the step's ntrp23
 * cubic by Illinois regula falsi (DESIGN.md section 11): te is the first point found with g_j = 0 or of the post-crossing
 * sign, ye the cubic there.  Events never change a step decision.
 * Records per packet, in ascending (te, ie) order over the solve: te[r*n+i], ye[(r*4+c)*n+i] (c = x, y, k, l) and ie[r*n+i]
 * (1-based event index) for r < ev_cap, NaN / 0 when unused; ne[i] counts every event found (> ev_cap: records were
 * dropped).  Any of te, ye, ie, ne may be NULL.  A terminal event stops its packet at the earliest terminal te* of the
 * step: records after te* are not kept, the packet's state becomes that record's ye, t_end = te*, status = 2, and the
 * dense rows after te* stay NaN.  Y, pstat (status 2 = terminal event), t_end and stats[0..4] as in
 * swrt_ode23_packets; stats[5] = events found, stats[6] = packets stopped by a terminal event.
 * SWRT_ERR_ARG: nev outside 1..SWRT_MAX_EVENTS, ev_cap < 0, an unknown kind, a direction outside {-1, 0, 1}, a terminal
 * flag outside {0, 1}, reserved != 0, a non-finite level, a tspan not strictly increasing.  Backward solves and a
 * tspan per packet with events: swrt_ode23_packets_tspans_events.                                                  */
int swrt_ode23_packets_events(swrt_handle* h, const double* tspan, int ntspan, double tmax, double rtol, double atol,
                              const swrt_event* ev, int nev, int ev_cap, double* Y, int32_t* pstat, double* t_end,
                              double* te, double* ye, int32_t* ie, int32_t* ne, int64_t stats[7]);
/* for i = 1:n, [t, Y, te, ye, ie] = ode23(odefun_i, tspan(:, i), y_i, odeset('Events', ...)); end -- the events of
 * swrt_ode23_packets_events on the solve of swrt_ode23_packets_tspans: a tspan row per packet (n x ntspan, column-major,
 * entry j of packet i at tspan[j*n + i]), each in its own direction tdir (+1 when its last entry is >= its first, else
 * -1), so back-traced, staggered and mixed-direction packets find their events in one call.  tmax, Y, pstat and t_end
 * as in swrt_ode23_packets_tspans; ev, ev_cap, te, ye, ie, ne, status 2 and stats[0..6] as in
 * swrt_ode23_packets_events.  Everything follows the packet's direction of integration:
 * - detection is unchanged: rising (g: < 0 to >= 0) is rising along the integration, i.e. as t decreases backward;
 * - te is located on [t, tnew] in integration order by the same Illinois regula falsi, mirrored for tdir = -1 (t -> -t
 *   gives te bit for bit up to sign);
 * - records are kept in order of encounter: ascending tdir*te, then ie;
 * - a terminal event stops its packet at the first terminal te* in integration order: records and dense rows beyond te*
 *   (tdir*(t - te*) > 0) are not kept / stay NaN.
 * A row of equal entries takes one step of size 0: it finds no event and keeps its state.  Apart from a terminal stop a
 * packet's solve is bit for bit that of swrt_ode23_packets_tspans.  SWRT_ERR_ARG, with the packets untouched: a row
 * entry not finite or stepping against its own row's direction, and every event fault swrt_ode23_packets_events
 * refuses.                                                                                                         */
int swrt_ode23_packets_tspans_events(swrt_handle* h, const double* tspan /* n x ntspan, column-major */, int ntspan,
                                     double tmax, double rtol, double atol, const swrt_event* ev, int nev, int ev_cap,
                                     double* Y, int32_t* pstat, double* t_end, double* te, double* ye, int32_t* ie,
                                     int32_t* ne, int64_t stats[7]);

/* ---- diagnostics -------------------------------------------------------------------------- */
/* histcounts(omega, edges) (analysis/load_data.m:39-47): counts[nedges-1], bin i = [e_i,e_i+1),
 * last bin closed; accumulate != 0 adds to counts instead of overwriting.                      */
int swrt_hist_omega(swrt_handle* h, int kind, double alpha, const double* edges, int nedges,
                    uint64_t* counts, int accumulate);
/* the same, but the counts stay on the device (u64[nedges-1], owned by the handle, valid until the
 * next histogram call) so that a multi-GPU host can all-reduce them in place (NCCL) without a
 * round trip through host memory; the handle's stream is synchronised on return              */
int swrt_hist_omega_dev(swrt_handle* h, int kind, double alpha, const double* edges, int nedges,
                        uint64_t** counts_dev);
/* pipelined form for multi-GPU diagnostics: _launch queues the histogram kernel behind the work already on the
 * handle's stream and returns at once; _wait blocks until THAT kernel has finished (not later work), after which
 * counts_dev may be snapshotted and all-reduced while the next interval's packet kernel runs                  */
int swrt_hist_omega_launch(swrt_handle* h, int kind, double alpha, const double* edges, int nedges,
                           uint64_t** counts_dev);
int swrt_hist_omega_wait(swrt_handle* h);
/* theoretical omega pdf of ideal_omega_distribution.m:3-11: omega_abs = omega0 + U(x_i).kvec_j over npts
 * points (the caller's grid XX(:),YY(:)) x nangles wavevectors (kvx,kvy = k_0*[cos(t) sin(t)]), counted
 * into histcounts-style bins; counts[nedges-1].                                                   */
int swrt_ideal_omega_hist(swrt_handle* h, double alpha, int64_t npts, const double* x, const double* y,
                          const double* kvx, const double* kvy, int nangles, double omega0,
                          const double* edges, int nedges, uint64_t* counts);
/* out[0]=sum omega, out[1]=sum Omega (omega+U.k), out[2]=max omega, out[3]=min omega,
 * out[4]=number of non-finite packets, out[5]=sum a, out[6]=n, out[7]=sum omega*a              */
int swrt_diag(swrt_handle* h, double alpha, double out[8]);
/* per-packet intrinsic and absolute frequency (symplectic_full_fourier.m:41,54-56)             */
int swrt_omega(swrt_handle* h, double alpha, double* omega, double* Omega_abs);
/* per-packet quantities for swrt_packet_quantity / swrt_hist2; every operation rounded on its own */
#define SWRT_Q_XMOD       0  /* x periodic in [0, L): r = x - L*floor(x/L); r < 0 -> r + L; then r >= L -> 0 */
#define SWRT_Q_YMOD       1  /* the same for y */
#define SWRT_Q_K          2
#define SWRT_Q_L          3
#define SWRT_Q_KMAG       4  /* sqrt(k*k + l*l), SWRT_EVENT_KMAG's expression */
#define SWRT_Q_THETA      5  /* atan2(l, k) in [-pi, pi] (CUDA atan2) */
#define SWRT_Q_OMEGA      6  /* omega_kernel's omega, bit-identical to swrt_omega */
#define SWRT_Q_OMEGA_ABS  7  /* Omega = omega + U.k at alpha, bit-identical to swrt_omega's Omega_abs; needs a flow */
/* out[n]: quantity q of every packet (alpha is used by the two frequencies only).  A multi-device handle fills each
 * shard's rows.  SWRT_ERR_ARG: an unknown q or a null out; SWRT_ERR_STATE: OMEGA_ABS without flow slot 0, or a
 * two-frame alpha without slot 1.                                                                                  */
int swrt_packet_quantity(swrt_handle* h, int q, double alpha, double* out /* n */);
/* N = histcounts2(Qx, Qy, xedges, yedges) of the packets' quantities qx, qy, each value exactly what
 * swrt_packet_quantity returns: counts (nxe-1) x (nye-1) column-major, counts[i + j*(nxe-1)] = N(i,j); bin
 * [e_i, e_i+1) on each axis, last bin closed; NaN or out of range in either coordinate is not counted; accumulate
 * != 0 adds to counts.  alpha is used by SWRT_Q_OMEGA / SWRT_Q_OMEGA_ABS only.  A multi-device handle SUM-all-reduces
 * the u64 counts of its shards (bit-exact under any sharding).  SWRT_ERR_ARG, with the handle usable: an unknown
 * quantity, nxe or nye outside 2..4096, edges not finite or decreasing, a null pointer; SWRT_ERR_STATE as in
 * swrt_packet_quantity.                                                                                            */
int swrt_hist2(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye,
               double alpha, uint64_t* counts, int accumulate);
/* per-packet weights for swrt_weight_scale / swrt_hist2_sums; a is the packets' wave action (1 when swrt_set_packets was
 * given a NULL a), every product rounded on its own                                                               */
#define SWRT_W_ACTION     0  /* a */
#define SWRT_W_ENERGY     1  /* omega*a, omega bit-identical to swrt_omega's (needs no flow) */
#define SWRT_W_PSEUDO_K   2  /* k*a */
#define SWRT_W_PSEUDO_L   3  /* l*a */
#define SWRT_MAX_WEIGHTS  4
/* scale_exp[v] = E, the least integer with |w| < 2^E for every finite weight w[v] of the ensemble (0 when all are zero
 * or non-finite); a multi-device handle MAX-all-reduces it over its devices.  alpha is the flow time of omega.
 * SWRT_ERR_ARG: nw outside 1..SWRT_MAX_WEIGHTS, an unknown kind, a null pointer.                                    */
int swrt_weight_scale(swrt_handle* h, const int32_t* w, int nw, double alpha, int32_t* scale_exp /* nw */);
/* Per-bin sums of nw weight kinds w[0..nw) over swrt_hist2's bins, as fixed-point integers that every sharding and
 * packet order sums to the same bits.  Each weight becomes q = rint(w * 2^(95-E)) (|q| <= 2^95, E = scale_exp[v], or
 * swrt_weight_scale's when scale_exp is NULL); its three 32-bit digits (signed like w) are added to int64 counters.
 * The sum is Sum(q) * 2^(E-95) rounded once to the nearest double (swrt_fixed_sums_to_double): exactly rounded when
 * all weights are within 2^42 of the largest (|w| >= 2^(E-43): q is w scaled, no rounding), else fixed-point to
 * 2^(E-95), each smaller weight off by at most 2^(E-96).
 * Binning, refusals and the bin rule are swrt_hist2's.  sums[(v*(nye-1) + j)*(nxe-1) + i] (may be NULL);
 * counts (may be NULL) = swrt_hist2's; acc (may be NULL) = acc[4*b + c], b the sums index: c = 0, 1, 2 the digit
 * counters of 2^0, 2^32, 2^64 and c = 3 the weights that were non-finite or >= 2^E in magnitude (such a bin's sum is
 * NaN).  A multi-device handle MAX-all-reduces the exponents and SUM-all-reduces acc and counts.  SWRT_ERR_ARG, with the
 * handle usable: swrt_hist2's refusals, nw outside 1..SWRT_MAX_WEIGHTS, an unknown kind, a scale_exp outside
 * -1073..1024, more than 2^31 - 1 packets (the counters' bound); SWRT_ERR_STATE as in swrt_packet_quantity.          */
int swrt_hist2_sums(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye,
                    double alpha, const int32_t* w, int nw, const int32_t* scale_exp, double* sums, uint64_t* counts,
                    int64_t* acc);
/* sums[v*nbins + b] = (acc[4*(v*nbins + b)] + acc[..+1]*2^32 + acc[..+2]*2^64) * 2^(scale_exp[v] - 95), rounded once to
 * the nearest double (ties to even; overflow to +-inf, subnormal results rounded at 2^-1074); NaN where acc[..+3] != 0.
 * Host only, needs no device: the final step of swrt_hist2_sums, and of a caller who all-reduces acc itself.         */
int swrt_fixed_sums_to_double(const int64_t* acc, int64_t nbins, int nw, const int32_t* scale_exp, double* sums);

/* ---- spectral <-> grid kit on the device (setup, not hot path) ----------------------------- */
/* fk = g2k(fg) (g2k.m:5-9) and fg = k2g(fk) (k2g.m:5-6, fulspec.m:10-19), column-major.         */
int swrt_g2k(int device, const double* fg, int nx, double* fk_re, double* fk_im);
int swrt_k2g(int device, const double* fk_re, const double* fk_im, int nx, double* fg);

/* ---- on-device one-layer QG frame producer (setup for time-evolving runs; not the hot path) --
 * qgsw_raytrace.m:111-137 (AB3 loop), :222-230 (filter), :216-220 (forcing), :270-286 (update()).
 * swrt_set_flow_from_qg fills a flow slot with psi = -q/(K_d2+K2) (grid_U.m:2) without leaving
 * the device.                                                                                   */
typedef struct swrt_qg swrt_qg;
int swrt_qg_create(int device, int nx, double L, double K_d2, double beta, double r_drag,
                   double force_strength, double f, double Cg, double dt,
                   const double* qk_re, const double* qk_im, swrt_qg** out);
int swrt_qg_step(swrt_qg* q, int nsteps);
int swrt_qg_get(swrt_qg* q, double* qk_re, double* qk_im);
int swrt_qg_get_grid(swrt_qg* q, double* qgrid);   /* q = k2g(qk), nx x nx column-major (the pv frame of :165-170) */
int swrt_qg_destroy(swrt_qg* q);
int swrt_set_flow_from_qg(swrt_handle* h, int slot, swrt_qg* q, double u_mean);

/* ---- on-device TWO-layer QG frame producer (qg2layersw_raytrace.m:120-181, update() :309-323) ------------
 * q1,q2: layer PV spectra (g2k layout).  The inversion matrix B (:137-143), the linear operator factor_L
 * (:146-150: shear advection + hyperdiffusion nu*K^(2 alpha) + drag r + beta) and expm(factor_L*dt) live on
 * the device; the CFL logic that picks dt (:156-165) is host control flow built on swrt_qg2_max_speed.     */
typedef struct swrt_qg2 swrt_qg2;
int swrt_qg2_create(int device, int nx, double L, double K_d2, double beta, double shear_strength, double r, double nu,
                    double alpha, const double* q1_re, const double* q1_im, const double* q2_re, const double* q2_im,
                    swrt_qg2** out);
int swrt_qg2_max_speed(swrt_qg2* q, double* U0);   /* sqrt(max(u.^2+v.^2)) of grid_U over both layers (:155-157) */
int swrt_qg2_step(swrt_qg2* q, double dt);         /* one AB1/AB2/AB3 + integrating-factor step (:166-181)       */
int swrt_qg2_get(swrt_qg2* q, int layer, double* qk_re, double* qk_im);
int swrt_qg2_destroy(swrt_qg2* q);
/* flow slot <- grid_U(qk(:,:,1), ..., shear_strength): top layer, one-layer inversion, mean shear (:187-188)  */
int swrt_set_flow_from_qg2(swrt_handle* h, int slot, swrt_qg2* q);

/* ---- instrumentation ---------------------------------------------------------------------- */
/* number of kernel launches issued by this handle since creation / since the last reset        */
int64_t swrt_launch_count(swrt_handle* h, int reset);
/* milliseconds spent in the dominant kernel of the most recent swrt_step / swrt_eval call,
 * measured with CUDA events on the handle's stream; nlaunch receives how many packet-stepping
 * runs it made: one per dense-kernel launch, one per anchored leapfrog run (whose drift, sort,
 * K1 and K2 launches of every sub-step are all inside the timed bracket and in swrt_launch_count) */
double  swrt_last_kernel_ms(swrt_handle* h, int* nlaunch);
/* executed real fp64 flops (spectral) or gathered bytes (Lagrange) per packet per evaluation   */
double  swrt_work_per_eval(const swrt_handle* h, int nplanes);
int     swrt_synchronize(swrt_handle* h);
/* run on a caller-owned CUDA stream (a cudaStream_t passed as void*; NULL = the handle's own) so
 * that the caller's events (e.g. torch.cuda.Event on torch's current stream) bracket the work   */
int     swrt_set_stream(swrt_handle* h, void* cuda_stream);
/* device-side stopwatch on the handle's stream: start records an event, stop records another,
 * waits for it and returns the elapsed milliseconds (<0 on error)                               */
int     swrt_timer_start(swrt_handle* h);
double  swrt_timer_stop(swrt_handle* h);
/* tuning knobs: 1 or 2 m-tiles per warp in the spectral kernel (0 = automatic); flags bits 3-4 = where the dense
 * kernel keeps the x twiddles of a step (0 automatic, 1 rotate in registers, 2 global / L2 table, 3 shared-memory
 * table with shrunk chunks else global); flags bit 0 = do
 * not use the psi-hat moment contraction (always contract the six planes); flags bit 1 (LAGRANGE6) =
 * blend two flow frames on the grid before the gather (half the gathers) instead of interpolating both
 * frames and blending the results as interpolate_U.m:19-23 does (the default, bit-faithful); flags
 * bit 2 (SPECTRAL, NUFFT) = run step_packet / step_packet_xka as separate evaluation + stage launches (the
 * composed route: 4-5 evaluation kernels + 5 point-wise kernels per step, state and planes through
 * HBM) instead of the fused kernel (one launch per run of steps, packet in registers)            */
int     swrt_set_tuning(swrt_handle* h, int mtiles, int flags);
/* planes the spectral kernel contracts for a six-plane evaluation: 3 when every flow slot was
 * given as psi-hat (moments N0,N1,N2; 6 nx^2 flops), else 6 (12 nx^2 flops); 0 in LAGRANGE6    */
int     swrt_contracted_planes(const swrt_handle* h);
/* diagnostic, host-only (no device needed): the launch geometry the dense kernel would use for an
 * nx^2 grid contracting `nplanes` planes with `mtiles` m-tiles per warp.  out[0..9] = n-tiles per
 * pass, ky passes, k-steps per pass (padded), k-steps per chunk, ring stages, chunk bytes, x twiddles
 * (0 = rotated in registers, 1 = per-step table in shared memory, 2 = per-step table in a per-CTA
 * global / L2 scratch), shared-memory twiddle-table bytes, dynamic shared memory bytes per CTA,
 * packed-stack bytes per flow slot.  Returns SWRT_OK or SWRT_ERR_ARG.                             */
int     swrt_spectral_geometry(int nx, int nplanes, int mtiles, int64_t out[10]);
/* roofline probe for the gather-bound modes (LAGRANGE6, NUFFT): the rate (GB/s of useful bytes) at which the device serves
 * scattered 64-byte segments of an L2-resident table of `table_bytes` (power of two, e.g. 16 MiB = the 512^2 NUFFT fine
 * grid) to quads of lanes, eight loads in flight per lane; best of `reps`.  Returns SWRT_OK or an error code.      */
int     swrt_gather_probe(int device, int64_t table_bytes, int reps, double* gbytes_per_s);

#ifdef __cplusplus
}
#endif
#endif /* SWRT_H */
