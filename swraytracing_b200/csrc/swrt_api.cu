// swrt_api.cu -- the C ABI of libswrt.so (include/swrt.h): handle, flow upload, packet state,
// evaluation, fused stepping, diagnostics.  Host logic only; all arithmetic is in the kernels.
#include "../../include/swrt.h"
#include "swrt_internal.h"

#include <cufft.h>
#include <nccl.h>          // types only: the library itself is dlopen()ed when a multi-device handle is created
#include <dlfcn.h>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace swrt;

namespace {

std::string g_create_error;

// plane subsets that get their own packed stack; SUB_PSI3 = the psi-hat moment planes (ids 7,8,9)
enum Subset { SUB_SIX = 0, SUB_SEVEN = 1, SUB_UV = 2, SUB_UVH = 3, SUB_PSI3 = 4, SUB_COUNT = 5 };
const int kSubsetN[SUB_COUNT] = {6, 7, 2, 3, 3};
const int kSubsetIds[SUB_COUNT][kMaxPlanes] = {
    {0, 1, 2, 3, 4, 5, 0}, {0, 1, 2, 3, 4, 5, 6}, {0, 1, 0, 0, 0, 0, 0}, {0, 1, 6, 0, 0, 0, 0}, {7, 8, 9, 0, 0, 0, 0}};

struct Stack {
    bool geom_ready = false;
    PackGeom g{};
    double* slot[2] = {nullptr, nullptr};
    bool slot_valid[2] = {false, false};
    double* blend = nullptr;
};

}  // namespace

struct swrt_handle {
    swrt_params p{};
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaEvent_t tm0 = nullptr, tm1 = nullptr;
    std::string err;
    // packets
    int64_t n = 0, cap = 0;
    double *x = nullptr, *y = nullptr, *k = nullptr, *l = nullptr, *a = nullptr;
    // spectral source planes per slot
    bool slot_set[2] = {false, false};
    int slot_npl[2] = {0, 0};
    double2* planes[2][kNumSrcPlanes] = {};
    bool psi_ok[2] = {false, false};      // slot was given as psi-hat: moment planes 7..9 are valid
    double u_mean[2] = {0.0, 0.0};
    bool disable_psi = false;
    bool preblend_grid = false;       // LAGRANGE6: blend the two grids before the gather (fast) instead of after (exact)
    bool unfused_rk4 = false;         // NUFFT: compose step_packet* from evaluation + glue launches (the dense mode's route)
    Stack stacks[SUB_COUNT];
    // lagrange grids per slot (node-interleaved, always 7 planes wide when H given else 6)
    double* grid[2] = {nullptr, nullptr};
    double* grid_blend = nullptr;
    int grid_npl = 0;
    // NUFFT mode: (u,v) fine grids per slot + blend, deconvolution factors, nf-point FFT work
    double* nufft_grid[2] = {nullptr, nullptr};
    double* nufft_blend = nullptr;
    double* nufft_h[2] = {nullptr, nullptr};   // optional H fine grid per slot (step_packet_xka)
    double* nufft_hblend = nullptr;
    double* nufft_invphi = nullptr;
    void* nufft_fft = nullptr;            // FftWork* for the nf-point transforms
    void* grid_fft = nullptr;             // FftWork* for the nx-point g2k / k2g of flow uploads (plan kept across calls)
    double* grid_tmp = nullptr;           // kMaxPlanes x nx^2 gridded planes before interleaving (kept across calls)
    // scratch
    int64_t scratch_cap = 0;
    double* e[kMaxPlanes] = {};
    double *xs = nullptr, *ys = nullptr, *ax = nullptr, *ay = nullptr, *om = nullptr, *Om = nullptr;
    double* diag_dev = nullptr;
    // ode23 (Bogacki-Shampine) work arrays: yt[4], f[4][4]
    int64_t bs_cap = 0;
    double* bs_yt[4] = {};
    double* bs_f[4][4] = {};
    unsigned long long* bs_norm_dev = nullptr;
    bool bs_ready = false;
    Ode23Ctl* ode_ctl = nullptr;          // swrt_ode23: the controller state on the device ...
    Ode23Ctl* ode_host = nullptr;         // ... and its pinned host image (set-up and read-back)
    cudaEvent_t ode_ev = nullptr;
    // swrt_ode23_packets: the per-packet controller state (Ode23Pkt: 10 double and 5 int arrays of pkt_cap entries, then the
    // report words), its pinned report image, and the alpha-1 planes of a two-frame SPECTRAL solve
    double* pkt_d = nullptr; int* pkt_i = nullptr; int64_t pkt_cap = 0;
    int* pkt_rep_host = nullptr;
    double* pkt_e1 = nullptr;
    // swrt_ode23_packets_events: the event values and records of the packets (Ode23Ev's arrays)
    double* ev_d = nullptr; size_t ev_dcap = 0;
    int* ev_i = nullptr; size_t ev_icap = 0;
    double* edges_dev = nullptr; int edges_cap = 0;
    std::vector<double> edges_host;       // what edges_dev currently holds
    unsigned long long* counts_dev = nullptr; int counts_cap = 0;
    // swrt_hist2: xedges then yedges on the device (h2_edges_host and h2_nxe: what they hold) and the u64 counts
    double* h2_edges_dev = nullptr; int h2_edges_cap = 0;
    std::vector<double> h2_edges_host; int h2_nxe = 0;
    unsigned long long* h2_counts_dev = nullptr; int64_t h2_counts_cap = 0;
    // swrt_weight_scale / swrt_hist2_sums: the biased scale exponents (kScaleBias) and their host image, the digit counters
    int* ws_exp_dev = nullptr; int ws_exp_host[SWRT_MAX_WEIGHTS] = {};
    long long* h2s_acc_dev = nullptr; int64_t h2s_acc_cap = 0;
    // instrumentation
    int64_t launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, hist_ev = nullptr;
    bool timing_valid = false;
    int last_nlaunch = 0;
    int mtiles = 0;
    // fused runs on a time-dependent flow: the operands (packed stacks / fine grids / Lagrange grids) of up to
    // kMaxFusedBlend steps, pre-blended at alpha_j and stored back to back
    double* arena = nullptr; size_t arena_cap = 0;
    double* twid = nullptr; size_t twid_cap = 0;          // global twiddle-table scratch of the dense kernel (atab == 2)
    int twiddle_pref = 0;                                 // swrt_set_tuning bits 3-4
    double* arena_h = nullptr; size_t arena_h_cap = 0;      // NUFFT (u,v,H,0) grids
    // anchored leapfrog (DESIGN.md section 3e): per-packet sort keys, per-anchor counts / offsets and the H' blocks of
    // every anchor
    int64_t anc_cap = 0;
    int* anc_key = nullptr; unsigned long long* anc_rank = nullptr; long long* anc_perm = nullptr;
    int anc_n = 0;
    unsigned long long *anc_cnt = nullptr, *anc_off = nullptr;
    double* anc_hexp = nullptr; size_t anc_hexp_cap = 0;
    // host staging of swrt_step_host / swrt_set_packets / swrt_get_packets (pinned ring + copy streams)
    struct Stager* stager = nullptr;
    // multi-device handle (swrt_params.ngpu > 1): one single-device child per GPU, contiguous packet shards
    int ngpu = 1;
    std::vector<swrt_handle*> shard;
    std::vector<int64_t> off;             // shard i holds packets [off[i], off[i+1])
    std::vector<ncclComm_t> comms;
    double* red_dev = nullptr;            // child: 3 x 8 doubles for the diagnostic all-reduces
};

namespace {

int fail(swrt_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

// multi-device handles (ngpu > 1) are served by the grp_* layer at the end of this file
#define GROUP(h, call) do { if ((h)->ngpu > 1) return call; } while (0)
int grp_create(const swrt_params* p, swrt_handle** out);
int grp_destroy(swrt_handle* g);
int grp_sync(swrt_handle* g);
int grp_set_packets(swrt_handle* g, int64_t n, const double* x, const double* y, const double* k, const double* l, const double* a);
int grp_get_packets(swrt_handle* g, double* x, double* y, double* k, double* l, double* a);
int grp_step_host(swrt_handle* g, int scheme, double dt, int nsteps, double alpha0, double dalpha, int64_t n,
                  const double* const in[5], double* const out[5]);
int grp_step(swrt_handle* g, int scheme, double dt, int nsteps, double alpha0, double dalpha, bool sync);
int grp_hist_omega(swrt_handle* g, int kind, double alpha, const double* edges, int nedges, uint64_t* counts, int accumulate);
int grp_hist_omega_dev(swrt_handle* g, int kind, double alpha, const double* edges, int nedges, uint64_t** counts_dev, bool wait);
int grp_diag(swrt_handle* g, double alpha, double out[8]);
int grp_bs23_begin(swrt_handle* g, double alpha, double threshold, double* rh_norm);
int grp_bs23_attempt(swrt_handle* g, double hstep, const double alpha[3], double threshold, double* err_norm);
int grp_ideal_omega_hist(swrt_handle* g, double alpha, int64_t npts, const double* x, const double* y, const double* kvx,
                         const double* kvy, int nangles, double omega0, const double* edges, int nedges, uint64_t* counts);
int grp_hist2(swrt_handle* g, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye, double alpha,
              uint64_t* counts, int accumulate);
int grp_weight_scale(swrt_handle* g, const WeightKinds& wk, double alpha, int32_t* scale_exp);
int grp_hist2_sums(swrt_handle* g, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye, double alpha,
                   const WeightKinds& wk, const int32_t* scale_exp, double* sums, uint64_t* counts, int64_t* acc);
int up(swrt_handle* g, swrt_handle* c, int rc);
inline double* at(double* p, int64_t lo) { return p ? p + lo : nullptr; }
void stager_free(swrt_handle* h);
// calls whose per-packet outputs are host arrays: each shard writes its slice (devices one after another; these are the
// inspection entry points, not the stepping path)
template <typename F>
int grp_each_slice(swrt_handle* g, F f) {
    for (size_t i = 0; i < g->shard.size(); i++) {
        swrt_handle* c = g->shard[i];
        if (g->off[i + 1] == g->off[i]) continue;
        int rc = f(c, g->off[i]);
        if (rc != SWRT_OK) return up(g, c, rc);
    }
    return SWRT_OK;
}

#define CU(h, expr)                                                                                   \
    do {                                                                                              \
        cudaError_t e__ = (expr);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return fail(h, e__ == cudaErrorMemoryAllocation ? SWRT_ERR_ALLOC : SWRT_ERR_CUDA,         \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

#define REQUIRE(h, cond, code, ...) \
    do { if (!(cond)) return fail(h, code, __VA_ARGS__); } while (0)

template <typename T> void dfree(T*& p) { if (p) { cudaFree(p); p = nullptr; } }

// scoped device temporary: freed on every exit path (the CU()/REQUIRE() macros return early)
template <typename T>
struct DevTmp {
    T* p = nullptr;
    DevTmp() = default;
    DevTmp(const DevTmp&) = delete;
    DevTmp& operator=(const DevTmp&) = delete;
    ~DevTmp() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t count) { return cudaMalloc(&p, count * sizeof(T)); }
};

// per-CTA global scratch of the dense kernel's twiddle table (PackGeom.atab == 2): one double per lane per k-step per warp
int ensure_twid(swrt_handle* h, const PackGeom& g, double** out) {
    *out = nullptr;
    if (g.atab != 2) return SWRT_OK;
    const size_t need = (size_t)h->num_sms * kCtasPerSm * kConsumerWarps * g.ksteps * 32;
    if (need > h->twid_cap) {
        dfree(h->twid); h->twid_cap = 0;
        CU(h, cudaMalloc(&h->twid, need * sizeof(double)));
        h->twid_cap = need;
    }
    *out = h->twid;
    return SWRT_OK;
}

int pick_mtiles(const swrt_handle* h, int64_t n) {
    if (h->mtiles == 1 || h->mtiles == 2) return h->mtiles;
    (void)n;
    return 1;
}

int ensure_scratch(swrt_handle* h, int64_t n) {
    if (n <= h->scratch_cap) return SWRT_OK;
    for (auto& p : h->e) dfree(p);
    dfree(h->xs); dfree(h->ys); dfree(h->ax); dfree(h->ay); dfree(h->om); dfree(h->Om);
    h->scratch_cap = 0;                       // a failed allocation below must not leave a stale capacity behind
    size_t b = (size_t)n * sizeof(double);
    for (auto& p : h->e) CU(h, cudaMalloc(&p, b));
    CU(h, cudaMalloc(&h->xs, b)); CU(h, cudaMalloc(&h->ys, b)); CU(h, cudaMalloc(&h->ax, b));
    CU(h, cudaMalloc(&h->ay, b)); CU(h, cudaMalloc(&h->om, b)); CU(h, cudaMalloc(&h->Om, b));
    h->scratch_cap = n;
    return SWRT_OK;
}

int ensure_packets(swrt_handle* h, int64_t n) {
    if (n > h->cap) {
        dfree(h->x); dfree(h->y); dfree(h->k); dfree(h->l); dfree(h->a);
        h->cap = 0; h->n = 0;
        size_t b = (size_t)n * sizeof(double);
        CU(h, cudaMalloc(&h->x, b)); CU(h, cudaMalloc(&h->y, b)); CU(h, cudaMalloc(&h->k, b));
        CU(h, cudaMalloc(&h->l, b)); CU(h, cudaMalloc(&h->a, b));
        h->cap = n;
    }
    h->n = n;
    return SWRT_OK;
}

// ---- spectral stacks ---------------------------------------------------------------------------
int ensure_stack(swrt_handle* h, int sub, int slot, int mtiles) {
    Stack& s = h->stacks[sub];
    const PackGeom want = make_geom(h->p.nx, kSubsetN[sub], kSubsetIds[sub], mtiles, h->twiddle_pref);
    // a packed stack is only valid for the exact geometry it was packed with (tile grouping, chunking, padding)
    if (!s.geom_ready || s.g.G != want.G || s.g.kc != want.kc || s.g.ksteps != want.ksteps || s.g.npass != want.npass ||
        s.g.total_doubles != want.total_doubles || s.g.atab != want.atab) {
        s.g = want;
        s.geom_ready = true;
        for (int i = 0; i < 2; i++) { dfree(s.slot[i]); s.slot_valid[i] = false; }
        dfree(s.blend);
    }
    s.g = want;
    if (s.slot_valid[slot]) return SWRT_OK;
    REQUIRE(h, h->slot_set[slot], SWRT_ERR_STATE, "flow slot %d has not been set", slot);
    REQUIRE(h, h->slot_npl[slot] >= (sub == SUB_SEVEN || sub == SUB_UVH ? 7 : 6), SWRT_ERR_STATE,
            "flow slot %d has no H plane (needed by this scheme)", slot);
    REQUIRE(h, sub != SUB_PSI3 || h->psi_ok[slot], SWRT_ERR_STATE, "flow slot %d was not given as psi-hat", slot);
    if (!s.slot[slot]) CU(h, cudaMalloc(&s.slot[slot], s.g.total_doubles * sizeof(double)));
    const double2* src[kNumSrcPlanes];
    for (int i = 0; i < kNumSrcPlanes; i++) src[i] = h->planes[slot][i] ? h->planes[slot][i] : h->planes[slot][0];
    launch_pack(s.g, src, s.slot[slot], h->stream);
    h->launches++;
    CU(h, cudaGetLastError());
    s.slot_valid[slot] = true;
    return SWRT_OK;
}

// returns the device stack holding (1-alpha)*slot0 + alpha*slot1 for this subset
int active_stack(swrt_handle* h, int sub, double alpha, int mtiles, const double** out, PackGeom* g) {
    int rc = ensure_stack(h, sub, 0, mtiles);
    if (rc) return rc;
    Stack& s = h->stacks[sub];
    *g = s.g;
    if (alpha == 0.0) { *out = s.slot[0]; return SWRT_OK; }
    REQUIRE(h, h->slot_set[1], SWRT_ERR_STATE, "alpha = %g but flow slot 1 has not been set", alpha);
    rc = ensure_stack(h, sub, 1, mtiles);
    if (rc) return rc;
    if (alpha == 1.0) { *out = s.slot[1]; return SWRT_OK; }
    if (!s.blend) CU(h, cudaMalloc(&s.blend, s.g.total_doubles * sizeof(double)));
    launch_axpby(s.blend, s.slot[0], s.slot[1], 1.0 - alpha, alpha, s.g.total_doubles, h->stream);
    h->launches++;
    *out = s.blend;
    return SWRT_OK;
}

int active_grid(swrt_handle* h, double alpha, const double** out) {
    REQUIRE(h, h->grid[0], SWRT_ERR_STATE, "flow slot 0 has not been set");
    if (alpha == 0.0) { *out = h->grid[0]; return SWRT_OK; }
    REQUIRE(h, h->grid[1], SWRT_ERR_STATE, "alpha = %g but flow slot 1 has not been set", alpha);
    if (alpha == 1.0) { *out = h->grid[1]; return SWRT_OK; }
    size_t nd = (size_t)h->p.nx * h->p.nx * h->grid_npl;
    if (!h->grid_blend) CU(h, cudaMalloc(&h->grid_blend, nd * sizeof(double)));
    launch_axpby(h->grid_blend, h->grid[0], h->grid[1], 1.0 - alpha, alpha, nd, h->stream);
    h->launches++;
    *out = h->grid_blend;
    return SWRT_OK;
}

// LAGRANGE6 frames for an evaluation at alpha: by default BOTH grids go to the kernel, which interpolates each and blends
// the results exactly as interpolate_U.m:19-23 does; with the pre-blend tuning flag one blended grid (half the gathers,
// equal in exact arithmetic, 1-ulp-level different in floating point)
int lag_frames(swrt_handle* h, double alpha, bool allow_exact, LagArgs& a) {
    a.grid2 = nullptr; a.alpha = 0.0;
    if (alpha == 0.0 || alpha == 1.0 || h->preblend_grid || !allow_exact) return active_grid(h, alpha, &a.grid);
    REQUIRE(h, h->grid[0], SWRT_ERR_STATE, "flow slot 0 has not been set");
    REQUIRE(h, h->grid[1], SWRT_ERR_STATE, "alpha = %g but flow slot 1 has not been set", alpha);
    a.grid = h->grid[0]; a.grid2 = h->grid[1]; a.alpha = alpha;
    return SWRT_OK;
}

void invalidate_slot(swrt_handle* h, int slot) {
    for (auto& s : h->stacks) s.slot_valid[slot] = false;
}

// the six velocity/gradient planes can come from the three psi-hat moment planes when every slot
// involved was uploaded with swrt_set_flow_spectral (halves the contraction work)
bool use_psi(const swrt_handle* h, double alpha) {
    return !h->disable_psi && h->psi_ok[0] && (alpha == 0.0 || h->psi_ok[1]);
}
void fill_psi_args(const swrt_handle* h, double alpha, SpecArgs& a) {
    a.psi = true;
    a.kappa = 2.0 * M_PI / h->p.L;
    // the kernel forms (1-alpha)*u_mean0 + alpha*u_mean1 itself (pinned roundings; alpha = 0 gives u_mean0 exactly)
    a.u_mean0 = h->u_mean[0]; a.u_mean1 = h->slot_set[1] ? h->u_mean[1] : 0.0;
    a.alpha0 = alpha; a.dalpha = 0.0; a.j0 = 0;
}

int active_nufft_grid(swrt_handle* h, double alpha, const double** out, const double** hout);
void fill_nufft_args(const swrt_handle* h, const double* grid, NufftArgs& a);
// SpecArgs / SpecRk4Args: grid spacing, nx, and 1/nx when nx is a power of two (exact), else 0
template <class A> void fill_spec_geom(const swrt_handle* h, A& a) {
    a.dx = h->p.L / h->p.nx; a.nxd = (double)h->p.nx;
    a.inv_nx = (h->p.nx & (h->p.nx - 1)) == 0 ? 1.0 / h->p.nx : 0.0;
}
// LagArgs: the grid geometry (the grids themselves are the caller's)
void fill_lag_args(const swrt_handle* h, LagArgs& a) {
    a.nx = h->p.nx; a.npl = h->grid_npl; a.dx = h->p.L / h->p.nx; a.bump = h->p.bump;
}
// LagArgs / NufftArgs of an evaluation: n device positions (xd, yd); out[c] receives the c-th plane of subset `sub`
template <class A> void fill_eval_io(A& a, int sub, int64_t n, const double* xd, const double* yd, double* const* out) {
    a.n = n; a.xin = xd; a.yin = yd;
    for (int c = 0; c < kSubsetN[sub]; c++) a.out[kSubsetIds[sub][c]] = out[c];
}

// evaluate subset planes at device positions into device outputs out[c] (c indexes subset planes)
int eval_dev(swrt_handle* h, int sub, double alpha, int64_t n, const double* xd, const double* yd,
             double* const* out) {
    if (n == 0) return SWRT_OK;
    if (h->p.mode == SWRT_MODE_SPECTRAL) {
        int mt = pick_mtiles(h, n);
        SpecArgs a{};
        const bool psi = (sub == SUB_SIX) && use_psi(h, alpha);
        int rc = active_stack(h, psi ? (int)SUB_PSI3 : sub, alpha, mt, &a.stack, &a.g);
        if (rc) return rc;
        if (psi) fill_psi_args(h, alpha, a);
        a.n = n; a.xin = xd; a.yin = yd;
        for (int c = 0; c < kSubsetN[sub]; c++) a.out[c] = out[c];
        fill_spec_geom(h, a);
        if ((rc = ensure_twid(h, a.g, &a.twid))) return rc;
        CU(h, launch_spectral(a, SPEC_EVAL, mt, h->num_sms, h->stream));
        h->launches++;
        return SWRT_OK;
    }
    if (h->p.mode == SWRT_MODE_NUFFT) {
        REQUIRE(h, sub != SUB_PSI3, SWRT_ERR_ARG, "bad plane subset");
        const bool need_h = (sub == SUB_SEVEN || sub == SUB_UVH);
        const double *g = nullptr, *gh = nullptr;
        int rc = active_nufft_grid(h, alpha, &g, need_h ? &gh : nullptr);
        if (rc) return rc;
        REQUIRE(h, !need_h || gh, SWRT_ERR_STATE, "flow has no H plane (needed by this scheme)");
        NufftArgs a{};
        fill_nufft_args(h, g, a);
        a.hgrid = gh;
        fill_eval_io(a, sub, n, xd, yd, out);
        CU(h, launch_nufft_eval(a, h->stream));
        h->launches++;
        return SWRT_OK;
    }
    LagArgs a{};
    int rc = lag_frames(h, alpha, true, a);
    if (rc) return rc;
    REQUIRE(h, !(sub == SUB_SEVEN || sub == SUB_UVH) || h->grid_npl == 7, SWRT_ERR_STATE, "no H grid was set");
    fill_lag_args(h, a);
    fill_eval_io(a, sub, n, xd, yd, out);
    CU(h, launch_lagrange_eval(a, h->stream));
    h->launches++;
    return SWRT_OK;
}

int d2h(swrt_handle* h, double* dst, const double* src, int64_t n) {
    if (!dst || n == 0) return SWRT_OK;
    CU(h, cudaMemcpyAsync(dst, src, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    return SWRT_OK;
}
int h2d(swrt_handle* h, double* dst, const double* src, int64_t n) {
    if (n == 0) return SWRT_OK;
    CU(h, cudaMemcpyAsync(dst, src, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    return SWRT_OK;
}

// ---- cuFFT-backed g2k / k2g on the device (setup path) -------------------------------------------
__global__ void real_to_complex_kernel(const double* __restrict__ in, double2* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_double2(in[i], 0.0);
}
// g2k.m:5-9: keep kx=-kmax..kmax, ky=0..kmax of fft2(fg)/nx^2.  full[ky'*nx + kx'] (x fastest)
__global__ void extract_half_kernel(const double2* __restrict__ full, int nx, double2* __restrict__ half) {
    int nkx = nx - 1, nky = nx / 2, kmax = nx / 2 - 1;
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nkx * nky) return;
    int kx = idx % nkx - kmax, ky = idx / nkx;
    int ix = kx < 0 ? kx + nx : kx;
    double2 v = full[(size_t)ky * nx + ix];
    double s = 1.0 / ((double)nx * (double)nx);
    half[idx] = make_double2(v.x * s, v.y * s);
}
// fulspec.m:10-19 scattered into FFT order (no fftshift needed): full[ky'*nx + kx']
__global__ void fulspec_kernel(const double2* __restrict__ half, int nx, double2* __restrict__ full) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nx * nx) return;
    int nkx = nx - 1, kmax = nx / 2 - 1;
    int ixp = idx % nx, iyp = idx / nx;
    int kx = ixp <= nx / 2 ? ixp : ixp - nx;     // nx/2 is the (zeroed) Nyquist line
    int ky = iyp <= nx / 2 ? iyp : iyp - nx;
    double2 v = make_double2(0.0, 0.0);
    if (kx != nx / 2 && ky != nx / 2 && kx >= -kmax && ky >= -kmax) {
        if (ky > 0) v = half[(size_t)ky * nkx + kx + kmax];
        else if (ky < 0) { v = half[(size_t)(-ky) * nkx + (-kx) + kmax]; v.y = -v.y; }
        else {
            if (kx >= 0) v = half[kx + kmax];
            else { v = half[-kx + kmax]; v.y = -v.y; }
        }
    }
    full[idx] = v;
}
__global__ void take_real_kernel(const double2* __restrict__ in, double* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i].x;
}

struct FftWork {
    int nx = 0; cufftHandle plan = 0; bool has_plan = false; double2* full = nullptr;
    ~FftWork() { if (has_plan) cufftDestroy(plan); if (full) cudaFree(full); }
    int init(int nx_, cudaStream_t st, std::string& err) {
        nx = nx_;
        if (cudaMalloc(&full, (size_t)nx * nx * sizeof(double2)) != cudaSuccess) { err = "cudaMalloc(fft work) failed"; return SWRT_ERR_ALLOC; }
        if (cufftPlan2d(&plan, nx, nx, CUFFT_Z2Z) != CUFFT_SUCCESS) { err = "cufftPlan2d failed"; return SWRT_ERR_CUDA; }
        has_plan = true;
        cufftSetStream(plan, st);
        return SWRT_OK;
    }
};

// grid (device, column-major real) -> half-plane coefficients (device double2, kx fastest)
int g2k_dev(FftWork& w, const double* grid_dev, double2* half_dev, cudaStream_t st, std::string& err) {
    size_t n = (size_t)w.nx * w.nx;
    real_to_complex_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(grid_dev, w.full, n);
    if (cufftExecZ2Z(w.plan, (cufftDoubleComplex*)w.full, (cufftDoubleComplex*)w.full, CUFFT_FORWARD) != CUFFT_SUCCESS) {
        err = "cufftExecZ2Z(forward) failed"; return SWRT_ERR_CUDA;
    }
    int nh = (w.nx - 1) * (w.nx / 2);
    extract_half_kernel<<<(nh + 255) / 256, 256, 0, st>>>(w.full, w.nx, half_dev);
    return SWRT_OK;
}
int k2g_dev(FftWork& w, const double2* half_dev, double* grid_dev, cudaStream_t st, std::string& err) {
    size_t n = (size_t)w.nx * w.nx;
    fulspec_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(half_dev, w.nx, w.full);
    if (cufftExecZ2Z(w.plan, (cufftDoubleComplex*)w.full, (cufftDoubleComplex*)w.full, CUFFT_INVERSE) != CUFFT_SUCCESS) {
        err = "cufftExecZ2Z(inverse) failed"; return SWRT_ERR_CUDA;
    }
    take_real_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w.full, grid_dev, n);
    return SWRT_OK;
}

__global__ void interleave_complex_kernel(const double* __restrict__ re, const double* __restrict__ im,
                                          double2* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_double2(re[i], im ? im[i] : 0.0);
}

// upload a host complex plane (separate re/im) into a device double2 plane
int upload_plane(swrt_handle* h, const double* re, const double* im, size_t n, double2** dst, double* tmp_re,
                 double* tmp_im) {
    if (!*dst) CU(h, cudaMalloc(dst, n * sizeof(double2)));
    CU(h, cudaMemcpyAsync(tmp_re, re, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (im) CU(h, cudaMemcpyAsync(tmp_im, im, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    interleave_complex_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(tmp_re, im ? tmp_im : nullptr, *dst, n);
    h->launches++;
    return SWRT_OK;
}

// ---- NUFFT mode set-up ---------------------------------------------------------------------------
// Gauss-Legendre nodes/weights on [-1,1] (Newton iteration on P_n)
static void gauss_legendre(int n, std::vector<double>& x, std::vector<double>& w) {
    x.assign(n, 0.0); w.assign(n, 0.0);
    for (int i = 0; i < (n + 1) / 2; i++) {
        double z = cos(M_PI * (i + 0.75) / (n + 0.5)), pp = 1.0;
        for (int it = 0; it < 100; it++) {
            double p1 = 1.0, p2 = 0.0;
            for (int j = 0; j < n; j++) { const double p3 = p2; p2 = p1; p1 = ((2.0 * j + 1.0) * z * p2 - j * p3) / (j + 1.0); }
            pp = n * (z * p1 - p2) / (z * z - 1.0);
            const double z1 = z; z = z1 - p1 / pp;
            if (fabs(z - z1) < 1e-16) break;
        }
        x[i] = -z; x[n - 1 - i] = z;
        w[i] = w[n - 1 - i] = 2.0 / ((1.0 - z * z) * pp * pp);
    }
}
// 1 / phihat(k), k = 0..kmax: phihat(k) = (w/2) * int_{-1}^{1} phi(z) cos(2 pi k (w/2) z / nf) dz  (unit fine-grid spacing)
static int nufft_init(swrt_handle* h) {
    if (h->nufft_invphi) return SWRT_OK;
    const int nx = h->p.nx, nf = (int)(kNufftSigma * nx), nky = nx / 2;
    std::vector<double> q, wq, inv(nky);
    gauss_legendre(128, q, wq);
    const double hw = kNufftW / 2.0;
    for (int k = 0; k < nky; k++) {
        double acc = 0.0;
        for (size_t j = 0; j < q.size(); j++) {
            const double phi = exp(kNufftBeta * (sqrt(fmax(0.0, 1.0 - q[j] * q[j])) - 1.0));
            acc += wq[j] * phi * cos(2.0 * M_PI * k * hw * q[j] / nf);
        }
        inv[k] = 1.0 / (hw * acc);
    }
    CU(h, cudaMalloc(&h->nufft_invphi, nky * sizeof(double)));
    CU(h, cudaMemcpy(h->nufft_invphi, inv.data(), nky * sizeof(double), cudaMemcpyHostToDevice));
    FftWork* fw = new (std::nothrow) FftWork();
    REQUIRE(h, fw, SWRT_ERR_ALLOC, "out of host memory");
    h->nufft_fft = fw;
    return fw->init(nf, h->stream, h->err);
}
// fine (u,v) grid of a slot from its u-hat, v-hat planes: deconvolve, zero-pad to nf, inverse FFT, interleave
int nufft_grid_from_planes(swrt_handle* h, int slot) {
    int rc = nufft_init(h);
    if (rc) return rc;
    const int nx = h->p.nx, nf = (int)(kNufftSigma * nx);
    const size_t n = (size_t)nf * nf;
    if (!h->nufft_grid[slot]) CU(h, cudaMalloc(&h->nufft_grid[slot], 2 * n * sizeof(double)));
    FftWork* fw = static_cast<FftWork*>(h->nufft_fft);
    cufftSetStream(fw->plan, h->stream);
    // flows that carry H = 1 + eta_g (raytrace_sw.m:49) also get a fine grid of 32-byte (u, v, H, 0) nodes, so that the
    // evaluations of step_packet_xka fetch a node with one 256-bit load
    const bool with_h = h->slot_npl[slot] == 7;
    if (with_h && !h->nufft_h[slot]) {
        CU(h, cudaMalloc(&h->nufft_h[slot], 4 * n * sizeof(double)));
        CU(h, cudaMemsetAsync(h->nufft_h[slot], 0, 4 * n * sizeof(double), h->stream));
    }
    if (!with_h) dfree(h->nufft_h[slot]);
    for (int c = 0; c < (with_h ? 3 : 2); c++) {
        launch_nufft_spread(h->planes[slot][c < 2 ? c : 6], nx, nf, h->nufft_invphi, fw->full, h->stream);
        if (cufftExecZ2Z(fw->plan, (cufftDoubleComplex*)fw->full, (cufftDoubleComplex*)fw->full, CUFFT_INVERSE) != CUFFT_SUCCESS)
            return fail(h, SWRT_ERR_CUDA, "cufftExecZ2Z(nufft) failed");
        if (c < 2) { launch_nufft_store(fw->full, nf, c, 2, h->nufft_grid[slot], h->stream); h->launches++; }
        if (with_h) { launch_nufft_store(fw->full, nf, c, 4, h->nufft_h[slot], h->stream); h->launches++; }
        h->launches += 2;
    }
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaGetLastError());
    return SWRT_OK;
}
// fine grids holding (1-alpha)*slot0 + alpha*slot1; *hout is null when no H plane was set (or not wanted)
int active_nufft_grid(swrt_handle* h, double alpha, const double** out, const double** hout) {
    REQUIRE(h, h->nufft_grid[0], SWRT_ERR_STATE, "flow slot 0 has not been set");
    const bool want_h = hout != nullptr;
    if (want_h) *hout = nullptr;
    if (alpha == 0.0) { *out = h->nufft_grid[0]; if (want_h) *hout = h->nufft_h[0]; return SWRT_OK; }
    REQUIRE(h, h->nufft_grid[1] && h->slot_set[1], SWRT_ERR_STATE, "alpha = %g but flow slot 1 has not been set", alpha);
    if (alpha == 1.0) { *out = h->nufft_grid[1]; if (want_h) *hout = h->nufft_h[1]; return SWRT_OK; }
    const int nf = (int)(kNufftSigma * h->p.nx);
    const size_t nd = (size_t)2 * nf * nf;
    if (!h->nufft_blend) CU(h, cudaMalloc(&h->nufft_blend, nd * sizeof(double)));
    launch_axpby(h->nufft_blend, h->nufft_grid[0], h->nufft_grid[1], 1.0 - alpha, alpha, nd, h->stream);   // interpolate_U.m:19-23
    h->launches++;
    *out = h->nufft_blend;
    if (want_h && h->nufft_h[0] && h->nufft_h[1]) {
        if (!h->nufft_hblend) CU(h, cudaMalloc(&h->nufft_hblend, 2 * nd * sizeof(double)));
        launch_axpby(h->nufft_hblend, h->nufft_h[0], h->nufft_h[1], 1.0 - alpha, alpha, 2 * nd, h->stream);   // (u,v,H,0) nodes
        h->launches++;
        *hout = h->nufft_hblend;
    }
    return SWRT_OK;
}
void fill_nufft_args(const swrt_handle* h, const double* grid, NufftArgs& a) {
    a.grid = reinterpret_cast<const double2*>(grid);
    a.nf = (int)(kNufftSigma * h->p.nx);
    a.dx = h->p.L / h->p.nx; a.nxd = (double)h->p.nx; a.beta = kNufftBeta;
    a.dscale = -kNufftSigma / (a.dx * (kNufftW / 2.0));
    a.f2 = h->p.f * h->p.f; a.gH = h->p.gH;
}

// the handle's nx-point FFT work area and plan, created on first use (plan creation costs ~1 ms: a per-call plan
// dominated every flow upload of the time-evolving drivers)
static int handle_fft(swrt_handle* h, FftWork** out) {
    if (!h->grid_fft) {
        FftWork* fw = new (std::nothrow) FftWork();
        REQUIRE(h, fw, SWRT_ERR_ALLOC, "out of host memory");
        int rc = fw->init(h->p.nx, h->stream, h->err);
        if (rc) { delete fw; return fail(h, rc, "FFT plan: %s", h->err.c_str()); }
        h->grid_fft = fw;
    }
    *out = static_cast<FftWork*>(h->grid_fft);
    cufftSetStream((*out)->plan, h->stream);
    return SWRT_OK;
}

// build the Lagrange grid of a slot from its spectral planes (k2g of every plane): grid_U.m:11-17
int grid_from_planes(swrt_handle* h, int slot) {
    const int nx = h->p.nx, npl = h->slot_npl[slot];
    FftWork* wp = nullptr;
    int rc = handle_fft(h, &wp);
    if (rc) return rc;
    FftWork& w = *wp;
    std::vector<double*> tmp(npl, nullptr);
    size_t n = (size_t)nx * nx;
    if (!h->grid_tmp) CU(h, cudaMalloc(&h->grid_tmp, (size_t)kMaxPlanes * n * sizeof(double)));
    for (int c = 0; c < npl; c++) {
        tmp[c] = h->grid_tmp + (size_t)c * n;
        rc = k2g_dev(w, h->planes[slot][c], tmp[c], h->stream, h->err);
        if (rc) return rc;
        h->launches += 3;
    }
    if (h->grid_npl != npl) {      // the plane count changed: the other slot's grid no longer matches and must be set again
        dfree(h->grid[0]); dfree(h->grid[1]); dfree(h->grid_blend); h->grid_npl = npl;
        h->slot_set[1 - slot] = false;
    }
    if (!h->grid[slot]) CU(h, cudaMalloc(&h->grid[slot], n * npl * sizeof(double)));
    launch_interleave_grid(tmp.data(), npl, nx, h->grid[slot], h->stream);
    h->launches++;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int swrt_version(void) { return SWRT_VERSION; }

int swrt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* swrt_last_error(const swrt_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int swrt_create(const swrt_params* p, swrt_handle** out) {
    if (!p || !out) return fail(nullptr, SWRT_ERR_ARG, "swrt_create: null argument");
    *out = nullptr;
    if (p->nx < 8 || (p->nx & 1)) return fail(nullptr, SWRT_ERR_ARG, "swrt_create: nx must be even and >= 8 (got %d)", p->nx);
    if (!(p->L > 0)) return fail(nullptr, SWRT_ERR_ARG, "swrt_create: L must be positive");
    if (p->mode != SWRT_MODE_SPECTRAL && p->mode != SWRT_MODE_LAGRANGE6 && p->mode != SWRT_MODE_NUFFT)
        return fail(nullptr, SWRT_ERR_ARG, "swrt_create: unknown mode %d", p->mode);
    if (p->ngpu < 0 || p->ngpu > 64) return fail(nullptr, SWRT_ERR_ARG, "swrt_create: ngpu = %d out of range", p->ngpu);
    if (p->ngpu > 1) return grp_create(p, out);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, SWRT_ERR_CUDA, "swrt_create: no CUDA device (%s); libswrt has no CPU path",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    }
    if (p->device < 0 || p->device >= ndev) return fail(nullptr, SWRT_ERR_ARG, "swrt_create: device %d out of range", p->device);
    if (cudaSetDevice(p->device) != cudaSuccess) return fail(nullptr, SWRT_ERR_CUDA, "cudaSetDevice failed");
    swrt_handle* h = new (std::nothrow) swrt_handle();
    if (!h) return fail(nullptr, SWRT_ERR_ALLOC, "out of host memory");
    h->p = *p;
    if (!(h->p.bump > 0)) h->p.bump = 1e-13;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, p->device) != cudaSuccess) {
        delete h;
        return fail(nullptr, SWRT_ERR_CUDA, "swrt_create: cudaGetDeviceProperties failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    h->num_sms = prop.multiProcessorCount;
    if (prop.major < 10) {
        delete h;
        return fail(nullptr, SWRT_ERR_CUDA, "swrt_create: device is sm_%d%d; libswrt is built for sm_100a only", prop.major, prop.minor);
    }
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess ||
        cudaEventCreate(&h->tm0) != cudaSuccess || cudaEventCreate(&h->tm1) != cudaSuccess ||
        cudaMalloc(&h->diag_dev, (8 + 296 * 8) * sizeof(double)) != cudaSuccess) {
        swrt_destroy(h);
        return fail(nullptr, SWRT_ERR_CUDA, "swrt_create: stream/event/alloc failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    h->stream = h->own_stream;
    *out = h;
    return SWRT_OK;
}

int swrt_destroy(swrt_handle* h) {
    if (!h) return SWRT_OK;
    if (h->ngpu > 1) return grp_destroy(h);
    cudaSetDevice(h->p.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    stager_free(h);
    dfree(h->arena); dfree(h->arena_h); dfree(h->red_dev); dfree(h->twid);
    dfree(h->x); dfree(h->y); dfree(h->k); dfree(h->l); dfree(h->a);
    for (int s = 0; s < 2; s++) {
        for (auto& p : h->planes[s]) dfree(p);
        dfree(h->grid[s]);
    }
    dfree(h->grid_blend);
    dfree(h->nufft_grid[0]); dfree(h->nufft_grid[1]); dfree(h->nufft_blend); dfree(h->nufft_invphi);
    dfree(h->nufft_h[0]); dfree(h->nufft_h[1]); dfree(h->nufft_hblend);
    if (h->nufft_fft) { delete static_cast<FftWork*>(h->nufft_fft); h->nufft_fft = nullptr; }
    if (h->grid_fft) { delete static_cast<FftWork*>(h->grid_fft); h->grid_fft = nullptr; }
    dfree(h->grid_tmp);
    for (auto& st : h->stacks) { dfree(st.slot[0]); dfree(st.slot[1]); dfree(st.blend); }
    dfree(h->anc_key); dfree(h->anc_rank); dfree(h->anc_perm);
    dfree(h->anc_cnt); dfree(h->anc_off);
    dfree(h->anc_hexp);
    for (auto& p : h->e) dfree(p);
    dfree(h->xs); dfree(h->ys); dfree(h->ax); dfree(h->ay); dfree(h->om); dfree(h->Om);
    dfree(h->diag_dev); dfree(h->edges_dev); dfree(h->counts_dev); dfree(h->bs_norm_dev);
    dfree(h->h2_edges_dev); dfree(h->h2_counts_dev); dfree(h->ws_exp_dev); dfree(h->h2s_acc_dev);
    for (auto& p : h->bs_yt) dfree(p);
    for (auto& row : h->bs_f) for (auto& p : row) dfree(p);
    dfree(h->ode_ctl);
    if (h->ode_host) cudaFreeHost(h->ode_host);
    dfree(h->pkt_d); dfree(h->pkt_i); dfree(h->pkt_e1); dfree(h->ev_d); dfree(h->ev_i);
    if (h->pkt_rep_host) cudaFreeHost(h->pkt_rep_host);
    if (h->ode_ev) cudaEventDestroy(h->ode_ev);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->hist_ev) cudaEventDestroy(h->hist_ev);
    if (h->tm0) cudaEventDestroy(h->tm0);
    if (h->tm1) cudaEventDestroy(h->tm1);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return SWRT_OK;
}

// ---- flow upload ------------------------------------------------------------------------------
static int finish_spectral_slot(swrt_handle* h, int slot, int npl) {
    h->psi_ok[slot] = false;
    h->slot_set[slot] = true;
    h->slot_npl[slot] = npl;
    invalidate_slot(h, slot);
    if (h->p.mode == SWRT_MODE_LAGRANGE6) return grid_from_planes(h, slot);
    if (h->p.mode == SWRT_MODE_NUFFT) return nufft_grid_from_planes(h, slot);
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

// psi-hat already on the device (double2, g2k layout) -> six planes + moment planes of a slot
static int set_flow_spectral_dev(swrt_handle* h, int slot, const double2* psi, double u_mean) {
    const int nkx = h->p.nx - 1, nky = h->p.nx / 2;
    const size_t n = (size_t)nkx * nky;
    int rc = SWRT_OK;
    for (int c = 0; c < 6 && rc == SWRT_OK; c++)
        if (!h->planes[slot][c] && cudaMalloc(&h->planes[slot][c], n * sizeof(double2)) != cudaSuccess)
            rc = fail(h, SWRT_ERR_ALLOC, "cudaMalloc(plane) failed");
    if (rc) return rc;
    dfree(h->planes[slot][6]);
    // wavenumbers kappa*kx: integers when L = 2*pi (SpectralScheme.m:12-25), 2*pi/L-scaled
    // otherwise (qg2layersw_raytrace.m:19-22)
    const double kappa = 2.0 * M_PI / h->p.L;
    launch_psi_to_planes(psi, h->planes[slot], nkx, nky, kappa, u_mean, h->stream);
    h->launches++;
    for (int c = 7; c < 10 && rc == SWRT_OK; c++)
        if (!h->planes[slot][c] && cudaMalloc(&h->planes[slot][c], n * sizeof(double2)) != cudaSuccess)
            rc = fail(h, SWRT_ERR_ALLOC, "cudaMalloc(moment plane) failed");
    if (rc) return rc;
    launch_psi_moments(psi, h->planes[slot][7], h->planes[slot][8], h->planes[slot][9], nkx, nky, h->stream);
    h->launches++;
    rc = finish_spectral_slot(h, slot, 6);
    if (rc == SWRT_OK) { h->psi_ok[slot] = true; h->u_mean[slot] = u_mean; }
    return rc;
}

// multi-device handle, psi-hat already on the first device (the QG producers): the first shard takes it in place, the
// others receive a peer copy (a frame is <= 2 MB: setup traffic, once per flow step)
static int grp_flow_from_psi_dev(swrt_handle* g, int slot, const double2* psi_dev0, double u_mean) {
    const size_t n = (size_t)(g->p.nx - 1) * (g->p.nx / 2);
    for (size_t i = 0; i < g->shard.size(); i++) {
        swrt_handle* c = g->shard[i];
        CU(g, cudaSetDevice(c->p.device));
        int rc;
        if (i == 0) rc = set_flow_spectral_dev(c, slot, psi_dev0, u_mean);
        else {
            DevTmp<double2> tmp;
            CU(g, tmp.alloc(n));
            CU(g, cudaMemcpyPeer(tmp.p, c->p.device, psi_dev0, g->shard[0]->p.device, n * sizeof(double2)));
            rc = set_flow_spectral_dev(c, slot, tmp.p, u_mean);
            cudaStreamSynchronize(c->stream);
        }
        if (rc) return up(g, c, rc);
    }
    g->slot_set[slot] = true;
    return SWRT_OK;
}

int swrt_set_flow_spectral(swrt_handle* h, int slot, const double* psik_re, const double* psik_im, int nkx, int nky,
                           double u_mean) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) {
        for (swrt_handle* c : h->shard) { int rc = swrt_set_flow_spectral(c, slot, psik_re, psik_im, nkx, nky, u_mean); if (rc) return up(h, c, rc); }
        h->slot_set[slot] = true;
        return SWRT_OK;
    }
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, slot == 0 || slot == 1, SWRT_ERR_ARG, "slot must be 0 or 1");
    REQUIRE(h, psik_re && psik_im, SWRT_ERR_ARG, "null psi-hat pointer");
    REQUIRE(h, nkx == h->p.nx - 1 && nky == h->p.nx / 2, SWRT_ERR_ARG, "psi-hat must be %d x %d (got %d x %d)",
            h->p.nx - 1, h->p.nx / 2, nkx, nky);
    size_t n = (size_t)nkx * nky;
    DevTmp<double> tr, ti;
    DevTmp<double2> psi;
    CU(h, tr.alloc(n)); CU(h, ti.alloc(n)); CU(h, psi.alloc(n));
    int rc = upload_plane(h, psik_re, psik_im, n, &psi.p, tr.p, ti.p);
    if (rc == SWRT_OK) rc = set_flow_spectral_dev(h, slot, psi.p, u_mean);
    cudaStreamSynchronize(h->stream);
    return rc;
}

int swrt_set_flow_planes_spectral(swrt_handle* h, int slot, const double* const* planes_re,
                                  const double* const* planes_im, int nplanes, int nkx, int nky) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) {
        for (swrt_handle* c : h->shard) { int rc = swrt_set_flow_planes_spectral(c, slot, planes_re, planes_im, nplanes, nkx, nky); if (rc) return up(h, c, rc); }
        h->slot_set[slot] = true;
        return SWRT_OK;
    }
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, slot == 0 || slot == 1, SWRT_ERR_ARG, "slot must be 0 or 1");
    REQUIRE(h, nplanes == 6 || nplanes == 7, SWRT_ERR_ARG, "nplanes must be 6 or 7");
    REQUIRE(h, planes_re && planes_im, SWRT_ERR_ARG, "null plane table");
    REQUIRE(h, nkx == h->p.nx - 1 && nky == h->p.nx / 2, SWRT_ERR_ARG, "planes must be %d x %d", h->p.nx - 1, h->p.nx / 2);
    size_t n = (size_t)nkx * nky;
    DevTmp<double> tr, ti;
    CU(h, tr.alloc(n)); CU(h, ti.alloc(n));
    int rc = SWRT_OK;
    for (int c = 0; c < nplanes && rc == SWRT_OK; c++) {
        if (!planes_re[c] || !planes_im[c]) { rc = fail(h, SWRT_ERR_ARG, "null plane %d", c); break; }
        rc = upload_plane(h, planes_re[c], planes_im[c], n, &h->planes[slot][c], tr.p, ti.p);
        if (rc == SWRT_OK && cudaStreamSynchronize(h->stream) != cudaSuccess) rc = fail(h, SWRT_ERR_CUDA, "sync failed");
    }
    if (nplanes == 6) dfree(h->planes[slot][6]);
    if (rc == SWRT_OK) rc = finish_spectral_slot(h, slot, nplanes);
    return rc;
}

int swrt_set_flow_grid(swrt_handle* h, int slot, const double* u, const double* v, const double* ux, const double* uy,
                       const double* vx, const double* vy, const double* H, int nx) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) {
        for (swrt_handle* c : h->shard) { int rc = swrt_set_flow_grid(c, slot, u, v, ux, uy, vx, vy, H, nx); if (rc) return up(h, c, rc); }
        h->slot_set[slot] = true;
        return SWRT_OK;
    }
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, slot == 0 || slot == 1, SWRT_ERR_ARG, "slot must be 0 or 1");
    REQUIRE(h, nx == h->p.nx, SWRT_ERR_ARG, "grid is %d^2 but the handle was created with nx = %d", nx, h->p.nx);
    REQUIRE(h, u && v && ux && uy && vx && vy, SWRT_ERR_ARG, "null grid plane");
    const double* src[kMaxPlanes] = {u, v, ux, uy, vx, vy, H};
    const int npl = H ? 7 : 6;
    size_t n = (size_t)nx * nx;
    std::vector<DevTmp<double>> tmpbuf(npl);
    std::vector<double*> tmp(npl, nullptr);
    int rc = SWRT_OK;
    for (int c = 0; c < npl; c++) {
        CU(h, tmpbuf[c].alloc(n));
        tmp[c] = tmpbuf[c].p;
        CU(h, cudaMemcpyAsync(tmp[c], src[c], n * 8, cudaMemcpyHostToDevice, h->stream));
    }
    if (h->p.mode == SWRT_MODE_LAGRANGE6) {
        if (h->grid_npl != npl) {
            dfree(h->grid[0]); dfree(h->grid[1]); dfree(h->grid_blend); h->grid_npl = npl;
            h->slot_set[1 - slot] = false;
        }
        if (!h->grid[slot]) CU(h, cudaMalloc(&h->grid[slot], n * npl * 8));
        launch_interleave_grid(tmp.data(), npl, nx, h->grid[slot], h->stream);
        h->launches++;
        h->slot_set[slot] = true; h->slot_npl[slot] = npl;
    } else {
        // SPECTRAL / NUFFT mode: g2k of every plane on the device (g2k.m:5-9)
        FftWork* wp = nullptr;
        rc = handle_fft(h, &wp);
        if (rc) return rc;
        FftWork& w = *wp;
        size_t nh = (size_t)(nx - 1) * (nx / 2);
        for (int c = 0; c < npl && rc == SWRT_OK; c++) {
            if (!h->planes[slot][c] && cudaMalloc(&h->planes[slot][c], nh * sizeof(double2)) != cudaSuccess) {
                rc = fail(h, SWRT_ERR_ALLOC, "cudaMalloc(plane) failed"); break;
            }
            rc = g2k_dev(w, tmp[c], h->planes[slot][c], h->stream, h->err);
            h->launches += 3;
        }
        if (npl == 6) dfree(h->planes[slot][6]);
        if (rc == SWRT_OK) { h->slot_set[slot] = true; h->slot_npl[slot] = npl; h->psi_ok[slot] = false; invalidate_slot(h, slot); }
        cudaStreamSynchronize(h->stream);
        if (rc == SWRT_OK && h->p.mode == SWRT_MODE_NUFFT) rc = nufft_grid_from_planes(h, slot);
    }
    cudaStreamSynchronize(h->stream);              // the temporaries are released on return
    if (rc == SWRT_OK) CU(h, cudaGetLastError());
    return rc;
}

// ---- evaluation -------------------------------------------------------------------------------
int swrt_eval(swrt_handle* h, double alpha, double* U, double* V, double* Ux, double* Uy, double* Vx, double* Vy) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_each_slice(h, [&](swrt_handle* c, int64_t lo) {
        return swrt_eval(c, alpha, at(U, lo), at(V, lo), at(Ux, lo), at(Uy, lo), at(Vx, lo), at(Vy, lo)); }));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "no flow has been set");
    int rc = ensure_scratch(h, h->n);
    if (rc) return rc;
    CU(h, cudaEventRecord(h->ev0, h->stream));
    if ((rc = eval_dev(h, SUB_SIX, alpha, h->n, h->x, h->y, h->e))) return rc;
    CU(h, cudaEventRecord(h->ev1, h->stream));
    h->timing_valid = true; h->last_nlaunch = 1;
    double* outs[6] = {U, V, Ux, Uy, Vx, Vy};
    for (int c = 0; c < 6; c++)
        if ((rc = d2h(h, outs[c], h->e[c], h->n))) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

int swrt_eval_at(swrt_handle* h, double alpha, int64_t n, const double* x, const double* y, double* U, double* V,
                 double* Ux, double* Uy, double* Vx, double* Vy, double* H) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) {   // caller-given points, independent of the packet state: the first device serves them
        int rc = swrt_eval_at(h->shard[0], alpha, n, x, y, U, V, Ux, Uy, Vx, Vy, H);
        return up(h, h->shard[0], rc);
    }
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, n >= 0 && (n == 0 || (x && y)), SWRT_ERR_ARG, "bad positions");
    REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "no flow has been set");
    if (n == 0) return SWRT_OK;
    int rc = ensure_scratch(h, n);
    if (rc) return rc;
    if ((rc = h2d(h, h->xs, x, n)) || (rc = h2d(h, h->ys, y, n))) return rc;
    const int sub = H ? SUB_SEVEN : SUB_SIX;
    if ((rc = eval_dev(h, sub, alpha, n, h->xs, h->ys, h->e))) return rc;
    double* outs[7] = {U, V, Ux, Uy, Vx, Vy, H};
    for (int c = 0; c < 7; c++)
        if ((rc = d2h(h, outs[c], h->e[c], n))) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

// odefun uses Cg (not Cg^2) in the production drivers (qgsw_raytrace.m:262, qg2layersw_raytrace.m:301) and gH in
// SW_zero_background_raytracing.m:182-184 (SWRT_FLAG_RHS_GH)
static inline double rhs_cgfac(const swrt_handle* h) { return (h->p.flags & SWRT_FLAG_RHS_GH) ? h->p.gH : sqrt(h->p.gH); }

int swrt_rhs(swrt_handle* h, double alpha, double* dxdt, double* dydt, double* dkdt, double* dldt) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_each_slice(h, [&](swrt_handle* c, int64_t lo) {
        return swrt_rhs(c, alpha, at(dxdt, lo), at(dydt, lo), at(dkdt, lo), at(dldt, lo)); }));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "no flow has been set");
    int rc = ensure_scratch(h, h->n);
    if (rc) return rc;
    if ((rc = eval_dev(h, SUB_SIX, alpha, h->n, h->x, h->y, h->e))) return rc;
    double* const fj[4] = {h->xs, h->ys, h->ax, h->ay};
    launch_rhs(Ode23ValView{}, 0, h->n, h->k, h->l, h->e, nullptr, h->p.f, h->p.gH, rhs_cgfac(h), fj, h->stream);
    h->launches++;
    if ((rc = d2h(h, dxdt, h->xs, h->n)) || (rc = d2h(h, dydt, h->ys, h->n)) || (rc = d2h(h, dkdt, h->ax, h->n)) ||
        (rc = d2h(h, dldt, h->ay, h->n)))
        return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

int swrt_interpolate(int device, const double* x, const double* y, int64_t n, const double* F, int nx, int ny,
                     double dx, double dy, double bump, double* FI) {
    if (!x || !y || !F || !FI || n < 0 || nx < 1 || ny < 1) return fail(nullptr, SWRT_ERR_ARG, "swrt_interpolate: bad argument");
    // interpolate.m:45-46 wraps BOTH stencil indices with nx, so F(ig,jg) reads columns up to nx: for an nx x ny array with
    // ny < nx MATLAB raises "index exceeds array bounds"; here that is an argument error, never an out-of-bounds read
    if (ny < nx) return fail(nullptr, SWRT_ERR_ARG, "swrt_interpolate: F is %d x %d but the stencil wraps both indices with nx (interpolate.m:45-46): "
                                                    "ny >= nx is required", nx, ny);
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail(nullptr, SWRT_ERR_CUDA, "swrt_interpolate: no CUDA device"); }
    if (n == 0) return SWRT_OK;
    DevTmp<double> dF, dx_, dy_, dout;
    const size_t nb = (size_t)n * 8, gb = (size_t)nx * ny * 8;
    if (dF.alloc((size_t)nx * ny) || dx_.alloc(n) || dy_.alloc(n) || dout.alloc(n)) {
        cudaGetLastError();
        return fail(nullptr, SWRT_ERR_ALLOC, "swrt_interpolate: cudaMalloc failed");
    }
    cudaError_t e = cudaMemcpy(dF.p, F, gb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dx_.p, x, nb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dy_.p, y, nb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_interpolate_single(dF.p, nx, ny, dx_.p, dy_.p, n, dx, dy, bump > 0 ? bump : 1e-13, dout.p, 0);
    if (e == cudaSuccess) e = cudaMemcpy(FI, dout.p, nb, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(nullptr, SWRT_ERR_CUDA, "swrt_interpolate: %s", cudaGetErrorString(e));
    return SWRT_OK;
}

}  // extern "C"

// ---- stepping ---------------------------------------------------------------------------------
// A "run" is up to m consecutive steps of one scheme executed by ONE launch per packet range with the packet in
// registers.  Steady flow: the whole call is one run.  Time-dependent flow (dalpha != 0): the operands of every step of the
// run -- packed stacks (SPECTRAL), fine grids (NUFFT), gridded frames (LAGRANGE6 RK4 / pre-blend tuning) -- are blended on
// the device at al_j = alpha0 + j*dalpha by ONE multi-blend launch and stored back to back in the handle's arena; the
// kernels read operand j in step j.  LAGRANGE6 leapfrog keeps interpolate_U.m's exact semantics instead (both frames
// gathered, results blended with al_j inside the kernel).
constexpr int kMaxFusedBlend = 32;

struct RunOps {
    int scheme = 0, m = 0;
    bool xka = false, composed = false;
    bool anchored = false;                // SPECTRAL leapfrog through K1 + K2 (run_anchored)
    double dt = 0, alpha0 = 0, dalpha = 0;
    int j0 = 0, mt = 1;
    SpecArgs sa{};
    SpecRk4Args ra{};
    NufftArgs na{};
    LagArgs la{};
};

static int ensure_arena(swrt_handle* h, double*& p, size_t& cap, size_t doubles) {
    if (doubles <= cap) return SWRT_OK;
    dfree(p); cap = 0;
    CU(h, cudaMalloc(&p, doubles * sizeof(double)));
    cap = doubles;
    return SWRT_OK;
}

// The SPECTRAL leapfrog on a psi-hat flow runs anchored (K1 per anchor cell, K2 per packet) on the grids
// anchor_log2_cells accepts; the choice depends on the grid, the scheme and the flow form only, never on the packet count,
// so that a packet's result is the same in every ensemble it is part of.
static bool anchored_leapfrog(const swrt_handle* h, int scheme, double alpha0, double dalpha) {
    return h->p.mode == SWRT_MODE_SPECTRAL && scheme == SWRT_SCHEME_LEAPFROG && anchor_log2_cells(h->p.nx) > 0 &&
           use_psi(h, dalpha != 0.0 ? 0.5 : alpha0);
}

static int ensure_anchor(swrt_handle* h, int64_t n, int nanc, size_t hexp_doubles) {
    if (n > h->anc_cap) {
        dfree(h->anc_key); dfree(h->anc_rank); dfree(h->anc_perm);
        h->anc_cap = 0;
        CU(h, cudaMalloc(&h->anc_key, (size_t)n * sizeof(int)));
        CU(h, cudaMalloc(&h->anc_rank, (size_t)n * sizeof(unsigned long long)));
        CU(h, cudaMalloc(&h->anc_perm, (size_t)n * sizeof(long long)));
        h->anc_cap = n;
    }
    if (nanc != h->anc_n) {
        dfree(h->anc_cnt); dfree(h->anc_off);
        h->anc_n = 0;
        CU(h, cudaMalloc(&h->anc_cnt, (size_t)nanc * sizeof(unsigned long long)));
        CU(h, cudaMalloc(&h->anc_off, (size_t)nanc * sizeof(unsigned long long)));
        h->anc_n = nanc;
    }
    return ensure_arena(h, h->anc_hexp, h->anc_hexp_cap, hexp_doubles);
}

// operands of steps j0 .. j0+m-1 of swrt_step(scheme, dt, ., alpha0, dalpha); blends are queued on h->stream
static int prepare_run(swrt_handle* h, int scheme, double dt, double alpha0, double dalpha, int j0, int m, RunOps& r) {
    int rc;
    const bool td = (dalpha != 0.0);
    const double alpha_first = alpha0 + j0 * dalpha;          // = alpha0 when the flow is steady
    r.scheme = scheme; r.m = m; r.xka = (scheme == SWRT_SCHEME_RK4_XKA);
    r.dt = dt; r.alpha0 = alpha0; r.dalpha = dalpha; r.j0 = j0;
    const double C0 = sqrt(h->p.gH);
    const int mode = h->p.mode;
    if (td) REQUIRE(h, h->slot_set[1], SWRT_ERR_STATE, "dalpha = %g but flow slot 1 has not been set", dalpha);
    if (mode == SWRT_MODE_SPECTRAL && scheme == SWRT_SCHEME_LEAPFROG) {
        SpecArgs& a = r.sa;
        r.anchored = anchored_leapfrog(h, scheme, alpha_first, dalpha);
        r.mt = r.anchored ? 1 : pick_mtiles(h, h->n);          // K1 reads the one-m-tile stack
        const bool psi = use_psi(h, td ? 0.5 : alpha_first);
        const int sub = psi ? SUB_PSI3 : SUB_SIX;
        if (!td) {
            if ((rc = active_stack(h, sub, alpha_first, r.mt, &a.stack, &a.g))) return rc;
            a.nstack = 1;
        } else {
            if ((rc = ensure_stack(h, sub, 0, r.mt)) || (rc = ensure_stack(h, sub, 1, r.mt))) return rc;
            Stack& s = h->stacks[sub];
            a.g = s.g;
            if ((rc = ensure_arena(h, h->arena, h->arena_cap, (size_t)m * s.g.total_doubles))) return rc;
            launch_axpby_multi(h->arena, s.slot[0], s.slot[1], alpha0, dalpha, j0, m, s.g.total_doubles, h->stream);
            h->launches++;
            a.stack = h->arena; a.nstack = m;
        }
        if (psi) { a.psi = true; a.kappa = 2.0 * M_PI / h->p.L; a.u_mean0 = h->u_mean[0]; a.u_mean1 = h->slot_set[1] ? h->u_mean[1] : 0.0; }
        a.alpha0 = alpha0; a.dalpha = dalpha; a.j0 = j0;
        a.x = h->x; a.y = h->y; a.k = h->k; a.l = h->l;
        fill_spec_geom(h, a);
        a.f2 = h->p.f * h->p.f; a.gH = h->p.gH; a.dt = dt; a.nsteps = m;
        return SWRT_OK;
    }
    if (mode == SWRT_MODE_NUFFT && (scheme == SWRT_SCHEME_LEAPFROG || !h->unfused_rk4)) {
        NufftArgs& a = r.na;
        const double *g = nullptr, *gh = nullptr;
        const size_t nd = (size_t)2 * (size_t)(kNufftSigma * h->p.nx) * (size_t)(kNufftSigma * h->p.nx);   // doubles per (u,v) grid
        if (!td) {
            if ((rc = active_nufft_grid(h, alpha_first, &g, r.xka ? &gh : nullptr))) return rc;
        } else {
            REQUIRE(h, h->nufft_grid[0] && h->nufft_grid[1], SWRT_ERR_STATE, "both flow slots must be set");
            if ((rc = ensure_arena(h, h->arena, h->arena_cap, (size_t)m * nd))) return rc;
            launch_axpby_multi(h->arena, h->nufft_grid[0], h->nufft_grid[1], alpha0, dalpha, j0, m, nd, h->stream);
            h->launches++;
            g = h->arena;
            if (r.xka && h->nufft_h[0] && h->nufft_h[1]) {
                if ((rc = ensure_arena(h, h->arena_h, h->arena_h_cap, (size_t)m * 2 * nd))) return rc;
                launch_axpby_multi(h->arena_h, h->nufft_h[0], h->nufft_h[1], alpha0, dalpha, j0, m, 2 * nd, h->stream);
                h->launches++;
                gh = h->arena_h;
            }
        }
        REQUIRE(h, !r.xka || gh, SWRT_ERR_STATE, "flow has no H plane (needed by this scheme)");
        fill_nufft_args(h, g, a);
        a.hgrid = gh;
        a.gstride = td ? nd / 2 : 0; a.hstride = td ? 2 * nd : 0;
        a.x = h->x; a.y = h->y; a.k = h->k; a.l = h->l; a.a = h->a;
        a.f = h->p.f; a.C0 = C0; a.dt = dt; a.nsteps = m;
        return SWRT_OK;
    }
    if (mode == SWRT_MODE_LAGRANGE6) {
        LagArgs& a = r.la;
        REQUIRE(h, !r.xka || h->grid_npl == 7, SWRT_ERR_STATE, "step_packet_xka needs the H grid");
        const bool exact_two = (scheme == SWRT_SCHEME_LEAPFROG) && !h->preblend_grid;
        if (!td) {
            if ((rc = lag_frames(h, alpha_first, exact_two, a))) return rc;
        } else if (exact_two) {
            REQUIRE(h, h->grid[0] && h->grid[1], SWRT_ERR_STATE, "both flow slots must be set");
            a.grid = h->grid[0]; a.grid2 = h->grid[1]; a.alpha = alpha0; a.dalpha = dalpha; a.j0 = j0;
        } else {
            REQUIRE(h, h->grid[0] && h->grid[1], SWRT_ERR_STATE, "both flow slots must be set");
            const size_t nd = (size_t)h->p.nx * h->p.nx * h->grid_npl;
            if ((rc = ensure_arena(h, h->arena, h->arena_cap, (size_t)m * nd))) return rc;
            launch_axpby_multi(h->arena, h->grid[0], h->grid[1], alpha0, dalpha, j0, m, nd, h->stream);
            h->launches++;
            a.grid = h->arena; a.grid2 = nullptr; a.gstride = nd;
        }
        fill_lag_args(h, a);
        a.x = h->x; a.y = h->y; a.k = h->k; a.l = h->l; a.a = h->a;
        a.f = h->p.f; a.gH = h->p.gH; a.C0 = C0; a.dt = dt; a.nsteps = m;
        return SWRT_OK;
    }
    if (mode == SWRT_MODE_SPECTRAL && !h->unfused_rk4) {
        // fused step_packet / step_packet_xka: stage stack A = (u,v[,H]), big stack B = six / psi-moment / seven planes
        SpecRk4Args& a = r.ra;
        r.mt = 1;
        const bool psi = !r.xka && use_psi(h, td ? 0.5 : alpha_first);
        const int subA = r.xka ? SUB_UVH : SUB_UV, subB = r.xka ? SUB_SEVEN : (psi ? SUB_PSI3 : SUB_SIX);
        if (!td) {
            if ((rc = active_stack(h, subA, alpha_first, 1, &a.stackA, &a.gA)) || (rc = active_stack(h, subB, alpha_first, 1, &a.stackB, &a.gB))) return rc;
            a.nstack = 1;
        } else {
            for (int sub : {subA, subB})
                for (int slot = 0; slot < 2; slot++)
                    if ((rc = ensure_stack(h, sub, slot, 1))) return rc;
            Stack& sa_ = h->stacks[subA];
            Stack& sb_ = h->stacks[subB];
            a.gA = sa_.g; a.gB = sb_.g;
            if ((rc = ensure_arena(h, h->arena, h->arena_cap, (size_t)m * sa_.g.total_doubles)) ||
                (rc = ensure_arena(h, h->arena_h, h->arena_h_cap, (size_t)m * sb_.g.total_doubles))) return rc;
            launch_axpby_multi(h->arena, sa_.slot[0], sa_.slot[1], alpha0, dalpha, j0, m, sa_.g.total_doubles, h->stream);
            launch_axpby_multi(h->arena_h, sb_.slot[0], sb_.slot[1], alpha0, dalpha, j0, m, sb_.g.total_doubles, h->stream);
            h->launches += 2;
            a.stackA = h->arena; a.stackB = h->arena_h; a.nstack = m;
        }
        a.psiB = psi;
        a.kappa = 2.0 * M_PI / h->p.L; a.u_mean0 = h->u_mean[0]; a.u_mean1 = h->slot_set[1] ? h->u_mean[1] : 0.0;
        a.alpha0 = alpha0; a.dalpha = dalpha; a.j0 = j0;
        a.x = h->x; a.y = h->y; a.k = h->k; a.l = h->l; a.a = h->a;
        fill_spec_geom(h, a);
        a.f = h->p.f; a.C0 = C0; a.dt = dt; a.nsteps = m;
        return SWRT_OK;
    }
    // the composed route (tuning flag 4, SPECTRAL and NUFFT): evaluation + glue launches per step
    r.composed = true;
    return ensure_scratch(h, h->n);
}

// step_packet / step_packet_xka composed point-wise from separate evaluation and stage launches (whole ensemble)
static int run_composed_rk4(swrt_handle* h, const RunOps& r) {
    int rc;
    const double C0 = sqrt(h->p.gH);
    for (int j = 0; j < r.m; j++) {
        const double alpha = r.alpha0 + (r.j0 + j) * r.dalpha;
        Rk4Args q{};
        q.n = h->n; q.x = h->x; q.y = h->y; q.k = h->k; q.l = h->l; q.a = h->a;
        q.xs = h->xs; q.ys = h->ys; q.ax = h->ax; q.ay = h->ay;
        q.dt = r.dt; q.f = h->p.f; q.C0 = C0; q.xka = r.xka;
        for (int stage = 0; stage < 4; stage++) {
            const double* px = stage == 0 ? h->x : h->xs;
            const double* py = stage == 0 ? h->y : h->ys;
            if (r.xka) {
                double* outs[3] = {h->e[0], h->e[1], h->e[6]};
                if ((rc = eval_dev(h, SUB_UVH, alpha, h->n, px, py, outs))) return rc;
            } else if (stage == 0) {
                // u,v and the gradients at the OLD position in one six-plane pass (step_packet.m:58-61)
                // (later stages only overwrite e[0], e[1], so e[2..5] keep the old-position gradients)
                if ((rc = eval_dev(h, SUB_SIX, alpha, h->n, px, py, h->e))) return rc;
            } else {
                double* outs[2] = {h->e[0], h->e[1]};
                if ((rc = eval_dev(h, SUB_UV, alpha, h->n, px, py, outs))) return rc;
            }
            h->last_nlaunch++;
            q.stage = stage; q.u = h->e[0]; q.v = h->e[1]; q.H = h->e[6];
            launch_rk4_stage(q, h->stream);
            h->launches++;
        }
        if (r.xka) {
            if ((rc = eval_dev(h, SUB_SEVEN, alpha, h->n, h->xs, h->ys, h->e))) return rc;
            h->last_nlaunch++;
        }
        q.u = h->e[0]; q.v = h->e[1]; q.H = h->e[6];
        q.ux = h->e[2]; q.uy = h->e[3]; q.vx = h->e[4]; q.vy = h->e[5];
        launch_rk4_final(q, h->stream);
        h->launches++;
    }
    return SWRT_OK;
}

// anchored leapfrog over packets [lo, lo+cnt), per step j: first half drift + anchor key, counting sort by anchor, K1 (the
// expansion blocks of every anchor cell from step j's stack), K2 (expansion, stage 2, kick, second half drift).
// No host synchronisation.
static int run_anchored(swrt_handle* h, const RunOps& r, int64_t lo, int64_t cnt) {
    const int mlog = anchor_log2_cells(h->p.nx);
    const int nanc = 1 << mlog;                        // anchor cells of 2^-mlog turns
    SpecArgs a = r.sa;
    a.n = cnt; a.x += lo; a.y += lo; a.k += lo; a.l += lo;
    a.anc_block = (size_t)a.g.npass * 2 * a.g.NT * 32;
    a.anc_h = std::ldexp(1.0, 1 - mlog);               // cell width in reduced_turns' t (one period = 2)
    a.zscale = M_PI * (double)a.g.kmax;
    int rc;
    if ((rc = ensure_anchor(h, cnt, nanc, (size_t)nanc * a.anc_block))) return rc;
    a.anc_cnt = h->anc_cnt; a.anc_off = h->anc_off;
    a.anc_perm = h->anc_perm; a.hexp = h->anc_hexp;
    const double inv_h = std::ldexp(1.0, mlog - 1);
    for (int j = 0; j < r.m; j++) {
        CU(h, cudaMemsetAsync(h->anc_cnt, 0, (size_t)nanc * sizeof(unsigned long long), h->stream));
        launch_anchor_key(a.x, a.y, a.k, a.l, cnt, a.dx, a.nxd, a.inv_nx, a.f2, a.gH, a.dt, inv_h, nanc, h->anc_cnt, h->anc_key,
                          h->anc_rank, h->stream);
        launch_anchor_scan(h->anc_cnt, h->anc_off, nanc, h->stream);
        launch_anchor_scatter(h->anc_key, h->anc_rank, h->anc_off, h->anc_perm, cnt, h->stream);
        CU(h, cudaGetLastError());
        const size_t so = a.nstack > 1 ? (size_t)j * a.g.total_doubles : 0;
        SpecArgs k1 = a;
        k1.stack = r.sa.stack + so;
        CU(h, launch_anchor_transform(k1, nanc, h->num_sms, h->stream));
        a.ev = j;
        CU(h, launch_anchored_step(a, nanc, h->stream));
        h->launches += 5;
    }
    h->last_nlaunch++;       // one packet-stepping run, as one dense-kernel launch is; swrt_launch_count has every kernel
    return SWRT_OK;
}

// the run's kernel over packets [lo, lo+cnt) on the handle's stream
static int launch_run(swrt_handle* h, const RunOps& r, int64_t lo, int64_t cnt) {
    if (cnt <= 0) return SWRT_OK;
    if (r.composed) {
        REQUIRE(h, lo == 0 && cnt == h->n, SWRT_ERR_STATE, "the composed RK4 route runs on the whole ensemble");
        return run_composed_rk4(h, r);
    }
    const int mode = h->p.mode;
    if (r.anchored) return run_anchored(h, r, lo, cnt);
    if (mode == SWRT_MODE_SPECTRAL && r.scheme != SWRT_SCHEME_LEAPFROG) {
        SpecRk4Args a = r.ra;
        a.n = cnt; a.x += lo; a.y += lo; a.k += lo; a.l += lo; a.a += lo;
        {   // joint geometry decides where the twiddle table lives; the global form needs the handle's scratch
            SpecRk4Args probe = a; size_t smem = 0;
            spectral_rk4_geometry(probe, &smem);
            if (probe.atab == 2) {
                PackGeom tg = a.gA; tg.atab = 2; tg.ksteps = probe.tab_ksteps;
                int rc2 = ensure_twid(h, tg, &a.twid);
                if (rc2) return rc2;
            }
        }
        CU(h, launch_spectral_rk4(a, r.xka, h->num_sms, h->stream));
    } else if (mode == SWRT_MODE_SPECTRAL) {
        SpecArgs a = r.sa;
        a.n = cnt; a.x += lo; a.y += lo; a.k += lo; a.l += lo;
#ifdef SWRT_TRACE
        static unsigned long long* tr = nullptr;
        if (!tr) { cudaMalloc(&tr, 8 * 640 * 8); }
        cudaMemset(tr, 0, 8 * 640 * 8);
        a.trace = tr;
#endif
        { int rc2 = ensure_twid(h, a.g, &a.twid); if (rc2) return rc2; }
        CU(h, launch_spectral(a, SPEC_LEAPFROG, r.mt, h->num_sms, h->stream));
#ifdef SWRT_TRACE
        {
            std::vector<unsigned long long> hb(8 * 640);
            cudaStreamSynchronize(h->stream);
            cudaMemcpy(hb.data(), tr, hb.size() * 8, cudaMemcpyDeviceToHost);
            FILE* fp = fopen("gpurun_out/trace.txt", "w");
            if (fp) {
                for (int w = 0; w < 8; w++) { for (int i = 0; i < 640; i++) fprintf(fp, "%llu ", hb[w * 640 + i]); fprintf(fp, "\n"); }
                fclose(fp);
            }
        }
#endif
    } else if (mode == SWRT_MODE_NUFFT) {
        NufftArgs a = r.na;
        a.n = cnt; a.x += lo; a.y += lo; a.k += lo; a.l += lo; a.a += lo;
        if (r.scheme == SWRT_SCHEME_LEAPFROG) CU(h, launch_nufft_leapfrog(a, h->stream));
        else CU(h, launch_nufft_rk4(a, r.xka, h->stream));
    } else {
        LagArgs a = r.la;
        a.n = cnt; a.x += lo; a.y += lo; a.k += lo; a.l += lo; a.a += lo;
        if (r.scheme == SWRT_SCHEME_LEAPFROG) CU(h, launch_lagrange_leapfrog(a, h->stream));
        else CU(h, launch_lagrange_rk4(a, r.xka, h->stream));
    }
    h->launches++; h->last_nlaunch++;
    return SWRT_OK;
}

static int check_step_args(swrt_handle* h, int scheme, double dt, int nsteps) {
    REQUIRE(h, nsteps >= 0, SWRT_ERR_ARG, "negative step count");
    REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "no flow has been set");
    REQUIRE(h, std::isfinite(dt), SWRT_ERR_ARG, "dt is not finite");
    REQUIRE(h, scheme == SWRT_SCHEME_LEAPFROG || scheme == SWRT_SCHEME_RK4_PACKET || scheme == SWRT_SCHEME_RK4_XKA, SWRT_ERR_ARG,
            "unknown scheme %d", scheme);
    return SWRT_OK;
}

static int step_impl(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha, bool sync) {
    if (!h) return SWRT_ERR_ARG;
    CU(h, cudaSetDevice(h->p.device));
    int rc = check_step_args(h, scheme, dt, nsteps);
    if (rc) return rc;
    if (nsteps == 0 || h->n == 0) return SWRT_OK;
    h->last_nlaunch = 0;
    const bool td = (dalpha != 0.0);
    for (int j0 = 0; j0 < nsteps;) {
        const int m = td ? (nsteps - j0 < kMaxFusedBlend ? nsteps - j0 : kMaxFusedBlend) : nsteps - j0;
        RunOps r;
        if ((rc = prepare_run(h, scheme, dt, alpha0, dalpha, j0, m, r))) return rc;
        if (j0 == 0) CU(h, cudaEventRecord(h->ev0, h->stream));        // after the blends: ev0..ev1 brackets the packet kernels
        if ((rc = launch_run(h, r, 0, h->n))) return rc;
        j0 += m;
    }
    CU(h, cudaEventRecord(h->ev1, h->stream));
    h->timing_valid = true;
    if (sync) CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

#include "swrt_staging.inc"   // host staging: pinned ring + helper threads (HostPipe)

extern "C" {

// ---- packets ----------------------------------------------------------------------------------
int swrt_packets_alloc_dev(swrt_handle* h, int64_t n) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, n >= 0, SWRT_ERR_ARG, "negative packet count");
    if (h->ngpu > 1) {
        const int64_t G = h->ngpu;
        for (int64_t i = 0; i <= G; i++) h->off[i] = (i * n) / G;
        h->n = n;
        for (int64_t i = 0; i < G; i++) { int rc = swrt_packets_alloc_dev(h->shard[i], h->off[i + 1] - h->off[i]); if (rc) return up(h, h->shard[i], rc); }
        return SWRT_OK;
    }
    CU(h, cudaSetDevice(h->p.device));
    int rc = ensure_packets(h, n);
    if (rc) return rc;
    launch_fill(h->a, 1.0, n, h->stream);
    return SWRT_OK;
}

int swrt_packets_dev(swrt_handle* h, double** x, double** y, double** k, double** l, double** a) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, h->ngpu <= 1, SWRT_ERR_STATE, "a multi-device handle has one set of buffers per shard (swrt_shard_info)");
    if (x) *x = h->x; if (y) *y = h->y; if (k) *k = h->k; if (l) *l = h->l; if (a) *a = h->a;
    return SWRT_OK;
}

int swrt_set_packets(swrt_handle* h, int64_t n, const double* x, const double* y, const double* k, const double* l,
                     const double* a) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_set_packets(h, n, x, y, k, l, a));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, n >= 0, SWRT_ERR_ARG, "negative packet count");
    REQUIRE(h, n == 0 || (x && y && k && l), SWRT_ERR_ARG, "null packet array");
    if (n == 0) { h->n = 0; h->bs_ready = false; return SWRT_OK; }
    CU(h, cudaStreamSynchronize(h->stream));          // earlier work on the packet buffers has finished
    const double* in[5] = {x, y, k, l, a};
    HostPipe p; RunOps r;
    int rc = pipe_setup(h, p, r, n, true, in, nullptr, 0, 0.0, 0, 0.0, 0.0);
    for (int c = 0; rc == SWRT_OK && c < p.nchunk; c++) rc = p.step(c);
    if (rc == SWRT_OK) rc = p.finish();
    return rc;
}

int swrt_get_packets(swrt_handle* h, double* x, double* y, double* k, double* l, double* a) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_get_packets(h, x, y, k, l, a));
    CU(h, cudaSetDevice(h->p.device));
    if (h->n == 0) return SWRT_OK;
    double* out[5] = {x, y, k, l, a};
    HostPipe p; RunOps r;
    int rc = pipe_setup(h, p, r, h->n, false, nullptr, out, 0, 0.0, 0, 0.0, 0.0);
    for (int c = 0; rc == SWRT_OK && c < p.nchunk; c++) rc = p.step(c);
    if (rc == SWRT_OK) rc = p.finish();
    return rc;
}

int64_t swrt_num_packets(const swrt_handle* h) { return h ? h->n : 0; }

int swrt_num_devices(const swrt_handle* h) { return h ? h->ngpu : 0; }

int swrt_shard_info(const swrt_handle* h, int i, int* device, int64_t* lo, int64_t* n) {
    if (!h || i < 0 || i >= h->ngpu) return SWRT_ERR_ARG;
    if (device) *device = h->p.device + i;
    if (lo) *lo = h->ngpu > 1 ? h->off[i] : 0;
    if (n) *n = h->ngpu > 1 ? h->off[i + 1] - h->off[i] : h->n;
    return SWRT_OK;
}

int swrt_step(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha) {
    if (h && h->ngpu > 1) return grp_step(h, scheme, dt, nsteps, alpha0, dalpha, true);
    return step_impl(h, scheme, dt, nsteps, alpha0, dalpha, true);
}
// same launches, no host wait: the caller overlaps host work (diagnostics of the previous interval, the next
// frame's upload) with the kernel; swrt_synchronize / any blocking call completes it
int swrt_step_async(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha) {
    if (h && h->ngpu > 1) return grp_step(h, scheme, dt, nsteps, alpha0, dalpha, false);
    return step_impl(h, scheme, dt, nsteps, alpha0, dalpha, false);
}

// host arrays in -> nsteps -> host arrays out (the call shape of ode_symplectic.m:1-4 / step_packet.m:1), pipelined over
// packet chunks: see HostPipe
int swrt_step_host(swrt_handle* h, int scheme, double dt, int nsteps, double alpha0, double dalpha, int64_t n, const double* x,
                   const double* y, const double* k, const double* l, const double* a, double* xo, double* yo, double* ko,
                   double* lo, double* ao) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, n >= 0, SWRT_ERR_ARG, "negative packet count");
    REQUIRE(h, n == 0 || (x && y && k && l), SWRT_ERR_ARG, "null packet array");
    const double* in[5] = {x, y, k, l, a};
    double* out[5] = {xo, yo, ko, lo, ao};
    if (h->ngpu > 1) {
        for (swrt_handle* c : h->shard) { int rc = check_step_args(c, scheme, dt, nsteps); if (rc) return up(h, c, rc); }
        return grp_step_host(h, scheme, dt, nsteps, alpha0, dalpha, n, in, out);
    }
    CU(h, cudaSetDevice(h->p.device));
    int rc = check_step_args(h, scheme, dt, nsteps);
    if (rc) return rc;
    if (n == 0) { h->n = 0; h->bs_ready = false; return SWRT_OK; }
    CU(h, cudaStreamSynchronize(h->stream));
    HostPipe p; RunOps r;
    rc = pipe_setup(h, p, r, n, true, in, out, scheme, dt, nsteps, alpha0, dalpha);
    for (int c = 0; rc == SWRT_OK && c < p.nchunk; c++) rc = p.step(c);
    if (rc == SWRT_OK) rc = p.finish();
    h->timing_valid = false;
    return rc;
}

// ---- diagnostics ------------------------------------------------------------------------------
static int compute_omega(swrt_handle* h, double alpha, bool need_abs) {
    int rc = ensure_scratch(h, h->n);
    if (rc) return rc;
    if (need_abs) {
        REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "absolute frequency needs a flow");
        double* outs[2] = {h->e[0], h->e[1]};
        if (h->p.mode != SWRT_MODE_LAGRANGE6) {
            if ((rc = eval_dev(h, SUB_UV, alpha, h->n, h->x, h->y, outs))) return rc;
        } else if ((rc = eval_dev(h, SUB_SIX, alpha, h->n, h->x, h->y, h->e))) return rc;
    }
    launch_omega(h->n, h->k, h->l, h->e[0], h->e[1], h->p.f, h->p.gH, h->om, need_abs ? h->Om : nullptr, h->stream);
    h->launches++;
    return SWRT_OK;
}

int swrt_omega(swrt_handle* h, double alpha, double* omega, double* Omega_abs) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_each_slice(h, [&](swrt_handle* c, int64_t lo) { return swrt_omega(c, alpha, at(omega, lo), at(Omega_abs, lo)); }));
    CU(h, cudaSetDevice(h->p.device));
    int rc = compute_omega(h, alpha, Omega_abs != nullptr);
    if (rc) return rc;
    if ((rc = d2h(h, omega, h->om, h->n)) || (rc = d2h(h, Omega_abs, h->Om, h->n))) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

// histogram into the handle's device counts buffer (left on the device, stream synchronised)
static int hist_to_device(swrt_handle* h, int kind, double alpha, const double* edges, int nedges) {
    REQUIRE(h, edges && nedges >= 2 && nedges <= 4096, SWRT_ERR_ARG, "bad edges (2 <= nedges <= 4096)");
    REQUIRE(h, kind == SWRT_HIST_INTRINSIC || kind == SWRT_HIST_ABSOLUTE, SWRT_ERR_ARG, "bad histogram kind");
    for (int i = 1; i < nedges; i++) REQUIRE(h, edges[i] >= edges[i - 1], SWRT_ERR_ARG, "edges must be non-decreasing");
    int rc = compute_omega(h, alpha, kind == SWRT_HIST_ABSOLUTE);
    if (rc) return rc;
    if (nedges > h->edges_cap) { dfree(h->edges_dev); CU(h, cudaMalloc(&h->edges_dev, (size_t)nedges * 8)); h->edges_cap = nedges; h->edges_host.clear(); }
    if (nedges - 1 > h->counts_cap) { dfree(h->counts_dev); CU(h, cudaMalloc(&h->counts_dev, (size_t)(nedges - 1) * 8)); h->counts_cap = nedges - 1; }
    if ((int)h->edges_host.size() != nedges || memcmp(h->edges_host.data(), edges, (size_t)nedges * 8) != 0) {
        h->edges_host.assign(edges, edges + nedges);          // upload only when the edges changed
        CU(h, cudaMemcpyAsync(h->edges_dev, h->edges_host.data(), (size_t)nedges * 8, cudaMemcpyHostToDevice, h->stream));
    }
    CU(h, cudaMemsetAsync(h->counts_dev, 0, (size_t)(nedges - 1) * 8, h->stream));
    launch_hist(h->n, kind == SWRT_HIST_ABSOLUTE ? h->Om : h->om, h->edges_dev, nedges, h->counts_dev, h->stream);
    h->launches++;
    return SWRT_OK;
}

int swrt_hist_omega(swrt_handle* h, int kind, double alpha, const double* edges, int nedges, uint64_t* counts,
                    int accumulate) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_hist_omega(h, kind, alpha, edges, nedges, counts, accumulate));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, counts, SWRT_ERR_ARG, "null counts");
    int rc = hist_to_device(h, kind, alpha, edges, nedges);
    if (rc) return rc;
    std::vector<uint64_t> tmp(nedges - 1);
    CU(h, cudaMemcpyAsync(tmp.data(), h->counts_dev, (size_t)(nedges - 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaGetLastError());
    for (int i = 0; i < nedges - 1; i++) counts[i] = accumulate ? counts[i] + tmp[i] : tmp[i];
    return SWRT_OK;
}

int swrt_hist_omega_dev(swrt_handle* h, int kind, double alpha, const double* edges, int nedges, uint64_t** counts_dev) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_hist_omega_dev(h, kind, alpha, edges, nedges, counts_dev, true));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, counts_dev, SWRT_ERR_ARG, "null counts_dev");
    int rc = hist_to_device(h, kind, alpha, edges, nedges);
    if (rc) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    *counts_dev = reinterpret_cast<uint64_t*>(h->counts_dev);
    return SWRT_OK;
}

// non-blocking form: the histogram kernel is queued behind whatever is on the handle's stream and an event is
// recorded after it; swrt_hist_omega_wait blocks on that event only (not on work queued afterwards)
int swrt_hist_omega_launch(swrt_handle* h, int kind, double alpha, const double* edges, int nedges, uint64_t** counts_dev) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_hist_omega_dev(h, kind, alpha, edges, nedges, counts_dev, false));    // histograms + all-reduce queued, no host wait
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, counts_dev, SWRT_ERR_ARG, "null counts_dev");
    int rc = hist_to_device(h, kind, alpha, edges, nedges);
    if (rc) return rc;
    if (!h->hist_ev) CU(h, cudaEventCreateWithFlags(&h->hist_ev, cudaEventDisableTiming));
    CU(h, cudaEventRecord(h->hist_ev, h->stream));
    *counts_dev = reinterpret_cast<uint64_t*>(h->counts_dev);
    return SWRT_OK;
}
int swrt_hist_omega_wait(swrt_handle* h) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) { int rc = swrt_hist_omega_wait(h->shard[0]); return up(h, h->shard[0], rc); }
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, h->hist_ev, SWRT_ERR_STATE, "swrt_hist_omega_launch has not been called");
    CU(h, cudaEventSynchronize(h->hist_ev));
    return SWRT_OK;
}

int swrt_ideal_omega_hist(swrt_handle* h, double alpha, int64_t npts, const double* x, const double* y, const double* kvx,
                          const double* kvy, int nangles, double omega0, const double* edges, int nedges, uint64_t* counts) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_ideal_omega_hist(h, alpha, npts, x, y, kvx, kvy, nangles, omega0, edges, nedges, counts));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, npts >= 0 && x && y && kvx && kvy && edges && counts, SWRT_ERR_ARG, "null argument");
    REQUIRE(h, nangles >= 1 && nangles <= 1024 && nedges >= 2 && nedges <= 4096, SWRT_ERR_ARG, "bad nangles / nedges");
    // the kernel keeps the edges, the bin counters and the wavevectors in (default-limit) dynamic shared memory
    REQUIRE(h, (size_t)nedges * 12 + (size_t)nangles * 16 <= 48 * 1024, SWRT_ERR_ARG,
            "nedges*12 + nangles*16 = %zu bytes exceeds the 48 KB shared-memory budget of the kernel", (size_t)nedges * 12 + (size_t)nangles * 16);
    REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "no flow has been set");
    for (int i = 1; i < nedges; i++) REQUIRE(h, edges[i] >= edges[i - 1], SWRT_ERR_ARG, "edges must be non-decreasing");
    int rc = ensure_scratch(h, npts > h->n ? npts : h->n);
    if (rc) return rc;
    if ((rc = h2d(h, h->xs, x, npts)) || (rc = h2d(h, h->ys, y, npts))) return rc;
    // the same six-plane evaluation swrt_eval_at performs, so U is bit-identical to what the caller can read back
    rc = eval_dev(h, SUB_SIX, alpha, npts, h->xs, h->ys, h->e);
    if (rc) return rc;
    double *dk = nullptr, *de = nullptr; unsigned long long* dc = nullptr;
    if (cudaMalloc(&dk, (size_t)2 * nangles * 8) || cudaMalloc(&de, (size_t)nedges * 8) || cudaMalloc(&dc, (size_t)(nedges - 1) * 8)) {
        cudaFree(dk); cudaFree(de); cudaFree(dc);
        return fail(h, SWRT_ERR_ALLOC, "cudaMalloc failed");
    }
    cudaMemcpyAsync(dk, kvx, (size_t)nangles * 8, cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(dk + nangles, kvy, (size_t)nangles * 8, cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(de, edges, (size_t)nedges * 8, cudaMemcpyHostToDevice, h->stream);
    cudaMemsetAsync(dc, 0, (size_t)(nedges - 1) * 8, h->stream);
    launch_ideal_hist(npts, h->e[0], h->e[1], dk, dk + nangles, nangles, omega0, de, nedges, dc, h->stream);
    h->launches++;
    cudaError_t e = cudaMemcpyAsync(counts, dc, (size_t)(nedges - 1) * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    cudaFree(dk); cudaFree(de); cudaFree(dc);
    if (e != cudaSuccess) return fail(h, SWRT_ERR_CUDA, "swrt_ideal_omega_hist: %s", cudaGetErrorString(e));
    return SWRT_OK;
}

// ---- swrt_packet_quantity / swrt_hist2 ----
static bool valid_quantity(int q) { return q >= SWRT_Q_XMOD && q <= SWRT_Q_OMEGA_ABS; }
// the packet arrays of the quantities qa, qb; om / Om computed first when one of them is a frequency (om also when
// omega_too: the energy weight)
static int quantity_inputs(swrt_handle* h, int qa, int qb, double alpha, PktQ& p, bool omega_too = false) {
    const bool need_abs = qa == SWRT_Q_OMEGA_ABS || qb == SWRT_Q_OMEGA_ABS;
    if (need_abs || omega_too || qa == SWRT_Q_OMEGA || qb == SWRT_Q_OMEGA) {
        int rc = compute_omega(h, alpha, need_abs);
        if (rc) return rc;
    }
    p = PktQ{h->x, h->y, h->k, h->l, h->om, h->Om, h->p.L};
    return SWRT_OK;
}

int swrt_packet_quantity(swrt_handle* h, int q, double alpha, double* out) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, valid_quantity(q), SWRT_ERR_ARG, "unknown packet quantity %d", q);
    REQUIRE(h, out, SWRT_ERR_ARG, "null out");
    GROUP(h, grp_each_slice(h, [&](swrt_handle* c, int64_t lo) { return swrt_packet_quantity(c, q, alpha, out + lo); }));
    CU(h, cudaSetDevice(h->p.device));
    int rc = ensure_scratch(h, h->n);
    if (rc) return rc;
    PktQ p;
    if ((rc = quantity_inputs(h, q, q, alpha, p))) return rc;
    launch_packet_quantity(h->n, q, p, h->xs, h->stream);
    h->launches++;
    if ((rc = d2h(h, out, h->xs, h->n))) return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaGetLastError());
    return SWRT_OK;
}

static int hist2_args(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye) {
    REQUIRE(h, valid_quantity(qx) && valid_quantity(qy), SWRT_ERR_ARG, "unknown packet quantity (%d, %d)", qx, qy);
    REQUIRE(h, xedges && yedges, SWRT_ERR_ARG, "null edges");
    REQUIRE(h, nxe >= 2 && nxe <= 4096 && nye >= 2 && nye <= 4096, SWRT_ERR_ARG, "bad edges (2 <= nxe, nye <= 4096): %d, %d", nxe, nye);
    for (int a = 0; a < 2; a++) {
        const double* e = a ? yedges : xedges;
        for (int i = 0, ne = a ? nye : nxe; i < ne; i++) {
            REQUIRE(h, std::isfinite(e[i]), SWRT_ERR_ARG, "%s edge %d is not finite", a ? "y" : "x", i);
            REQUIRE(h, i == 0 || e[i] >= e[i - 1], SWRT_ERR_ARG, "%s edges must be non-decreasing (edge %d)", a ? "y" : "x", i);
        }
    }
    return SWRT_OK;
}
// h2_edges_dev holding xedges then yedges, and room for the u64 counts in h2_counts_dev (queued, no host wait)
static int hist2_buffers(swrt_handle* h, const double* xedges, int nxe, const double* yedges, int nye) {
    const int ne = nxe + nye;
    const int64_t nb = (int64_t)(nxe - 1) * (nye - 1);
    if (ne > h->h2_edges_cap) {
        dfree(h->h2_edges_dev); h->h2_edges_cap = 0; h->h2_edges_host.clear();
        CU(h, cudaMalloc(&h->h2_edges_dev, (size_t)ne * 8));
        h->h2_edges_cap = ne;
    }
    if (nb > h->h2_counts_cap) {
        dfree(h->h2_counts_dev); h->h2_counts_cap = 0;
        CU(h, cudaMalloc(&h->h2_counts_dev, (size_t)nb * 8));
        h->h2_counts_cap = nb;
    }
    if (h->h2_nxe != nxe || (int)h->h2_edges_host.size() != ne || memcmp(h->h2_edges_host.data(), xedges, (size_t)nxe * 8) != 0 ||
        memcmp(h->h2_edges_host.data() + nxe, yedges, (size_t)nye * 8) != 0) {
        h->h2_edges_host.assign(xedges, xedges + nxe);            // upload only when the edges changed
        h->h2_edges_host.insert(h->h2_edges_host.end(), yedges, yedges + nye);
        h->h2_nxe = nxe;
        CU(h, cudaMemcpyAsync(h->h2_edges_dev, h->h2_edges_host.data(), (size_t)ne * 8, cudaMemcpyHostToDevice, h->stream));
    }
    return SWRT_OK;
}
// the histogram into h2_counts_dev (queued, no host wait); the arguments have been checked
static int hist2_to_device(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye,
                           double alpha) {
    int rc;
    PktQ p;
    if ((rc = quantity_inputs(h, qx, qy, alpha, p))) return rc;
    if ((rc = hist2_buffers(h, xedges, nxe, yedges, nye))) return rc;
    const int64_t nb = (int64_t)(nxe - 1) * (nye - 1);
    CU(h, cudaMemsetAsync(h->h2_counts_dev, 0, (size_t)nb * 8, h->stream));
    CU(h, launch_hist2(h->n, qx, qy, p, h->h2_edges_dev, nxe, nye, h->h2_counts_dev, h->stream));
    h->launches++;
    return SWRT_OK;
}

int swrt_hist2(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye, double alpha,
               uint64_t* counts, int accumulate) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, counts, SWRT_ERR_ARG, "null counts");
    int rc = hist2_args(h, qx, xedges, nxe, qy, yedges, nye);
    if (rc) return rc;
    GROUP(h, grp_hist2(h, qx, xedges, nxe, qy, yedges, nye, alpha, counts, accumulate));
    CU(h, cudaSetDevice(h->p.device));
    if ((rc = hist2_to_device(h, qx, xedges, nxe, qy, yedges, nye, alpha))) return rc;
    const size_t nb = (size_t)(nxe - 1) * (nye - 1);
    std::vector<uint64_t> tmp(nb);
    CU(h, cudaMemcpyAsync(tmp.data(), h->h2_counts_dev, nb * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaGetLastError());
    for (size_t i = 0; i < nb; i++) counts[i] = accumulate ? counts[i] + tmp[i] : tmp[i];
    return SWRT_OK;
}

// ---- swrt_weight_scale / swrt_hist2_sums ----
static int weight_args(swrt_handle* h, const int32_t* w, int nw, WeightKinds& wk) {
    REQUIRE(h, w, SWRT_ERR_ARG, "null weight kinds");
    REQUIRE(h, nw >= 1 && nw <= SWRT_MAX_WEIGHTS, SWRT_ERR_ARG, "nw = %d outside 1..%d", nw, SWRT_MAX_WEIGHTS);
    wk = WeightKinds{nw, {0, 0, 0, 0}};
    for (int v = 0; v < nw; v++) {
        REQUIRE(h, w[v] >= SWRT_W_ACTION && w[v] <= SWRT_W_PSEUDO_L, SWRT_ERR_ARG, "unknown weight kind %d", (int)w[v]);
        wk.kind[v] = w[v];
    }
    return SWRT_OK;
}
static bool needs_omega(const WeightKinds& wk) {
    for (int v = 0; v < wk.n; v++) if (wk.kind[v] == SWRT_W_ENERGY) return true;
    return false;
}
static int32_t unbias_exp(int be) { return be ? be - kScaleBias : 0; }
// the inputs of the quantities qx, qy and of the weights, then each kind's biased scale exponent into ws_exp_dev: the
// caller's (given) or computed by the scale kernel (queued, no host wait)
static int weight_scale_to_device(swrt_handle* h, int qx, int qy, double alpha, const WeightKinds& wk, const int32_t* given) {
    PktQ p;
    int rc = quantity_inputs(h, qx, qy, alpha, p, needs_omega(wk));
    if (rc) return rc;
    if (!h->ws_exp_dev) CU(h, cudaMalloc(&h->ws_exp_dev, SWRT_MAX_WEIGHTS * sizeof(int)));
    if (given) {
        for (int v = 0; v < wk.n; v++) h->ws_exp_host[v] = given[v] + kScaleBias;
        CU(h, cudaMemcpyAsync(h->ws_exp_dev, h->ws_exp_host, wk.n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        return SWRT_OK;
    }
    CU(h, cudaMemsetAsync(h->ws_exp_dev, 0, SWRT_MAX_WEIGHTS * sizeof(int), h->stream));
    launch_weight_scale(h->n, wk, p, h->a, h->ws_exp_dev, h->stream);
    h->launches++;
    return SWRT_OK;
}
// the digit counters (and, want_counts, the u64 counts) into h2s_acc_dev / h2_counts_dev after weight_scale_to_device
// (queued, no host wait)
static int hist2_sums_to_device(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye,
                                const WeightKinds& wk, bool want_counts) {
    int rc = hist2_buffers(h, xedges, nxe, yedges, nye);
    if (rc) return rc;
    const int64_t nb = (int64_t)(nxe - 1) * (nye - 1), nacc = 4 * nb * wk.n;
    if (nacc > h->h2s_acc_cap) {
        dfree(h->h2s_acc_dev); h->h2s_acc_cap = 0;
        CU(h, cudaMalloc(&h->h2s_acc_dev, (size_t)nacc * 8));
        h->h2s_acc_cap = nacc;
    }
    CU(h, cudaMemsetAsync(h->h2s_acc_dev, 0, (size_t)nacc * 8, h->stream));
    if (want_counts) CU(h, cudaMemsetAsync(h->h2_counts_dev, 0, (size_t)nb * 8, h->stream));
    const PktQ p{h->x, h->y, h->k, h->l, h->om, h->Om, h->p.L};          // om / Om filled by weight_scale_to_device
    CU(h, launch_hist2_sums(h->n, qx, qy, p, h->a, wk, h->ws_exp_dev, h->h2_edges_dev, nxe, nye, h->h2s_acc_dev,
                            want_counts ? h->h2_counts_dev : nullptr, h->stream));
    h->launches++;
    return SWRT_OK;
}
// c's exponents, accumulators and counts to the host, then the sums (err: the handle that reports a failure)
static int hist2_sums_finish(swrt_handle* err, swrt_handle* c, int64_t nb, int nw, double* sums, uint64_t* counts, int64_t* acc) {
    std::vector<int64_t> tmp;
    if (!acc) { tmp.resize((size_t)(4 * nb * nw)); acc = tmp.data(); }
    int be[SWRT_MAX_WEIGHTS] = {};
    CU(err, cudaSetDevice(c->p.device));
    CU(err, cudaMemcpyAsync(be, c->ws_exp_dev, nw * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(err, cudaMemcpyAsync(acc, c->h2s_acc_dev, (size_t)(4 * nb * nw) * 8, cudaMemcpyDeviceToHost, c->stream));
    if (counts) CU(err, cudaMemcpyAsync(counts, c->h2_counts_dev, (size_t)nb * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(err, cudaStreamSynchronize(c->stream));
    CU(err, cudaGetLastError());
    int32_t E[SWRT_MAX_WEIGHTS];
    for (int v = 0; v < nw; v++) E[v] = unbias_exp(be[v]);
    return sums ? swrt_fixed_sums_to_double(acc, nb, nw, E, sums) : SWRT_OK;
}

int swrt_weight_scale(swrt_handle* h, const int32_t* w, int nw, double alpha, int32_t* scale_exp) {
    if (!h) return SWRT_ERR_ARG;
    WeightKinds wk;
    int rc = weight_args(h, w, nw, wk);
    if (rc) return rc;
    REQUIRE(h, scale_exp, SWRT_ERR_ARG, "null scale_exp");
    GROUP(h, grp_weight_scale(h, wk, alpha, scale_exp));
    CU(h, cudaSetDevice(h->p.device));
    if ((rc = weight_scale_to_device(h, SWRT_Q_K, SWRT_Q_K, alpha, wk, nullptr))) return rc;
    CU(h, cudaMemcpyAsync(h->ws_exp_host, h->ws_exp_dev, nw * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaGetLastError());
    for (int v = 0; v < nw; v++) scale_exp[v] = unbias_exp(h->ws_exp_host[v]);
    return SWRT_OK;
}

int swrt_hist2_sums(swrt_handle* h, int qx, const double* xedges, int nxe, int qy, const double* yedges, int nye,
                    double alpha, const int32_t* w, int nw, const int32_t* scale_exp, double* sums, uint64_t* counts,
                    int64_t* acc) {
    if (!h) return SWRT_ERR_ARG;
    int rc = hist2_args(h, qx, xedges, nxe, qy, yedges, nye);
    if (rc) return rc;
    WeightKinds wk;
    if ((rc = weight_args(h, w, nw, wk))) return rc;
    for (int v = 0; scale_exp && v < nw; v++)
        REQUIRE(h, scale_exp[v] >= -1073 && scale_exp[v] <= 1024, SWRT_ERR_ARG, "scale_exp[%d] = %d outside -1073..1024", v, (int)scale_exp[v]);
    REQUIRE(h, h->n <= INT32_MAX, SWRT_ERR_ARG, "%lld packets: the digit counters hold at most 2^31 - 1", (long long)h->n);
    GROUP(h, grp_hist2_sums(h, qx, xedges, nxe, qy, yedges, nye, alpha, wk, scale_exp, sums, counts, acc));
    CU(h, cudaSetDevice(h->p.device));
    if ((rc = weight_scale_to_device(h, qx, qy, alpha, wk, scale_exp))) return rc;
    if ((rc = hist2_sums_to_device(h, qx, xedges, nxe, qy, yedges, nye, wk, counts != nullptr))) return rc;
    return hist2_sums_finish(h, h, (int64_t)(nxe - 1) * (nye - 1), nw, sums, counts, acc);
}

// one bin: (c[0] + c[1] 2^32 + c[2] 2^64) 2^(E-95) rounded once to the nearest double, NaN when c[3] != 0
static double fixed_to_double(const int64_t* c, int32_t E) {
    if (c[3] != 0) return NAN;
    using u128 = unsigned __int128;
    using i128 = __int128;
    const i128 t = (i128)c[1] * ((i128)1 << 32) + c[0];                // |t| < 2^96
    const i128 hi = (i128)c[2] + (t >> 64);                               // S = hi 2^64 + lo, 0 <= lo < 2^64
    const uint64_t lo = (uint64_t)t;
    const bool neg = hi < 0;
    u128 m = ((u128)hi << 64) | lo;                                       // S mod 2^128 ...
    if (neg) m = -m;                                                      // ... and |S| < 2^128
    if (m == 0) return 0.0;
    const uint64_t mh = (uint64_t)(m >> 64);
    const int bits = mh ? 128 - __builtin_clzll(mh) : 64 - __builtin_clzll((uint64_t)m);
    const int64_t e0 = (int64_t)E - 95;                                   // the weight of m's bit 0
    const int64_t lead = e0 + bits - 1;
    if (lead > 1023) return neg ? -HUGE_VAL : HUGE_VAL;
    const int64_t qexp = std::max<int64_t>(lead - 52, -1074);            // the quantum of the result's binade
    uint64_t r;
    int64_t rexp = qexp;
    if (qexp <= e0) {
        r = (uint64_t)m;                                                  // at most 53 bits: exact
        rexp = e0;
    } else {
        const int64_t sh = qexp - e0;
        if (sh > 128) {
            r = 0;                                                        // m < 2^128 <= half a quantum
        } else {
            r = sh == 128 ? 0 : (uint64_t)(m >> sh);
            const u128 rem = sh == 128 ? m : m & (((u128)1 << sh) - 1), half = (u128)1 << (sh - 1);
            if (rem > half || (rem == half && (r & 1))) r++;              // ties to even
        }
    }
    const double v = std::ldexp((double)r, (int)rexp);                   // r <= 2^53: exact, or +inf past DBL_MAX
    return neg ? -v : v;
}

int swrt_fixed_sums_to_double(const int64_t* acc, int64_t nbins, int nw, const int32_t* scale_exp, double* sums) {
    if (nbins < 0 || nw < 0 || (nbins > 0 && nw > 0 && (!acc || !scale_exp || !sums))) return SWRT_ERR_ARG;
    for (int v = 0; v < nw; v++)
        for (int64_t b = 0; b < nbins; b++) sums[v * nbins + b] = fixed_to_double(acc + 4 * (v * nbins + b), scale_exp[v]);
    return SWRT_OK;
}

// the eight diagnostics of this handle's packets into h->diag_dev (queued, no host wait)
static int diag_launch(swrt_handle* h, double alpha) {
    int rc = compute_omega(h, alpha, h->slot_set[0]);
    if (rc) return rc;
    launch_diag(h->n, h->x, h->y, h->k, h->l, h->a, h->om, h->slot_set[0] ? h->Om : h->om, h->diag_dev, h->stream);
    h->launches += 2;
    return SWRT_OK;
}

int swrt_diag(swrt_handle* h, double alpha, double out[8]) {
    if (!h || !out) return SWRT_ERR_ARG;
    GROUP(h, grp_diag(h, alpha, out));
    CU(h, cudaSetDevice(h->p.device));
    int rc = diag_launch(h, alpha);
    if (rc) return rc;
    CU(h, cudaMemcpyAsync(out, h->diag_dev, 8 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

// ---- ode23 building blocks --------------------------------------------------------------------
static int bs23_setup(swrt_handle* h, Bs23Args& a) {
    int rc = ensure_scratch(h, h->n);
    if (rc) return rc;
    if (h->n > h->bs_cap) {
        for (auto& p : h->bs_yt) dfree(p);
        for (auto& row : h->bs_f) for (auto& p : row) dfree(p);
        h->bs_cap = 0; h->bs_ready = false;
        size_t b = (size_t)h->n * sizeof(double);
        for (auto& p : h->bs_yt) CU(h, cudaMalloc(&p, b));
        for (auto& row : h->bs_f) for (auto& p : row) CU(h, cudaMalloc(&p, b));
        h->bs_cap = h->n; h->bs_ready = false;
    }
    if (!h->bs_norm_dev) CU(h, cudaMalloc(&h->bs_norm_dev, sizeof(unsigned long long)));
    a.n = h->n;
    a.y[0] = h->x; a.y[1] = h->y; a.y[2] = h->k; a.y[3] = h->l;
    for (int c = 0; c < 4; c++) { a.yt[c] = h->bs_yt[c]; for (int j = 0; j < 4; j++) a.f[j][c] = h->bs_f[j][c]; }
    return SWRT_OK;
}
// f_j = odefun(alpha, state) with state = (sx, sy, sk, sl) device arrays
static int bs23_rhs(swrt_handle* h, double alpha, double* const st[4], double* const fj[4]) {
    int rc = eval_dev(h, SUB_SIX, alpha, h->n, st[0], st[1], h->e);
    if (rc) return rc;
    launch_rhs(Ode23ValView{}, 0, h->n, st[2], st[3], h->e, nullptr, h->p.f, h->p.gH, rhs_cgfac(h), fj, h->stream);
    h->launches++;
    return SWRT_OK;
}
static int bs23_read_norm(swrt_handle* h, double* out) {
    unsigned long long bits = 0;
    CU(h, cudaMemcpyAsync(&bits, h->bs_norm_dev, sizeof bits, cudaMemcpyDeviceToHost, h->stream));
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaGetLastError());
    memcpy(out, &bits, sizeof bits);
    return SWRT_OK;
}

// f1 and the scale norm of this handle's packets into bs_norm_dev (queued, no host wait)
static int bs23_begin_launch(swrt_handle* h, double alpha, double threshold) {
    REQUIRE(h, h->slot_set[0], SWRT_ERR_STATE, "no flow has been set");
    Bs23Args a{};
    int rc = bs23_setup(h, a);
    if (rc) return rc;
    double* f1[4] = {a.f[0][0], a.f[0][1], a.f[0][2], a.f[0][3]};
    if ((rc = bs23_rhs(h, alpha, a.y, f1))) return rc;
    CU(h, cudaMemsetAsync(h->bs_norm_dev, 0, sizeof(unsigned long long), h->stream));
    launch_bs23_norm<1>(a, Ode23ValView{}, threshold, h->bs_norm_dev, h->stream);
    h->launches++;
    h->bs_ready = true;
    return SWRT_OK;
}

int swrt_bs23_begin(swrt_handle* h, double alpha, double threshold, double* rh_norm) {
    if (!h || !rh_norm) return SWRT_ERR_ARG;
    GROUP(h, grp_bs23_begin(h, alpha, threshold, rh_norm));
    CU(h, cudaSetDevice(h->p.device));
    int rc = bs23_begin_launch(h, alpha, threshold);
    if (rc) return rc;
    return bs23_read_norm(h, rh_norm);
}

static int bs23_attempt_launch(swrt_handle* h, double hstep, const double alpha[3], double threshold) {
    REQUIRE(h, h->bs_ready && h->bs_cap >= h->n, SWRT_ERR_STATE, "swrt_bs23_begin has not been called");
    Bs23Args a{};
    int rc = bs23_setup(h, a);
    if (rc) return rc;
    double* f2[4] = {a.f[1][0], a.f[1][1], a.f[1][2], a.f[1][3]};
    double* f3[4] = {a.f[2][0], a.f[2][1], a.f[2][2], a.f[2][3]};
    double* f4[4] = {a.f[3][0], a.f[3][1], a.f[3][2], a.f[3][3]};
    const Ode23ValView v{hstep, {alpha[0], alpha[1], alpha[2]}};
    launch_bs23_stage(a, v, 0, h->stream);
    if ((rc = bs23_rhs(h, alpha[0], a.yt, f2))) return rc;
    launch_bs23_stage(a, v, 1, h->stream);
    if ((rc = bs23_rhs(h, alpha[1], a.yt, f3))) return rc;
    launch_bs23_stage(a, v, 2, h->stream);   // ynew
    if ((rc = bs23_rhs(h, alpha[2], a.yt, f4))) return rc;
    CU(h, cudaMemsetAsync(h->bs_norm_dev, 0, sizeof(unsigned long long), h->stream));
    launch_bs23_norm<0>(a, v, threshold, h->bs_norm_dev, h->stream);
    h->launches += 4;
    return SWRT_OK;
}

int swrt_bs23_attempt(swrt_handle* h, double hstep, const double alpha[3], double threshold, double* err_norm) {
    if (!h || !alpha || !err_norm) return SWRT_ERR_ARG;
    GROUP(h, grp_bs23_attempt(h, hstep, alpha, threshold, err_norm));
    CU(h, cudaSetDevice(h->p.device));
    int rc = bs23_attempt_launch(h, hstep, alpha, threshold);
    if (rc) return rc;
    return bs23_read_norm(h, err_norm);
}

int swrt_bs23_accept(swrt_handle* h) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) {
        for (swrt_handle* c : h->shard) { int rc = swrt_bs23_accept(c); if (rc) return up(h, c, rc); }
        return SWRT_OK;
    }
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, h->bs_ready, SWRT_ERR_STATE, "swrt_bs23_begin has not been called");
    Bs23Args a{};
    int rc = bs23_setup(h, a);
    if (rc) return rc;
    launch_bs23_accept(a, Ode23ValView{}, h->stream);
    h->launches++;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

int swrt_bs23_interp(swrt_handle* h, double hstep, double s, double* x, double* y, double* k, double* l) {
    if (!h || !x || !y || !k || !l) return SWRT_ERR_ARG;
    GROUP(h, grp_each_slice(h, [&](swrt_handle* c, int64_t lo) { return swrt_bs23_interp(c, hstep, s, x + lo, y + lo, k + lo, l + lo); }));
    CU(h, cudaSetDevice(h->p.device));
    REQUIRE(h, h->bs_ready && h->bs_cap >= h->n, SWRT_ERR_STATE, "swrt_bs23_attempt has not been called");
    Bs23Args a{};
    int rc = bs23_setup(h, a);
    if (rc) return rc;
    if (s == 1.0) {   // an output time that coincides with the step end gets ynew itself (ode23: tspan(next) == tnew)
        if ((rc = d2h(h, x, a.yt[0], h->n)) || (rc = d2h(h, y, a.yt[1], h->n)) || (rc = d2h(h, k, a.yt[2], h->n)) ||
            (rc = d2h(h, l, a.yt[3], h->n)))
            return rc;
        CU(h, cudaStreamSynchronize(h->stream));
        return SWRT_OK;
    }
    // BI = [1 -4/3 5/9; 0 1 -2/3; 0 4/3 -8/9; 0 -1 1] (ntrp23), columns weighted by s, s^2, s^3
    const double s2 = s * s, s3 = s2 * s;
    const double w[4] = {hstep * (s - 4.0 / 3.0 * s2 + 5.0 / 9.0 * s3), hstep * (s2 - 2.0 / 3.0 * s3),
                         hstep * (4.0 / 3.0 * s2 - 8.0 / 9.0 * s3), hstep * (-s2 + s3)};
    double* out[4] = {h->xs, h->ys, h->ax, h->ay};
    launch_bs23_interp(a, w, out, h->stream);
    h->launches++;
    if ((rc = d2h(h, x, h->xs, h->n)) || (rc = d2h(h, y, h->ys, h->n)) || (rc = d2h(h, k, h->ax, h->n)) ||
        (rc = d2h(h, l, h->ay, h->n)))
        return rc;
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

// ---- spectral <-> grid kit ----------------------------------------------------------------------
int swrt_g2k(int device, const double* fg, int nx, double* fk_re, double* fk_im) {
    if (!fg || !fk_re || !fk_im || nx < 4 || (nx & 1)) return fail(nullptr, SWRT_ERR_ARG, "swrt_g2k: bad argument");
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail(nullptr, SWRT_ERR_CUDA, "swrt_g2k: no CUDA device"); }
    FftWork w; std::string err;
    int rc = w.init(nx, 0, err);
    if (rc) return fail(nullptr, rc, "swrt_g2k: %s", err.c_str());
    size_t n = (size_t)nx * nx, nh = (size_t)(nx - 1) * (nx / 2);
    double* dg = nullptr; double2* dh = nullptr;
    if (cudaMalloc(&dg, n * 8) || cudaMalloc(&dh, nh * 16)) { cudaFree(dg); return fail(nullptr, SWRT_ERR_ALLOC, "swrt_g2k: cudaMalloc failed"); }
    cudaMemcpy(dg, fg, n * 8, cudaMemcpyHostToDevice);
    rc = g2k_dev(w, dg, dh, 0, err);
    std::vector<double2> hh(nh);
    if (!rc && cudaMemcpy(hh.data(), dh, nh * 16, cudaMemcpyDeviceToHost) != cudaSuccess) rc = SWRT_ERR_CUDA;
    cudaFree(dg); cudaFree(dh);
    if (rc) return fail(nullptr, rc, "swrt_g2k: %s", err.c_str());
    for (size_t i = 0; i < nh; i++) { fk_re[i] = hh[i].x; fk_im[i] = hh[i].y; }
    return SWRT_OK;
}

int swrt_k2g(int device, const double* fk_re, const double* fk_im, int nx, double* fg) {
    if (!fg || !fk_re || !fk_im || nx < 4 || (nx & 1)) return fail(nullptr, SWRT_ERR_ARG, "swrt_k2g: bad argument");
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail(nullptr, SWRT_ERR_CUDA, "swrt_k2g: no CUDA device"); }
    FftWork w; std::string err;
    int rc = w.init(nx, 0, err);
    if (rc) return fail(nullptr, rc, "swrt_k2g: %s", err.c_str());
    size_t n = (size_t)nx * nx, nh = (size_t)(nx - 1) * (nx / 2);
    std::vector<double2> hh(nh);
    for (size_t i = 0; i < nh; i++) hh[i] = make_double2(fk_re[i], fk_im[i]);
    double* dg = nullptr; double2* dh = nullptr;
    if (cudaMalloc(&dg, n * 8) || cudaMalloc(&dh, nh * 16)) { cudaFree(dg); return fail(nullptr, SWRT_ERR_ALLOC, "swrt_k2g: cudaMalloc failed"); }
    cudaMemcpy(dh, hh.data(), nh * 16, cudaMemcpyHostToDevice);
    rc = k2g_dev(w, dh, dg, 0, err);
    if (!rc && cudaMemcpy(fg, dg, n * 8, cudaMemcpyDeviceToHost) != cudaSuccess) rc = SWRT_ERR_CUDA;
    cudaFree(dg); cudaFree(dh);
    if (rc) return fail(nullptr, rc, "swrt_k2g: %s", err.c_str());
    return SWRT_OK;
}

}  // extern "C"

#include "swrt_qg.inc"        // one- and two-layer QG frame producers

extern "C" {

// ---- instrumentation --------------------------------------------------------------------------
int64_t swrt_launch_count(swrt_handle* h, int reset) {
    if (!h) return 0;
    if (h->ngpu > 1) { int64_t v = 0; for (swrt_handle* c : h->shard) v += swrt_launch_count(c, reset); return v; }
    int64_t v = h->launches;
    if (reset) h->launches = 0;
    return v;
}

double swrt_last_kernel_ms(swrt_handle* h, int* nlaunch) {
    if (!h) return -1.0;
    if (h->ngpu > 1) {      // the slowest device's kernel time
        double worst = -1.0;
        for (swrt_handle* c : h->shard) {
            if (c->n == 0) continue;
            const double ms = swrt_last_kernel_ms(c, nlaunch);
            if (ms < 0) return -1.0;
            if (ms > worst) worst = ms;
        }
        return worst;
    }
    if (!h->timing_valid) return -1.0;
    cudaSetDevice(h->p.device);
    if (cudaEventSynchronize(h->ev1) != cudaSuccess) return -1.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return -1.0;
    if (nlaunch) *nlaunch = h->last_nlaunch;
    return (double)ms;
}

double swrt_work_per_eval(const swrt_handle* h, int nplanes) {
    if (!h) return 0.0;
    if (h->ngpu > 1) return swrt_work_per_eval(h->shard[0], nplanes);
    if (h->p.mode == SWRT_MODE_SPECTRAL) {
        if (nplanes == 3 && anchor_log2_cells(h->p.nx) > 0 && h->n > 0) {
            // the anchored leapfrog on a psi-hat flow: K2 runs 2 k-steps (R = 8 orders) per packet over the padded columns,
            // K1 the fp64 flops of its transforms (every anchor cell, whatever the occupancy), spread over the packets
            const PackGeom g = make_geom(h->p.nx, 3, kSubsetIds[SUB_PSI3], 1, h->twiddle_pref);
            const double cols = (double)g.npass * g.NT * 8, k2_packet = 2.0 * kAnchorOrders * cols;
            return k2_packet + anchor_transform_flops(g) / (double)h->n;
        }
        // executed DMMA flops per packet per evaluation: (kx>=0 count) * (ky count) * planes * 8
        // flops per folded complex MAC ... = 2 * nplanes * nx^2 for the unpadded problem
        return 2.0 * nplanes * (double)h->p.nx * (double)h->p.nx;
    }
    // gathered bytes: w^2 = 324 nodes; 16-byte (u,v) nodes give all six planes, 32-byte (u,v,H,0) nodes the seven
    if (h->p.mode == SWRT_MODE_NUFFT) return (double)kNufftW * kNufftW * (nplanes >= 7 ? 32.0 : 16.0);
    return 36.0 * nplanes * 8.0;   // gathered bytes
}

int swrt_synchronize(swrt_handle* h) {
    if (!h) return SWRT_ERR_ARG;
    GROUP(h, grp_sync(h));
    CU(h, cudaSetDevice(h->p.device));
    CU(h, cudaStreamSynchronize(h->stream));
    return SWRT_OK;
}

int swrt_set_stream(swrt_handle* h, void* cuda_stream) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, h->ngpu <= 1, SWRT_ERR_STATE, "a multi-device handle runs one stream per device; a caller stream belongs to one");
    CU(h, cudaSetDevice(h->p.device));
    CU(h, cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return SWRT_OK;
}

int swrt_timer_start(swrt_handle* h) {
    if (!h) return SWRT_ERR_ARG;
    if (h->ngpu > 1) {
        for (swrt_handle* c : h->shard) { int rc = swrt_timer_start(c); if (rc) return up(h, c, rc); }
        return SWRT_OK;
    }
    CU(h, cudaSetDevice(h->p.device));
    CU(h, cudaEventRecord(h->tm0, h->stream));
    return SWRT_OK;
}

double swrt_timer_stop(swrt_handle* h) {
    if (!h) return -1.0;
    if (h->ngpu > 1) {      // device time of the slowest device
        double worst = -1.0;
        for (swrt_handle* c : h->shard) { const double ms = swrt_timer_stop(c); if (ms < 0) return -1.0; if (ms > worst) worst = ms; }
        return worst;
    }
    cudaSetDevice(h->p.device);
    float ms = 0.f;
    if (cudaEventRecord(h->tm1, h->stream) != cudaSuccess || cudaEventSynchronize(h->tm1) != cudaSuccess ||
        cudaEventElapsedTime(&ms, h->tm0, h->tm1) != cudaSuccess) {
        h->err = "swrt_timer_stop: event timing failed";
        return -1.0;
    }
    return (double)ms;
}

int swrt_set_tuning(swrt_handle* h, int mtiles, int flags) {
    if (!h) return SWRT_ERR_ARG;
    REQUIRE(h, mtiles >= 0 && mtiles <= 2, SWRT_ERR_ARG, "mtiles must be 0, 1 or 2");
    for (swrt_handle* c : h->shard) swrt_set_tuning(c, mtiles, flags);
    h->mtiles = mtiles;
    h->disable_psi = (flags & 1) != 0;
    h->preblend_grid = (flags & 2) != 0;
    h->unfused_rk4 = (flags & 4) != 0;
    h->twiddle_pref = (flags >> 3) & 3;
    return SWRT_OK;
}

int swrt_contracted_planes(const swrt_handle* h) {
    if (!h || h->p.mode != SWRT_MODE_SPECTRAL) return 0;
    if (h->ngpu > 1) return swrt_contracted_planes(h->shard[0]);
    return use_psi(h, h->slot_set[1] ? 0.5 : 0.0) ? 3 : 6;
}

int swrt_gather_probe(int device, int64_t table_bytes, int reps, double* gbytes_per_s) {
    if (!gbytes_per_s || table_bytes < (1 << 16) || (table_bytes & (table_bytes - 1)) || table_bytes > ((int64_t)1 << 31) || reps < 1)
        return fail(nullptr, SWRT_ERR_ARG, "swrt_gather_probe: bad argument (table_bytes must be a power of two in [64 KiB, 2 GiB])");
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail(nullptr, SWRT_ERR_CUDA, "swrt_gather_probe: no CUDA device"); }
    const double v = gather_probe((size_t)table_bytes, 64, reps, 0);
    if (v < 0) return fail(nullptr, SWRT_ERR_CUDA, "swrt_gather_probe: %s", cudaGetErrorString(cudaGetLastError()));
    *gbytes_per_s = v;
    return SWRT_OK;
}

int swrt_spectral_geometry(int nx, int nplanes, int mtiles, int64_t out[10]) {
    if (!out || nx < 4 || (nx & 1) || nplanes < 1 || nplanes > kMaxPlanes || mtiles < 1 || mtiles > 2)
        return fail(nullptr, SWRT_ERR_ARG, "swrt_spectral_geometry: bad argument");
    int ids[kMaxPlanes];
    for (int i = 0; i < kMaxPlanes; i++) ids[i] = i;
    const PackGeom g = make_geom(nx, nplanes, ids, mtiles);
    out[0] = g.NT; out[1] = g.npass; out[2] = g.ksteps; out[3] = g.kc; out[4] = g.nstages;
    out[5] = (int64_t)(g.chunk_doubles * 8); out[6] = g.atab;
    out[7] = g.atab == 1 ? (int64_t)g.ksteps * 32 * 8 * kConsumerWarps : 0;
    out[8] = (int64_t)spectral_smem_bytes(g);
    out[9] = (int64_t)(g.total_doubles * 8);
    return SWRT_OK;
}

}  // extern "C"

#include "swrt_group.inc"     // multi-device handles: sharding + in-library NCCL
#include "swrt_ode23.inc"     // swrt_ode23: a whole ode23 solve with the controller on the device
#include "swrt_ode23_packets.inc"   // swrt_ode23_packets: the same solve with one controller per packet
