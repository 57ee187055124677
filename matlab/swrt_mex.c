/* swrt_mex.c -- MEX gateway over libswrt.so (include/swrt.h) for MATLAB / GNU Octave.
 *
 *   [out...] = swrt_mex('command', args...)
 *
 * The gateway holds no logic: it unpacks mxArrays (column-major fp64), calls one C-ABI function and packs the result.
 * Engine / QG-producer handles travel as uint64 scalars (1-based slots of the tables below).  Errors are raised with
 * mexErrMsgIdAndTxt("swrt:...") only after the C call has returned (libswrt never throws); temporaries come from
 * mxCalloc, which MATLAB / Octave release when mexFunction returns or errors out.
 *
 * Complex storage: Octave's mkoctfile --mex and MATLAB's default (-R2017b) API keep separate real / imaginary arrays
 * (mxGetPr / mxGetPi), which is what the C ABI takes.  Built with MATLAB's interleaved API (mex -R2018a, which defines
 * MX_HAS_INTERLEAVED_COMPLEX = 1) the gateway de-interleaves / interleaves through temporaries (mxGetComplexDoubles).
 *
 * Build:   mkoctfile --mex swrt_mex.c -I../include -L../swraytracing_b200 -lswrt
 *          mex [-R2018a] swrt_mex.c -I../include -L../swraytracing_b200 -lswrt          (MATLAB)
 * Neither tool exists in the development image: the file is compiled against matlab/stub/mex.h and EXECUTED, command by
 * command, by tests/mex_harness (a small implementation of the mx / mex functions used here) in both storage layouts. */
#include <string.h>
#include "mex.h"
#include "swrt.h"

#ifndef MX_HAS_INTERLEAVED_COMPLEX
#define MX_HAS_INTERLEAVED_COMPLEX 0
#endif

#define MAXH 64
static swrt_handle* g_handles[MAXH];
static swrt_qg* g_qg[MAXH];
static swrt_qg2* g_qg2[MAXH];
static int g_locked = 0;

static void destroy_all(void) {
    for (int i = 0; i < MAXH; i++) {
        if (g_handles[i]) { swrt_destroy(g_handles[i]); g_handles[i] = NULL; }
        if (g_qg[i]) { swrt_qg_destroy(g_qg[i]); g_qg[i] = NULL; }
        if (g_qg2[i]) { swrt_qg2_destroy(g_qg2[i]); g_qg2[i] = NULL; }
    }
}
static void fail(swrt_handle* h, const char* what) { mexErrMsgIdAndTxt("swrt:call", "%s: %s", what, swrt_last_error(h)); }
static void need(int nrhs, int n, const char* usage) {
    if (nrhs < n) mexErrMsgIdAndTxt("swrt:usage", "usage: swrt_mex(%s)", usage);
}
static uint64_t id_of(const mxArray* a) { return mxIsDouble(a) ? (uint64_t)mxGetScalar(a) : *(uint64_t*)mxGetData(a); }
static swrt_handle* H(const mxArray* a) {
    uint64_t id = id_of(a);
    if (id < 1 || id > MAXH || !g_handles[id - 1]) mexErrMsgIdAndTxt("swrt:handle", "invalid handle");
    return g_handles[id - 1];
}
static mxArray* new_id(uint64_t id) {
    mxArray* o = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
    *(uint64_t*)mxGetData(o) = id;
    return o;
}
static double* vec(mxArray** out, size_t n) { *out = mxCreateDoubleMatrix(n, 1, mxREAL); return mxGetPr(*out); }
/* Output i of a multi-output command.  plhs[] has room for max(nlhs, 1) pointers only: a caller that asks for fewer outputs
   than the command can give ("[px, py, pk, pl] = swrt_mex('get_packets', eng)" in shims/ode_symplectic.m) must not have the
   rest written past the end of plhs -- those go to scratch memory that MATLAB / Octave release when mexFunction returns.
   (Found by executing the shims: tests/test_shims_executed.py.) */
static int g_nlhs = 0;
static double* outv(mxArray* plhs[], int i, size_t n) {
    if (i == 0 || i < g_nlhs) return vec(&plhs[i], n);
    return (double*)mxCalloc(n ? n : 1, sizeof(double));
}
static double* opt(const mxArray* prhs[], int nrhs, int i) { return (i < nrhs && !mxIsEmpty(prhs[i])) ? mxGetPr(prhs[i]) : NULL; }
static double sc(const mxArray* prhs[], int nrhs, int i, double dflt) { return i < nrhs ? mxGetScalar(prhs[i]) : dflt; }

/* separate real / imaginary views of a (possibly real) double array; a real input gets a zero imaginary part */
typedef struct { const double* re; const double* im; } cview;
static cview cin(const mxArray* a) {
    cview v;
    size_t n = mxGetNumberOfElements(a);
#if MX_HAS_INTERLEAVED_COMPLEX
    if (mxIsComplex(a)) {
        const mxComplexDouble* z = mxGetComplexDoubles(a);
        double* re = (double*)mxCalloc(n ? n : 1, sizeof(double));
        double* im = (double*)mxCalloc(n ? n : 1, sizeof(double));
        for (size_t i = 0; i < n; i++) { re[i] = z[i].real; im[i] = z[i].imag; }
        v.re = re; v.im = im;
        return v;
    }
    v.re = mxGetDoubles(a);
#else
    v.re = mxGetPr(a);
    if (mxIsComplex(a)) { v.im = mxGetPi(a); return v; }
#endif
    v.im = (const double*)mxCalloc(n ? n : 1, sizeof(double));
    return v;
}
/* a complex m x n output filled from separate re / im buffers */
static mxArray* cout_(size_t m, size_t n, const double* re, const double* im) {
    mxArray* o = mxCreateDoubleMatrix(m, n, mxCOMPLEX);
#if MX_HAS_INTERLEAVED_COMPLEX
    mxComplexDouble* z = mxGetComplexDoubles(o);
    for (size_t i = 0; i < m * n; i++) { z[i].real = re[i]; z[i].imag = im[i]; }
#else
    memcpy(mxGetPr(o), re, m * n * sizeof(double));
    memcpy(mxGetPi(o), im, m * n * sizeof(double));
#endif
    return o;
}
static int free_slot(void** table) {
    int s = 0;
    while (s < MAXH && table[s]) s++;
    if (s == MAXH) mexErrMsgIdAndTxt("swrt:handle", "too many handles");
    return s;
}

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    g_nlhs = nlhs;
    char cmd[48];
    if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], cmd, sizeof cmd)) mexErrMsgIdAndTxt("swrt:usage", "swrt_mex('command', ...)");
    if (!g_locked) { mexLock(); mexAtExit(destroy_all); g_locked = 1; }
    (void)nlhs;

    /* ---- handle-free commands ---- */
    if (!strcmp(cmd, "create")) {           /* h = ('create', nx, L, f, gH [, mode, device, bump, flags, ngpu]) */
        need(nrhs, 5, "'create', nx, L, f, gH [, mode, device, bump, flags, ngpu]");
        swrt_params p; memset(&p, 0, sizeof p);
        p.nx = (int)mxGetScalar(prhs[1]); p.L = mxGetScalar(prhs[2]); p.f = mxGetScalar(prhs[3]); p.gH = mxGetScalar(prhs[4]);
        p.mode = (int)sc(prhs, nrhs, 5, SWRT_MODE_SPECTRAL);
        p.device = (int)sc(prhs, nrhs, 6, 0);
        p.bump = sc(prhs, nrhs, 7, 1e-13);
        p.flags = (int)sc(prhs, nrhs, 8, 0);
        p.ngpu = (int)sc(prhs, nrhs, 9, 1);
        int slot = free_slot((void**)g_handles);
        if (swrt_create(&p, &g_handles[slot])) fail(NULL, "swrt_create");
        plhs[0] = new_id((uint64_t)slot + 1);
        return;
    }
    if (!strcmp(cmd, "device_count")) { plhs[0] = mxCreateDoubleScalar((double)swrt_device_count()); return; }
    if (!strcmp(cmd, "version")) { plhs[0] = mxCreateDoubleScalar((double)swrt_version()); return; }
    if (!strcmp(cmd, "interpolate")) {      /* FI = ('interpolate', x, y, F, dx, dy [, bump]) */
        need(nrhs, 6, "'interpolate', x, y, F, dx, dy [, bump]");
        size_t n = mxGetNumberOfElements(prhs[1]);
        if (mxGetNumberOfElements(prhs[2]) != n) mexErrMsgIdAndTxt("swrt:usage", "interpolate: x and y differ in size");
        plhs[0] = mxCreateDoubleMatrix(mxGetM(prhs[1]), mxGetN(prhs[1]), mxREAL);
        if (swrt_interpolate(0, mxGetPr(prhs[1]), mxGetPr(prhs[2]), (int64_t)n, mxGetPr(prhs[3]), (int)mxGetM(prhs[3]), (int)mxGetN(prhs[3]),
                             mxGetScalar(prhs[4]), mxGetScalar(prhs[5]), sc(prhs, nrhs, 6, 1e-13), mxGetPr(plhs[0])))
            fail(NULL, "swrt_interpolate");
        return;
    }
    if (!strcmp(cmd, "k2g")) {              /* fg = ('k2g', fk) */
        need(nrhs, 2, "'k2g', fk");
        int nx = (int)mxGetM(prhs[1]) + 1;
        cview z = cin(prhs[1]);
        plhs[0] = mxCreateDoubleMatrix(nx, nx, mxREAL);
        if (swrt_k2g(0, z.re, z.im, nx, mxGetPr(plhs[0]))) fail(NULL, "swrt_k2g");
        return;
    }
    if (!strcmp(cmd, "g2k")) {              /* fk = ('g2k', fg) */
        need(nrhs, 2, "'g2k', fg");
        int nx = (int)mxGetM(prhs[1]);
        size_t nh = (size_t)(nx - 1) * (nx / 2);
        double* re = (double*)mxCalloc(nh ? nh : 1, sizeof(double)); double* im = (double*)mxCalloc(nh ? nh : 1, sizeof(double));
        if (swrt_g2k(0, mxGetPr(prhs[1]), nx, re, im)) fail(NULL, "swrt_g2k");
        plhs[0] = cout_(nx - 1, nx / 2, re, im);
        return;
    }
    if (!strcmp(cmd, "qg_create")) {        /* q = ('qg_create', nx, L, K_d2, beta, r_drag, force, f, Cg, dt, qk [, device]) */
        need(nrhs, 11, "'qg_create', nx, L, K_d2, beta, r_drag, force_strength, f, Cg, dt, qk [, device]");
        cview z = cin(prhs[10]);
        int slot = free_slot((void**)g_qg);
        if (swrt_qg_create((int)sc(prhs, nrhs, 11, 0), (int)mxGetScalar(prhs[1]), mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                           mxGetScalar(prhs[5]), mxGetScalar(prhs[6]), mxGetScalar(prhs[7]), mxGetScalar(prhs[8]), mxGetScalar(prhs[9]), z.re, z.im,
                           &g_qg[slot])) fail(NULL, "swrt_qg_create");
        plhs[0] = new_id((uint64_t)slot + 1);
        return;
    }
    if (!strcmp(cmd, "qg2_create")) {       /* q = ('qg2_create', nx, L, K_d2, beta, shear, r, nu, alpha, q1k, q2k [, device]) */
        need(nrhs, 11, "'qg2_create', nx, L, K_d2, beta, shear_strength, r, nu, alpha, q1k, q2k [, device]");
        cview a = cin(prhs[9]), b = cin(prhs[10]);
        int slot = free_slot((void**)g_qg2);
        if (swrt_qg2_create((int)sc(prhs, nrhs, 11, 0), (int)mxGetScalar(prhs[1]), mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                            mxGetScalar(prhs[5]), mxGetScalar(prhs[6]), mxGetScalar(prhs[7]), mxGetScalar(prhs[8]), a.re, a.im, b.re, b.im,
                            &g_qg2[slot])) fail(NULL, "swrt_qg2_create");
        plhs[0] = new_id((uint64_t)slot + 1);
        return;
    }
    /* ---- QG frame producers (handle = producer id) ---- */
    if (!strncmp(cmd, "qg_", 3) || !strncmp(cmd, "qg2_", 4)) {
        need(nrhs, 2, "'qg*_...', q, ...");
        uint64_t id = id_of(prhs[1]);
        int two = !strncmp(cmd, "qg2_", 4);
        if (id < 1 || id > MAXH || (two ? (void*)g_qg2[id - 1] : (void*)g_qg[id - 1]) == NULL) mexErrMsgIdAndTxt("swrt:handle", "invalid QG handle");
        if (!two) {
            swrt_qg* q = g_qg[id - 1];
            if (!strcmp(cmd, "qg_step")) { if (swrt_qg_step(q, (int)sc(prhs, nrhs, 2, 1))) fail(NULL, cmd); }
            else if (!strcmp(cmd, "qg_destroy")) { swrt_qg_destroy(q); g_qg[id - 1] = NULL; }
            else if (!strcmp(cmd, "qg_get") || !strcmp(cmd, "qg_get_grid")) {      /* qk = ('qg_get', q, nx) ; qgrid = ('qg_get_grid', q, nx) */
                need(nrhs, 3, "'qg_get', q, nx");
                int nx = (int)mxGetScalar(prhs[2]);
                if (!strcmp(cmd, "qg_get")) {
                    size_t nh = (size_t)(nx - 1) * (nx / 2);
                    double* re = (double*)mxCalloc(nh, sizeof(double)); double* im = (double*)mxCalloc(nh, sizeof(double));
                    if (swrt_qg_get(q, re, im)) fail(NULL, cmd);
                    plhs[0] = cout_(nx - 1, nx / 2, re, im);
                } else {
                    plhs[0] = mxCreateDoubleMatrix(nx, nx, mxREAL);
                    if (swrt_qg_get_grid(q, mxGetPr(plhs[0]))) fail(NULL, cmd);
                }
            } else mexErrMsgIdAndTxt("swrt:usage", "unknown command '%s'", cmd);
        } else {
            swrt_qg2* q = g_qg2[id - 1];
            if (!strcmp(cmd, "qg2_step")) { need(nrhs, 3, "'qg2_step', q, dt"); if (swrt_qg2_step(q, mxGetScalar(prhs[2]))) fail(NULL, cmd); }
            else if (!strcmp(cmd, "qg2_max_speed")) { plhs[0] = mxCreateDoubleMatrix(1, 1, mxREAL); if (swrt_qg2_max_speed(q, mxGetPr(plhs[0]))) fail(NULL, cmd); }
            else if (!strcmp(cmd, "qg2_destroy")) { swrt_qg2_destroy(q); g_qg2[id - 1] = NULL; }
            else if (!strcmp(cmd, "qg2_get")) {                                    /* qk = ('qg2_get', q, layer, nx) */
                need(nrhs, 4, "'qg2_get', q, layer, nx");
                int nx = (int)mxGetScalar(prhs[3]);
                size_t nh = (size_t)(nx - 1) * (nx / 2);
                double* re = (double*)mxCalloc(nh, sizeof(double)); double* im = (double*)mxCalloc(nh, sizeof(double));
                if (swrt_qg2_get(q, (int)mxGetScalar(prhs[2]), re, im)) fail(NULL, cmd);
                plhs[0] = cout_(nx - 1, nx / 2, re, im);
            } else mexErrMsgIdAndTxt("swrt:usage", "unknown command '%s'", cmd);
        }
        return;
    }

    /* ---- engine commands ---- */
    if (nrhs < 2) mexErrMsgIdAndTxt("swrt:usage", "missing handle");
    swrt_handle* h = H(prhs[1]);
    size_t n = (size_t)swrt_num_packets(h);

    if (!strcmp(cmd, "destroy")) {
        swrt_destroy(h); g_handles[id_of(prhs[1]) - 1] = NULL;
    } else if (!strcmp(cmd, "num_packets")) {
        plhs[0] = mxCreateDoubleScalar((double)n);
    } else if (!strcmp(cmd, "num_devices")) {
        plhs[0] = mxCreateDoubleScalar((double)swrt_num_devices(h));
    } else if (!strcmp(cmd, "set_flow_spectral")) {   /* (h, slot, psik [, u_mean]) */
        need(nrhs, 4, "'set_flow_spectral', h, slot, psik [, u_mean]");
        cview z = cin(prhs[3]);
        if (swrt_set_flow_spectral(h, (int)mxGetScalar(prhs[2]), z.re, z.im, (int)mxGetM(prhs[3]), (int)mxGetN(prhs[3]), sc(prhs, nrhs, 4, 0.0))) fail(h, cmd);
    } else if (!strcmp(cmd, "set_flow_planes_spectral")) {   /* (h, slot, uk, vk, uxk, uyk, vxk, vyk [, Hk]) */
        need(nrhs, 9, "'set_flow_planes_spectral', h, slot, uk, vk, uxk, uyk, vxk, vyk [, Hk]");
        int np = (nrhs > 9 && !mxIsEmpty(prhs[9])) ? 7 : 6;
        const double* re[7]; const double* im[7];
        for (int c = 0; c < np; c++) { cview z = cin(prhs[3 + c]); re[c] = z.re; im[c] = z.im; }
        if (swrt_set_flow_planes_spectral(h, (int)mxGetScalar(prhs[2]), re, im, np, (int)mxGetM(prhs[3]), (int)mxGetN(prhs[3]))) fail(h, cmd);
    } else if (!strcmp(cmd, "set_flow_grid")) {       /* (h, slot, u, v, ux, uy, vx, vy [, H]) */
        need(nrhs, 9, "'set_flow_grid', h, slot, u, v, ux, uy, vx, vy [, H]");
        if (swrt_set_flow_grid(h, (int)mxGetScalar(prhs[2]), mxGetPr(prhs[3]), mxGetPr(prhs[4]), mxGetPr(prhs[5]), mxGetPr(prhs[6]), mxGetPr(prhs[7]),
                               mxGetPr(prhs[8]), opt(prhs, nrhs, 9), (int)mxGetM(prhs[3]))) fail(h, cmd);
    } else if (!strcmp(cmd, "set_flow_from_qg")) {    /* (h, slot, q [, u_mean]) */
        need(nrhs, 4, "'set_flow_from_qg', h, slot, q [, u_mean]");
        uint64_t id = id_of(prhs[3]);
        if (id < 1 || id > MAXH || !g_qg[id - 1]) mexErrMsgIdAndTxt("swrt:handle", "invalid QG handle");
        if (swrt_set_flow_from_qg(h, (int)mxGetScalar(prhs[2]), g_qg[id - 1], sc(prhs, nrhs, 4, 0.0))) fail(h, cmd);
    } else if (!strcmp(cmd, "set_flow_from_qg2")) {   /* (h, slot, q) */
        need(nrhs, 4, "'set_flow_from_qg2', h, slot, q");
        uint64_t id = id_of(prhs[3]);
        if (id < 1 || id > MAXH || !g_qg2[id - 1]) mexErrMsgIdAndTxt("swrt:handle", "invalid QG handle");
        if (swrt_set_flow_from_qg2(h, (int)mxGetScalar(prhs[2]), g_qg2[id - 1])) fail(h, cmd);
    } else if (!strcmp(cmd, "set_packets")) {         /* (h, x, y, k, l [, a]) */
        need(nrhs, 6, "'set_packets', h, x, y, k, l [, a]");
        size_t m = mxGetNumberOfElements(prhs[2]);
        for (int i = 3; i < 6; i++) if (mxGetNumberOfElements(prhs[i]) != m) mexErrMsgIdAndTxt("swrt:usage", "set_packets: arrays differ in size");
        if (swrt_set_packets(h, (int64_t)m, mxGetPr(prhs[2]), mxGetPr(prhs[3]), mxGetPr(prhs[4]), mxGetPr(prhs[5]), opt(prhs, nrhs, 6))) fail(h, cmd);
    } else if (!strcmp(cmd, "get_packets")) {         /* [x, y, k, l, a] = ... */
        double* o[5]; for (int i = 0; i < 5; i++) o[i] = outv(plhs, i, n);
        if (swrt_get_packets(h, o[0], o[1], o[2], o[3], o[4])) fail(h, cmd);
    } else if (!strcmp(cmd, "eval")) {                /* [U, V, Ux, Uy, Vx, Vy] = (h, alpha) */
        double* o[6]; for (int i = 0; i < 6; i++) o[i] = outv(plhs, i, n);
        if (swrt_eval(h, sc(prhs, nrhs, 2, 0.0), o[0], o[1], o[2], o[3], o[4], o[5])) fail(h, cmd);
    } else if (!strcmp(cmd, "eval_at")) {             /* [U, V, Ux, Uy, Vx, Vy] = (h, alpha, x, y) */
        need(nrhs, 5, "'eval_at', h, alpha, x, y");
        size_t m = mxGetNumberOfElements(prhs[3]); double* o[6]; for (int i = 0; i < 6; i++) o[i] = outv(plhs, i, m);
        if (mxGetNumberOfElements(prhs[4]) != m) mexErrMsgIdAndTxt("swrt:usage", "eval_at: x and y differ in size");
        if (swrt_eval_at(h, mxGetScalar(prhs[2]), (int64_t)m, mxGetPr(prhs[3]), mxGetPr(prhs[4]), o[0], o[1], o[2], o[3], o[4], o[5], NULL)) fail(h, cmd);
    } else if (!strcmp(cmd, "rhs")) {                 /* [dxdt, dydt, dkdt, dldt] = (h, alpha) */
        double* o[4]; for (int i = 0; i < 4; i++) o[i] = outv(plhs, i, n);
        if (swrt_rhs(h, sc(prhs, nrhs, 2, 0.0), o[0], o[1], o[2], o[3])) fail(h, cmd);
    } else if (!strcmp(cmd, "step")) {                /* (h, scheme, dt, nsteps [, alpha0, dalpha]) */
        need(nrhs, 5, "'step', h, scheme, dt, nsteps [, alpha0, dalpha]");
        if (swrt_step(h, (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[4]), sc(prhs, nrhs, 5, 0.0), sc(prhs, nrhs, 6, 0.0))) fail(h, cmd);
    } else if (!strcmp(cmd, "step_host")) {           /* [x, y, k, l, a] = (h, scheme, dt, nsteps, x, y, k, l [, a, alpha0, dalpha]) */
        need(nrhs, 9, "'step_host', h, scheme, dt, nsteps, x, y, k, l [, a, alpha0, dalpha]");
        size_t m = mxGetNumberOfElements(prhs[5]);
        for (int i = 6; i < 9; i++) if (mxGetNumberOfElements(prhs[i]) != m) mexErrMsgIdAndTxt("swrt:usage", "step_host: arrays differ in size");
        double* o[5]; for (int i = 0; i < 5; i++) o[i] = outv(plhs, i, m);
        if (swrt_step_host(h, (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), (int)mxGetScalar(prhs[4]), sc(prhs, nrhs, 10, 0.0), sc(prhs, nrhs, 11, 0.0),
                           (int64_t)m, mxGetPr(prhs[5]), mxGetPr(prhs[6]), mxGetPr(prhs[7]), mxGetPr(prhs[8]), opt(prhs, nrhs, 9), o[0], o[1], o[2], o[3], o[4]))
            fail(h, cmd);
    } else if (!strcmp(cmd, "bs23_begin")) {          /* rh = (h, alpha, threshold)          -- ode23 building blocks */
        need(nrhs, 4, "'bs23_begin', h, alpha, threshold");
        plhs[0] = mxCreateDoubleMatrix(1, 1, mxREAL);
        if (swrt_bs23_begin(h, mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), mxGetPr(plhs[0]))) fail(h, cmd);
    } else if (!strcmp(cmd, "bs23_attempt")) {        /* err = (h, hstep, [a2 a3 a4], threshold) */
        need(nrhs, 5, "'bs23_attempt', h, hstep, [a2 a3 a4], threshold");
        plhs[0] = mxCreateDoubleMatrix(1, 1, mxREAL);
        if (mxGetNumberOfElements(prhs[3]) != 3) mexErrMsgIdAndTxt("swrt:usage", "bs23_attempt: alpha must have 3 entries");
        if (swrt_bs23_attempt(h, mxGetScalar(prhs[2]), mxGetPr(prhs[3]), mxGetScalar(prhs[4]), mxGetPr(plhs[0]))) fail(h, cmd);
    } else if (!strcmp(cmd, "bs23_accept")) {         /* (h) */
        if (swrt_bs23_accept(h)) fail(h, cmd);
    } else if (!strcmp(cmd, "bs23_interp")) {         /* [x, y, k, l] = (h, hstep, s)        -- ntrp23 */
        need(nrhs, 4, "'bs23_interp', h, hstep, s");
        double* o[4]; for (int i = 0; i < 4; i++) o[i] = outv(plhs, i, n);
        if (swrt_bs23_interp(h, mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), o[0], o[1], o[2], o[3])) fail(h, cmd);
    } else if (!strcmp(cmd, "ode23")) {               /* [stats, Y] = (h, tspan, tmax, rtol, atol)  -- whole solve, controller on the device */
        need(nrhs, 6, "'ode23', h, tspan, tmax, rtol, atol");
        int nt = (int)mxGetNumberOfElements(prhs[2]);
        int64_t st[4];
        double* Y = NULL;
        if (nlhs > 1) { plhs[1] = mxCreateDoubleMatrix((size_t)n, nt > 2 ? (size_t)4 * nt : 0, mxREAL); if (nt > 2) Y = mxGetPr(plhs[1]); }
        /* Y is n x (4*numel(tspan)): reshape(Y, n, 4, []) gives the state [x y k l] of every packet at every tspan entry */
        if (swrt_ode23(h, mxGetPr(prhs[2]), nt, mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), mxGetScalar(prhs[5]), Y, st, NULL, 0)) fail(h, cmd);
        plhs[0] = mxCreateDoubleMatrix(1, 4, mxREAL);
        for (int i = 0; i < 4; i++) mxGetPr(plhs[0])[i] = (double)st[i];
    } else if (!strcmp(cmd, "ode23_packets")) {       /* [stats, Y, pstat, t_end] = (h, tspan, tmax, rtol, atol)  -- one controller per packet, tspan shared or one row each */
        need(nrhs, 6, "'ode23_packets', h, tspan, tmax, rtol, atol");
        /* tspan a vector: shared by every packet; an n x m matrix (m >= 2): row i is packet i's own tspan */
        size_t tm = mxGetM(prhs[2]), tn = mxGetN(prhs[2]);
        int per_row = tm > 1 && tn > 1;
        if (per_row && tm != (size_t)n)
            mexErrMsgIdAndTxt("swrt:usage", "ode23_packets: a tspan matrix must be n x m (one row per packet), got %d x %d", (int)tm, (int)tn);
        int nt = per_row ? (int)tn : (int)mxGetNumberOfElements(prhs[2]);
        int64_t st[5];
        double *Y = NULL, *t_end = NULL;
        if (nlhs > 1) { plhs[1] = mxCreateDoubleMatrix((size_t)n, nt > 2 ? (size_t)4 * nt : 0, mxREAL); if (nt > 2) Y = mxGetPr(plhs[1]); }
        /* pstat: n x 3 = accepted steps, rejected steps, status (0 reached tfinal, 1 stopped); t_end: n x 1 */
        int32_t* ps = nlhs > 2 ? (int32_t*)mxCalloc((size_t)3 * (n > 0 ? n : 1), sizeof(int32_t)) : NULL;
        if (nlhs > 3) t_end = outv(plhs, 3, n);
        if ((per_row ? swrt_ode23_packets_tspans : swrt_ode23_packets)(h, mxGetPr(prhs[2]), nt, mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                                                                      mxGetScalar(prhs[5]), Y, ps, t_end, st))
            fail(h, cmd);
        plhs[0] = mxCreateDoubleMatrix(1, 5, mxREAL);
        for (int i = 0; i < 5; i++) mxGetPr(plhs[0])[i] = (double)st[i];
        if (ps) {
            plhs[2] = mxCreateDoubleMatrix((size_t)n, 3, mxREAL);
            for (size_t i = 0; i < 3 * n; i++) mxGetPr(plhs[2])[i] = (double)ps[i];
            mxFree(ps);
        }
    } else if (!strcmp(cmd, "ode23_events") || !strcmp(cmd, "ode23_tspans_events")) {
        /* [stats, Y, pstat, t_end, te, ye, ie, ne] = (h, tspan, tmax, rtol, atol, ev, ev_cap).  'ode23_tspans_events': tspan
           is a vector shared by every packet, in either direction, or an n x m matrix (m >= 2) whose row i is packet i's
           own; the events then follow each packet's direction of integration */
        int spans = !strcmp(cmd, "ode23_tspans_events");
        need(nrhs, 8, spans ? "'ode23_tspans_events', h, tspan, tmax, rtol, atol, ev, ev_cap" : "'ode23_events', h, tspan, tmax, rtol, atol, ev, ev_cap");
        int nt = (int)mxGetNumberOfElements(prhs[2]);
        const double* tsp = mxGetPr(prhs[2]);
        double* rows = NULL;
        if (spans) {
            size_t tm = mxGetM(prhs[2]), tn = mxGetN(prhs[2]);
            if (tm > 1 && tn > 1) {
                if (tm != (size_t)n)
                    mexErrMsgIdAndTxt("swrt:usage", "ode23_tspans_events: a tspan matrix must be n x m (one row per packet), got %d x %d",
                                      (int)tm, (int)tn);
                nt = (int)tn;
            } else {                                   /* the shared vector as every packet's row */
                rows = (double*)mxCalloc(n * (size_t)nt > 0 ? n * (size_t)nt : 1, sizeof(double));
                for (int j = 0; j < nt; j++)
                    for (size_t i = 0; i < n; i++) rows[(size_t)j * n + i] = tsp[j];
                tsp = rows;
            }
        }
        /* ev: nev x 4, columns [kind level direction terminal] */
        int nev = (int)mxGetM(prhs[6]), cap = (int)mxGetScalar(prhs[7]);
        if (mxGetN(prhs[6]) != 4) mexErrMsgIdAndTxt("swrt:usage", "%s: ev must be nev x 4 = [kind level direction terminal]", cmd);
        if (nev < 1 || nev > SWRT_MAX_EVENTS) mexErrMsgIdAndTxt("swrt:usage", "%s: 1 to %d events", cmd, SWRT_MAX_EVENTS);
        const double* e = mxGetPr(prhs[6]);
        swrt_event ev[SWRT_MAX_EVENTS];
        for (int j = 0; j < nev; j++) {
            ev[j].kind = (int32_t)e[j]; ev[j].level = e[nev + j]; ev[j].direction = (int32_t)e[2 * nev + j];
            ev[j].terminal = (int32_t)e[3 * nev + j]; ev[j].reserved = 0;
        }
        size_t nc = cap > 0 ? (size_t)cap : 0;
        int64_t st[7];
        double *Y = NULL, *t_end = NULL;
        if (nlhs > 1) { plhs[1] = mxCreateDoubleMatrix((size_t)n, nt > 2 ? (size_t)4 * nt : 0, mxREAL); if (nt > 2) Y = mxGetPr(plhs[1]); }
        int32_t* ps = nlhs > 2 ? (int32_t*)mxCalloc((size_t)3 * (n > 0 ? n : 1), sizeof(int32_t)) : NULL;
        if (nlhs > 3) t_end = outv(plhs, 3, n);
        /* te, ie: n x ev_cap (record r of packet i in row i, column r); ye: n x 4*ev_cap (reshape(ye, n, 4, []) gives
           [x y k l] of every record); ne: n x 1 */
        double *te = NULL, *ye = NULL;
        int32_t *ie = NULL, *ne = NULL;
        if (nlhs > 4) { plhs[4] = mxCreateDoubleMatrix((size_t)n, nc, mxREAL); te = mxGetPr(plhs[4]); }
        if (nlhs > 5) { plhs[5] = mxCreateDoubleMatrix((size_t)n, 4 * nc, mxREAL); ye = mxGetPr(plhs[5]); }
        if (nlhs > 6) ie = (int32_t*)mxCalloc(n * nc > 0 ? n * nc : 1, sizeof(int32_t));
        if (nlhs > 7) ne = (int32_t*)mxCalloc(n > 0 ? n : 1, sizeof(int32_t));
        int rc = (spans ? swrt_ode23_packets_tspans_events : swrt_ode23_packets_events)(
            h, tsp, nt, mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), mxGetScalar(prhs[5]), ev, nev, cap, Y, ps, t_end, te, ye, ie, ne, st);
        if (rows) mxFree(rows);
        if (rc) fail(h, cmd);
        plhs[0] = mxCreateDoubleMatrix(1, 7, mxREAL);
        for (int i = 0; i < 7; i++) mxGetPr(plhs[0])[i] = (double)st[i];
        if (ps) {
            plhs[2] = mxCreateDoubleMatrix((size_t)n, 3, mxREAL);
            for (size_t i = 0; i < 3 * n; i++) mxGetPr(plhs[2])[i] = (double)ps[i];
            mxFree(ps);
        }
        if (ie) {
            plhs[6] = mxCreateDoubleMatrix((size_t)n, nc, mxREAL);
            for (size_t i = 0; i < n * nc; i++) mxGetPr(plhs[6])[i] = (double)ie[i];
            mxFree(ie);
        }
        if (ne) {
            plhs[7] = mxCreateDoubleMatrix((size_t)n, 1, mxREAL);
            for (size_t i = 0; i < n; i++) mxGetPr(plhs[7])[i] = (double)ne[i];
            mxFree(ne);
        }
    } else if (!strcmp(cmd, "hist_omega")) {          /* counts = (h, kind, alpha, edges) */
        need(nrhs, 5, "'hist_omega', h, kind, alpha, edges");
        int ne = (int)mxGetNumberOfElements(prhs[4]);
        if (ne < 2) mexErrMsgIdAndTxt("swrt:usage", "hist_omega: at least two edges");
        plhs[0] = mxCreateNumericMatrix(1, ne - 1, mxUINT64_CLASS, mxREAL);
        if (swrt_hist_omega(h, (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), mxGetPr(prhs[4]), ne, (uint64_t*)mxGetData(plhs[0]), 0)) fail(h, cmd);
    } else if (!strcmp(cmd, "ideal_omega_hist")) {    /* counts = (h, alpha, x, y, kvx, kvy, omega0, edges) */
        need(nrhs, 9, "'ideal_omega_hist', h, alpha, x, y, kvx, kvy, omega0, edges");
        int ne = (int)mxGetNumberOfElements(prhs[8]);
        if (ne < 2) mexErrMsgIdAndTxt("swrt:usage", "ideal_omega_hist: at least two edges");
        plhs[0] = mxCreateNumericMatrix(1, ne - 1, mxUINT64_CLASS, mxREAL);
        if (swrt_ideal_omega_hist(h, mxGetScalar(prhs[2]), (int64_t)mxGetNumberOfElements(prhs[3]), mxGetPr(prhs[3]), mxGetPr(prhs[4]), mxGetPr(prhs[5]),
                                  mxGetPr(prhs[6]), (int)mxGetNumberOfElements(prhs[5]), mxGetScalar(prhs[7]), mxGetPr(prhs[8]), ne,
                                  (uint64_t*)mxGetData(plhs[0]))) fail(h, cmd);
    } else if (!strcmp(cmd, "hist2")) {               /* N = (h, qx, xedges, qy, yedges [, alpha])  -- histcounts2, N double */
        need(nrhs, 6, "'hist2', h, qx, xedges, qy, yedges [, alpha]");
        int nxe = (int)mxGetNumberOfElements(prhs[3]), nye = (int)mxGetNumberOfElements(prhs[5]);
        if (nxe < 2 || nye < 2) mexErrMsgIdAndTxt("swrt:usage", "hist2: at least two edges on each axis");
        size_t nb = (size_t)(nxe - 1) * (size_t)(nye - 1);
        uint64_t* c = (uint64_t*)mxCalloc(nb, sizeof(uint64_t));
        if (swrt_hist2(h, (int)mxGetScalar(prhs[2]), mxGetPr(prhs[3]), nxe, (int)mxGetScalar(prhs[4]), mxGetPr(prhs[5]), nye,
                       sc(prhs, nrhs, 6, 0.0), c, 0)) fail(h, cmd);
        plhs[0] = mxCreateDoubleMatrix((size_t)nxe - 1, (size_t)nye - 1, mxREAL);
        for (size_t i = 0; i < nb; i++) mxGetPr(plhs[0])[i] = (double)c[i];
        mxFree(c);
    } else if (!strcmp(cmd, "hist2_sums")) {          /* [S, N] = (h, qx, xedges, qy, yedges, wkinds [, alpha]) */
        /* S(i, j + (v-1)*(nye-1)): kind wkinds(v) summed over bin (i, j), i.e. reshape(S, nxe-1, nye-1, []) is the
         * (nxe-1) x (nye-1) x nw array; N as in 'hist2' */
        need(nrhs, 7, "'hist2_sums', h, qx, xedges, qy, yedges, wkinds [, alpha]");
        int nxe = (int)mxGetNumberOfElements(prhs[3]), nye = (int)mxGetNumberOfElements(prhs[5]);
        int nw = (int)mxGetNumberOfElements(prhs[6]);
        if (nxe < 2 || nye < 2) mexErrMsgIdAndTxt("swrt:usage", "hist2_sums: at least two edges on each axis");
        if (nw < 1 || nw > SWRT_MAX_WEIGHTS) mexErrMsgIdAndTxt("swrt:usage", "hist2_sums: 1 to %d weight kinds", SWRT_MAX_WEIGHTS);
        int32_t wk[SWRT_MAX_WEIGHTS];
        for (int v = 0; v < nw; v++) wk[v] = (int32_t)mxGetPr(prhs[6])[v];
        size_t nb = (size_t)(nxe - 1) * (size_t)(nye - 1);
        uint64_t* c = nlhs > 1 ? (uint64_t*)mxCalloc(nb, sizeof(uint64_t)) : NULL;
        plhs[0] = mxCreateDoubleMatrix((size_t)nxe - 1, (size_t)(nye - 1) * (size_t)nw, mxREAL);
        if (swrt_hist2_sums(h, (int)mxGetScalar(prhs[2]), mxGetPr(prhs[3]), nxe, (int)mxGetScalar(prhs[4]), mxGetPr(prhs[5]), nye,
                            sc(prhs, nrhs, 7, 0.0), wk, nw, NULL, mxGetPr(plhs[0]), c, NULL)) fail(h, cmd);
        if (nlhs > 1) {
            plhs[1] = mxCreateDoubleMatrix((size_t)nxe - 1, (size_t)nye - 1, mxREAL);
            for (size_t i = 0; i < nb; i++) mxGetPr(plhs[1])[i] = (double)c[i];
            mxFree(c);
        }
    } else if (!strcmp(cmd, "packet_quantity")) {     /* q = (h, qkind [, alpha]) */
        need(nrhs, 3, "'packet_quantity', h, qkind [, alpha]");
        if (swrt_packet_quantity(h, (int)mxGetScalar(prhs[2]), sc(prhs, nrhs, 3, 0.0), vec(&plhs[0], n))) fail(h, cmd);
    } else if (!strcmp(cmd, "diag")) {                /* d = (h, alpha) */
        if (swrt_diag(h, sc(prhs, nrhs, 2, 0.0), vec(&plhs[0], 8))) fail(h, cmd);
    } else if (!strcmp(cmd, "omega")) {               /* [omega, Omega] = (h, alpha) */
        double* a = outv(plhs, 0, n); double* b = outv(plhs, 1, n);
        if (swrt_omega(h, sc(prhs, nrhs, 2, 0.0), a, b)) fail(h, cmd);
    } else if (!strcmp(cmd, "set_tuning")) {          /* (h, mtiles, flags) */
        need(nrhs, 4, "'set_tuning', h, mtiles, flags");
        if (swrt_set_tuning(h, (int)mxGetScalar(prhs[2]), (int)mxGetScalar(prhs[3]))) fail(h, cmd);
    } else if (!strcmp(cmd, "synchronize")) {
        if (swrt_synchronize(h)) fail(h, cmd);
    } else {
        mexErrMsgIdAndTxt("swrt:usage", "unknown command '%s'", cmd);
    }
}
