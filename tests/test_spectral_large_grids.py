"""The dense SPECTRAL kernels above 128^2, and at the smallest grids, against the C oracle's long-double Fourier sums.

Above 128^2 make_geom moves a step's x twiddles from the shared-memory table to the per-CTA global (L2) scratch, splits
the stack into several ky passes, zero-pads the k-steps up to a whole chunk for most sizes, and off powers of two
reduces positions with fmod.  The psi-hat leapfrog at 256^2 and 512^2 runs anchored (test_spectral_anchored.py), so the
dense leapfrog, the fused RK4 steppers and the ode23 evaluations are checked here on their own at those sizes.

* evaluation at every size of EVAL_SIZES: psi-hat, six and seven planes, both m-tiles, all four twiddle homes;
* the dense leapfrog (six planes, psi-hat with and without the moment planes): one step and 8 two-frame sub-steps;
* the fused RK4 steppers step_packet / step_packet_xka: 2 steps, steady and two-frame;
* ode23 at 256^2 (coupled, dense output, backward, per packet) and at 512^2;
* a CPU guard: EVAL_SIZES reaches every class of dense-kernel geometry the planner produces for even nx in 8..1024.

Trajectories are measured by the largest difference relative to the largest increment of each component, so that a
wrong twiddle of a small mode is not hidden under the size of x or k."""
import numpy as np
import pytest

import swraytracing_b200 as S
from swraytracing_b200 import workloads as W
from oracle import c_oracle as CO
from oracle import swrt_oracle as O
import ode23_backward_oracle as B

# Grid sizes of the evaluation tests (here and test_gpu_parity.test_spectral_eval_vs_exact_sum).  Some classes only one
# size of the list reaches: 8 and 10 (one pass, padded k-steps), 30 (one pass, not a power of two), 66 and 96 (several
# passes with the shared-memory table, off powers of two), 258 (L2 table, padded) and 384 (L2 table, unpadded, fmod
# reduction) for some plane counts.  test_eval_sizes_reach_every_geometry_class fails when the planner adds a class.
EVAL_SIZES = [8, 10, 16, 30, 32, 36, 48, 64, 66, 96, 128, 130, 192, 256, 258, 384, 512, 1024]
PLANE_COUNTS = (3, 6, 7)             # psi-hat moments, six velocity / gradient planes, six + H
TOL_FIELD = 1e-12                    # evaluation: of max|plane| (the exact sums' own accuracy is ~1e-16)
TOL_STEP = 1e-12                     # one leapfrog step: of the increment
TOL_SUBSTEPS = 1e-9                  # 8 two-frame leapfrog sub-steps, 2 RK4 steps, ode23 solves: of the increment
TOL_RK4 = 1e-11                      # 2 fused RK4 steps: of the increment, the bound that holds at 64^2 and 128^2


def geometry_class(nx, npl):
    """(planes, twiddle home, single ky pass, zero-padded k-steps, power of two) of the one-m-tile dense kernel"""
    g = S.engine.spectral_geometry(nx, npl, 1)
    return (npl, g["twiddle_table"], g["npass"] == 1, g["ksteps"] > (nx // 2 + 1) // 2, nx & (nx - 1) == 0)


def test_eval_sizes_reach_every_geometry_class():
    every = {}
    for nx in range(8, 1025, 2):
        for npl in PLANE_COUNTS:
            every.setdefault(geometry_class(nx, npl), nx)
    hit = {geometry_class(nx, npl) for nx in EVAL_SIZES for npl in PLANE_COUNTS}
    missing = {c: nx for c, nx in every.items() if c not in hit}
    assert not missing, f"no size in EVAL_SIZES for these classes (class: smallest nx): {missing}"


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def edge_positions(L, dx):
    """the edge positions of test_edge_cases_empty_single_ragged_nonfinite on this grid: a huge and a tiny negative
    position, +-L, grid nodes and +-L/2"""
    x = np.array([1e6 + 0.123, -1e-20, L, -L, 0.0, 5 * dx, -3 * dx, L / 2, -L / 2])
    y = np.array([-L / 2, L, 7 * dx, -1e-20, 1e6 + 0.123, -L, L / 2, 0.0, 2 * dx])
    return x, y


def sample(name, nx, nrand, seed=5):
    """workload ``name`` at nx (C3: L = 2 pi; C4: L = 20 with the mean shear; C5: the step_packet_xka state) and
    ``nrand`` seeded positions in [-3L, 3L] followed by the edge positions; k, l are the workload's"""
    w = W.make_workload(name, n_packets=nrand + 9, nx=nx)
    xe, ye = edge_positions(w.L, w.dx)
    rs = np.random.RandomState(seed)
    x = np.concatenate([rs.uniform(-3 * w.L, 3 * w.L, nrand), xe])
    y = np.concatenate([rs.uniform(-3 * w.L, 3 * w.L, nrand), ye])
    return w, (x, y, w.k.copy(), w.l.copy())


def eta_scale(w):
    return 0.3 / np.abs(W._fulspec_ifft(w.psik)).max()          # |eta| <= 0.3, so that H = 1 + eta stays positive


def planes_at(w, alpha=0.0, seven=False):
    """the coefficient planes of the flow (1 - alpha)*frame 0 + alpha*frame 1"""
    psik = w.psik if alpha == 0.0 else (1.0 - alpha) * w.psik + alpha * w.psik2
    return W.planes_from_psik(psik, w.L, w.u_mean, etak=eta_scale(w) * psik if seven else None)


def engine(w, form, two=False):
    """form: psi (psi-hat upload, moment planes), psi6 (psi-hat upload, six planes contracted), planes (six planes),
    seven (six planes + H)"""
    e = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL)
    for slot in (0, 1) if two else (0,):
        if form in ("psi", "psi6"):
            e.set_flow_spectral(w.psik if slot == 0 else w.psik2, slot, w.u_mean)
        else:
            e.set_flow_planes_spectral(planes_at(w, float(slot), seven=form == "seven"), slot)
    if form == "psi6":
        e.set_tuning(use_psi_moments=False)
    return e


def scaled_err(got, ref):
    scale = np.abs(ref).max(axis=1, keepdims=True)
    scale[scale == 0] = 1.0
    return float((np.abs(got - ref) / scale).max())


def rel_increment_err(got, ref, start):
    d_got = np.stack(got) - np.stack(start)
    d_ref = np.stack(ref) - np.stack(start)
    scale = np.abs(d_ref).max(axis=1, keepdims=True)
    scale[scale == 0] = 1.0
    return float((np.abs(d_got - d_ref) / scale).max())


# ------------------------------------------------------------------------------------------------
# evaluation: every geometry class, every twiddle home, seven planes
# ------------------------------------------------------------------------------------------------
TUNINGS = [(1, 0), (1, 1), (1, 2), (1, 3), (2, 0)]      # (m-tiles, twiddle home); two m-tiles always rotate in registers


def eval_errors(nx, name):
    """{(form, mtiles, twiddles): error} of eval_at against the exact sums; asserts the reversed ensemble is bit-exact"""
    w, (x, y, _, _) = sample(name, nx, 64)
    ref = CO.spectral_eval(x, y, planes_at(w, seven=True), w.dx, nx, precise=True)
    xr, yr = x[::-1].copy(), y[::-1].copy()
    errs = {}
    for form, npl in (("psi", 3), ("planes", 6), ("seven", 6)):
        with engine(w, form) as e:
            assert e.contracted_planes() == npl
            seven = form == "seven"
            for mt, tw in TUNINGS:
                e.set_tuning(mt, twiddles=tw)
                got = e.eval_at(x, y, with_H=seven)
                errs[(form, mt, tw)] = scaled_err(got, ref[:7 if seven else 6])
                rev = e.eval_at(xr, yr, with_H=seven)
                assert np.array_equal(rev[:, ::-1], got), (form, mt, tw)   # a packet's value does not depend on its slot
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("nx", EVAL_SIZES)
@pytest.mark.parametrize("name", ["C3", "C4"])
def test_eval_every_twiddle_home_and_seven_planes(nx, name):
    errs = eval_errors(nx, name)
    bad = {k: v for k, v in errs.items() if not v < TOL_FIELD}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# the dense leapfrog
# ------------------------------------------------------------------------------------------------
LEAPFROG_SIZES = [8, 10, 192, 256, 512, 1024]


def leapfrog_errors(nx, name, form, m=8, make=None):
    """(one step, m two-frame sub-steps at alpha_j = (j + 1/2)/m) against CO.leapfrog_spectral, relative to the
    increment; ``make(w, form, two)`` builds the engine (default: this file's dense-mode ``engine``)"""
    w, (x, y, k, l) = sample(name, nx, 40)
    with (make or engine)(w, form, two=True) as e:
        if make is None:
            assert e.contracted_planes() == (3 if form == "psi" else 6)
        e.set_packets(x, y, k, l)
        e.step(S.SCHEME_LEAPFROG, w.dt, 1)
        got1 = e.get_packets()
        xs, ys, ks, ls = (v[-25:] for v in (x, y, k, l))          # 16 random + the edge positions
        a0, da = 0.5 / m, 1.0 / m
        e.set_packets(xs, ys, ks, ls)
        e.step(S.SCHEME_LEAPFROG, w.dt / m, m, a0, da)           # pre-blended stacks, one per sub-step
        gotm = e.get_packets()
    ref1 = CO.leapfrog_spectral(x, y, k, l, planes_at(w), w.dx, nx, w.f, w.gH, w.dt, 1, precise=True)
    refm = (xs, ys, ks, ls)
    for j in range(m):
        refm = CO.leapfrog_spectral(*refm, planes_at(w, a0 + j * da), w.dx, nx, w.f, w.gH, w.dt / m, 1, precise=True)
    return rel_increment_err(got1, ref1, (x, y, k, l)), rel_increment_err(gotm, refm, (xs, ys, ks, ls))


@pytest.mark.gpu
@pytest.mark.parametrize("nx", LEAPFROG_SIZES)
@pytest.mark.parametrize("name", ["C3", "C4"])
@pytest.mark.parametrize("form", ["planes", "psi6", "psi"])
def test_leapfrog_against_the_exact_sum(nx, name, form):
    """planes and psi6 take the dense kernel on six contracted planes at every size; psi takes it on the psi-hat moment
    planes, except at 256^2 and 512^2 where it runs anchored and must meet the same bounds"""
    e1, em = leapfrog_errors(nx, name, form)
    assert e1 < TOL_STEP and em < TOL_SUBSTEPS, (e1, em)


# ------------------------------------------------------------------------------------------------
# the fused RK4 steppers (spectral_rk4_kernel)
# ------------------------------------------------------------------------------------------------
RK4_SIZES = [64, 128, 130, 256, 512]              # 64 and 128 (shared-memory table) calibrate TOL_RK4
RK4_CASES = [("rk4_packet", "psi"), ("rk4_packet", "planes"), ("rk4_packet", "two-frame"), ("rk4_xka", "planes"),
             ("rk4_xka", "two-frame")]


def rk4_error(nx, scheme, flow, make=None, unfused=False):
    """2 fused steps (the composed launches with ``unfused``) against step_packet / step_packet_xka with exact-sum
    fields; wave action as in test_spectral_fused_rk4_equals_the_composed_launches"""
    xka = scheme == "rk4_xka"
    two = flow == "two-frame"
    w, (x, y, k, l) = sample("C4" if two else "C5", nx, 55)
    a = np.linspace(0.5, 2.0, x.size)
    seven = xka or flow == "planes"
    m = 2
    a0, da = (0.5 / m, 1.0 / m) if two else (0.0, 0.0)
    with (make or engine)(w, "seven" if seven else "psi", two=two) as e:
        if unfused:
            e.set_tuning(unfused_rk4=True)
        e.set_packets(x, y, k, l, a)
        e.step(S.SCHEME_RK4_XKA if xka else S.SCHEME_RK4_PACKET, w.dt, m, a0, da)
        got = e.get_packets(with_a=True)
    ev = lambda xx, yy, pl: CO.spectral_eval(xx, yy, pl, w.dx, nx, precise=True)
    ref = (x, y, k, l, a)
    for j in range(m):
        ref = O.rk4_step_batch(*ref, w.dt, w.Cg, w.f, None, w.dx, xka, mode="spectral",
                               planes_k=planes_at(w, a0 + j * da, seven=seven), nx=nx, eval_planes=ev)
    if xka:
        assert np.abs(got[4] - a).max() > 1e-6                  # wave action does evolve
    return rel_increment_err(got, ref, (x, y, k, l, a))


@pytest.mark.gpu
@pytest.mark.parametrize("nx", RK4_SIZES)
@pytest.mark.parametrize("scheme,flow", RK4_CASES)
def test_fused_rk4_against_the_exact_sum(nx, scheme, flow):
    err = rk4_error(nx, scheme, flow)
    assert err < TOL_RK4, err


# ------------------------------------------------------------------------------------------------
# ode23 (the device-chosen evaluation frame, the per-packet plane blend) at 256^2 and 512^2
# ------------------------------------------------------------------------------------------------
T_ODE = 0.4


def ray_ode(w, n, two):
    """odefun of generate_raytracing_ode with the six fields from the exact sums of the frame blended at t / T_ODE"""
    def eval6(xx, yy, al):
        return CO.spectral_eval(xx, yy, planes_at(w, al if two else 0.0), w.dx, w.nx, precise=True)
    return O.generate_raytracing_ode(None, None, n, w.f, w.Cg, T_ODE if two else np.inf, w.dx, eval6=eval6)


def c3_packets(nx):
    w, pk = sample("C3", nx, 7)
    return w, np.stack(pk)


def mixed_tspans(n, nt=5, seed=3):
    """per-packet tspans: forward [T - t, T], backward [t, 0] and zero-length rows, in turn"""
    rs = np.random.RandomState(seed)
    T = rs.uniform(0.5, 1.0, n) * T_ODE
    ts = np.empty((nt, n))
    for i in range(n):
        ts[:, i] = (np.linspace(T_ODE - T[i], T_ODE, nt), np.linspace(T[i], 0.0, nt), np.full(nt, T[i]))[i % 3]
    return ts


def ode23_errors(nx, form, two, make=None, packets=c3_packets, tspans=False):
    """Engine.ode23 over [0, T], a 7-entry dense tspan forward and backward, and Engine.ode23_packets on every other
    packet (with ``tspans`` also on mixed_tspans, one tspan per packet), against the oracle's ode23; the step counts
    must be identical"""
    w, pk = packets(nx)
    n = pk.shape[1]
    tmax = T_ODE if two else None
    errs = {}
    sub = pk[:, ::2]
    ts2 = mixed_tspans(sub.shape[1])
    with (make or engine)(w, form, two=two) as e:
        for key, tspan in (("final", [0.0, T_ODE]), ("dense", T_ODE * np.linspace(0, 1, 7)),
                           ("backward", T_ODE * np.linspace(1, 0, 7))):
            e.set_packets(*pk)
            st = e.ode23(tspan, tmax)
            yref, sref = B.ode23(ray_ode(w, n, two), tspan, pk.ravel())
            assert (st["nsteps"], st["nfailed"], st["nfevals"]) == (sref["nsteps"], sref["nfailed"], sref["nfevals"]), key
            assert st["nsteps"] >= 10                              # MaxStep = 0.1*|tf - t0|
            if key == "final":
                errs[key] = rel_increment_err(np.stack(e.get_packets()), yref.reshape(4, n), pk)
            else:
                assert np.array_equal(st["Y"][0], pk)
                errs[key] = max(rel_increment_err(st["Y"][j], yref[j].reshape(4, n), pk) for j in range(1, 7))
        e.set_packets(*sub)
        st = e.ode23_packets([0.0, T_ODE], tmax)
        got = np.stack(e.get_packets())
        if tspans:
            e.set_packets(*sub)
            st2 = e.ode23_packets(ts2, tmax)
            got2 = np.stack(e.get_packets())
    ref, ref2 = [], []
    for i in range(sub.shape[1]):
        yi, si = B.ode23(ray_ode(w, 1, two), [0.0, T_ODE], sub[:, i])
        ref.append(yi)
        assert (st["steps"][i], st["rejected"][i]) == (si["nsteps"], si["nfailed"]), i
        if tspans:
            Yi, si = B.ode23(ray_ode(w, 1, two), ts2[:, i], sub[:, i])
            ref2.append(Yi)
            assert (st2["steps"][i], st2["rejected"][i]) == (si["nsteps"], si["nfailed"]), ("tspans", i)
    assert np.all(st["status"] == 0)
    errs["packets"] = rel_increment_err(got, np.stack(ref, axis=1), sub)
    if tspans:
        assert np.all(st2["status"] == 0)
        Y2 = np.stack(ref2, axis=2)                               # (nt, 4, n)
        assert np.array_equal(st2["Y"][0], sub) and np.array_equal(got2[:, 2::3], sub[:, 2::3])
        errs["tspans"] = max(rel_increment_err(st2["Y"][j], Y2[j], sub) for j in range(1, ts2.shape[0]))
        errs["tspans final"] = rel_increment_err(got2, Y2[-1], sub)
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["psi", "planes"])
@pytest.mark.parametrize("two", [False, True])
def test_ode23_256(form, two):
    errs = ode23_errors(256, form, two)
    assert max(errs.values()) < TOL_SUBSTEPS, errs


def ode23_steady_error(nx, make=None, packets=c3_packets):
    """one coupled steady solve over [0, T] on a psi-hat flow against the oracle: identical counts, error of the increment"""
    w, pk = packets(nx)
    with (make or engine)(w, "psi") as e:
        e.set_packets(*pk)
        st = e.ode23([0.0, T_ODE], None)
        got = np.stack(e.get_packets())
    yref, sref = B.ode23(ray_ode(w, pk.shape[1], False), [0.0, T_ODE], pk.ravel())
    assert (st["nsteps"], st["nfailed"], st["nfevals"]) == (sref["nsteps"], sref["nfailed"], sref["nfevals"])
    return rel_increment_err(got, yref.reshape(4, -1), pk)


@pytest.mark.gpu
def test_ode23_512_steady():
    err = ode23_steady_error(512)
    assert err < TOL_SUBSTEPS, err
