"""The SPECTRAL paths on flows that weight every wavenumber alike, against long-double references.

The flows of the production workloads fall off as psi-hat ~ K^-3, so a mode at kmax carries ~1/kmax of a k = 1 mode's
weight in a gradient plane and ~1/kmax^2 in u: a wrong twiddle of a high mode in the dense kernel, or a wrong high-kx
column of the anchored leapfrog's transform (K1, anchor_transform_kernel), is diluted by 10^2 - 10^5 before it reaches a
1e-12 bound.  Here the white flow (|u-hat|^2 + |v-hat|^2 flat up to the truncation) and single modes put the whole
weight on the wavenumbers under test:

* dense eval_at at every twiddle home and m-tile count, psi-hat and six-plane uploads, 256^2 and 512^2;
* the leapfrog -- anchored (psi-hat upload) and dense (six planes) -- one step and 8 two-frame sub-steps; the single
  modes at kx = +-kmax, +-(kmax - 1) with one ky in every ky pass, on packets in every anchor-cell residue, put the
  high-kx columns of K1's transform and each of its 64 pre-twiddle phases on their own behind a 1e-12 bound.

What no test here can see: an error of one ulp in one of K1's twiddles or pre-twiddles moves the expansion blocks by
~1e-16 of their size, four orders below the bound and at the level of the transform's own rounding.  A relative error
of 1e-11 in a pre-twiddle, or in a pass twiddle that a kmax mode passes through, fails the anchored tests below."""
import numpy as np
import pytest

import swraytracing_b200 as S
from oracle import c_oracle as CO
from test_spectral_large_grids import TUNINGS, scaled_err, rel_increment_err
from test_nufft_large_grids import (white_flow, single_modes, single_mode_flow, flow_planes, sparse_eval, eval_positions,
                                    cexact)

SIZES = [256, 512]
TOL_FIELD = 1e-12                    # evaluation: of max|plane|
TOL_STEP = 1e-12                     # one leapfrog step: of the increment
TOL_SUBSTEPS = 1e-9                  # 8 two-frame sub-steps: of the increment


def spectral_engine(w, form, two=False):
    """form: psi (psi-hat upload: moment planes, the anchored leapfrog at 256^2 and 512^2), planes (six planes)"""
    e = S.Engine(w.nx, w.L, w.f, w.gH, S.MODE_SPECTRAL)
    for slot in (0, 1) if two else (0,):
        if form == "psi":
            e.set_flow_spectral(w.psik if slot == 0 else w.psik2, slot, w.u_mean)
        else:
            e.set_flow_planes_spectral(flow_planes(w, float(slot)), slot)
    return e


def eval_errors(w, ref_fn):
    x, y = eval_positions(w)
    ref = ref_fn(x, y, flow_planes(w), w.dx, w.nx)
    errs = {}
    for form in ("psi", "planes"):
        with spectral_engine(w, form) as e:
            for mt, tw in TUNINGS:
                e.set_tuning(mt, twiddles=tw)
                errs[(form, mt, tw)] = scaled_err(e.eval_at(x, y), ref)
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("nx", SIZES)
def test_eval_white_flow_every_twiddle_home(nx):
    errs = eval_errors(white_flow(nx), cexact)
    bad = {k: v for k, v in errs.items() if not v < TOL_FIELD}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("nx", SIZES)
def test_eval_single_modes_every_twiddle_home(nx):
    bad = {}
    for kx, ky in single_modes(nx):
        errs = eval_errors(single_mode_flow(nx, kx, ky), sparse_eval)
        bad.update({(kx, ky) + k: v for k, v in errs.items() if not v < TOL_FIELD})
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# the leapfrog
# ------------------------------------------------------------------------------------------------
def leapfrog_ref(x, y, k, l, w, alphas, dt, ref_fn):
    """orc_leapfrog_spectral's arithmetic, operation for operation, with the planes of the flow at alphas[j] in step j"""
    h, f2, gH = dt / 2, w.f * w.f, w.gH
    for al in alphas:
        om = np.sqrt(f2 + gH * (k * k + l * l))
        x = x + h * (gH * k / om)
        y = y + h * (gH * l / om)
        F = ref_fn(x, y, flow_planes(w, al), w.dx, w.nx)
        x = x + dt * F[0]
        y = y + dt * F[1]
        k0, l0 = k, l
        k = k0 - dt * (F[2] * k0 + F[4] * l0)
        l = l0 - dt * (F[3] * k0 + F[5] * l0)
        om = np.sqrt(f2 + gH * (k * k + l * l))
        x = x + h * (gH * k / om)
        y = y + h * (gH * l / om)
    return x, y, k, l


def test_leapfrog_reference_is_the_c_oracle():
    """leapfrog_ref with the C oracle's sums is CO.leapfrog_spectral bit for bit (two-frame, edge positions included)"""
    w = white_flow(48)
    got = leapfrog_ref(w.x, w.y, w.k, w.l, w, [0.25, 0.75], w.dt / 2, cexact)
    ref = (w.x, w.y, w.k, w.l)
    for al in (0.25, 0.75):
        ref = CO.leapfrog_spectral(*ref, flow_planes(w, al), w.dx, w.nx, w.f, w.gH, w.dt / 2, 1, precise=True)
    assert np.array_equal(np.stack(got), np.stack(ref))


def leapfrog_errors(w, form, ref_fn, m=8):
    """(one step, m two-frame sub-steps at alpha_j = (j + 1/2)/m) on residue_packets, of the increment"""
    x, y, k, l = residue_packets(w, w.dt)
    a0, da = 0.5 / m, 1.0 / m
    with spectral_engine(w, form, two=True) as e:
        e.set_packets(x, y, k, l)
        e.step(S.SCHEME_LEAPFROG, w.dt, 1)
        got1 = e.get_packets()
        e.set_packets(x, y, k, l)
        e.step(S.SCHEME_LEAPFROG, w.dt / m, m, a0, da)
        gotm = e.get_packets()
    ref1 = leapfrog_ref(x, y, k, l, w, [0.0], w.dt, ref_fn)
    refm = leapfrog_ref(x, y, k, l, w, [a0 + j * da for j in range(m)], w.dt / m, ref_fn)
    return rel_increment_err(got1, ref1, (x, y, k, l)), rel_increment_err(gotm, refm, (x, y, k, l))


def residue_packets(w, dt, seed=11):
    """64 packets that the first half drift of a step of ``dt`` puts in anchor cells 64 q + s of every residue s (K1's
    pre-twiddle phase: cell c = floor(64 mod(x/dx, nx))) at random q, then the edge positions.  The 64 lie within half a
    period of the origin: a step moves a packet by ~1e-3, and at |x| ~ 3L one rounding of x + dt u -- which an evaluation
    error of 1e-14 of a single mode at kmax flips now and then -- is already 1.4e-12 of that."""
    rs = np.random.RandomState(seed)
    th = rs.uniform(0, 2 * np.pi, 73)
    k, l = 10 * np.cos(th), 10 * np.sin(th)
    om = np.sqrt(w.f * w.f + w.gH * (k * k + l * l))
    q = rs.randint(-w.nx // 2, w.nx // 2 - 1, 64)
    x = (q + (np.arange(64) + 0.5) / 64) * w.dx - dt / 2 * (w.gH * k[:64] / om[:64])
    y = rs.uniform(-w.L / 2, w.L / 2, 64)
    return np.concatenate([x, w.x[-9:]]), np.concatenate([y, w.y[-9:]]), k, l


def pass_modes(nx):
    """kx = +-kmax, +-(kmax - 1) with one ky in each ky pass of the psi-hat stack (an own residue in every pass)"""
    kmax = nx // 2 - 1
    npass = S.engine.spectral_geometry(nx, 3, 1)["npass"]
    per = (nx // 2) // npass
    kys = [p * per + (5 * p) % per for p in range(npass)]
    return [(kx, ky) for ky in kys for kx in (kmax, -kmax, kmax - 1, -(kmax - 1)) if ky or kx > 0]


@pytest.mark.gpu
@pytest.mark.parametrize("nx", SIZES)
@pytest.mark.parametrize("form", ["psi", "planes"])
def test_leapfrog_white_flow(nx, form):
    e1, em = leapfrog_errors(white_flow(nx), form, cexact)
    assert e1 < TOL_STEP and em < TOL_SUBSTEPS, (e1, em)


@pytest.mark.gpu
@pytest.mark.parametrize("nx", SIZES)
@pytest.mark.parametrize("form", ["psi", "planes"])
def test_leapfrog_single_modes_in_every_pass(nx, form):
    bad = {}
    for kx, ky in pass_modes(nx):
        e1, em = leapfrog_errors(single_mode_flow(nx, kx, ky), form, sparse_eval)
        if not (e1 < TOL_STEP and em < TOL_SUBSTEPS):
            bad[(kx, ky)] = (e1, em)
    assert not bad, bad
