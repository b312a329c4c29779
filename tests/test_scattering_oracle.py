"""CPU checks of the scattering extension (DESIGN.md 4.7) on the oracle with scattering (tests/scattering_oracle.py):
sigma = 0 is the emission oracle bit for bit, a single cell follows the closed form of the source iteration, a
conservative box and a thermal + scattering equilibrium reach their fixed points, and the new entry points reject bad
arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import emission_oracle
import scattering_oracle
from radiativetransfer_b200 import workloads as W

NDIR = 192
WEIGHT = float(np.float32(1.0) / np.float32(NDIR))   # equiSources.f90:1386, single-precision division
# the discrete fixed point of a scattering box is uvb * NDIR * WEIGHT up to O((NDIR * WEIGHT - 1) * tau), 3e-8 * tau
FIXED_POINT_BAR = 1e-6


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


@pytest.mark.parametrize("grid", ["uniform", "nested"])
def test_zero_sigma_is_the_emission_oracle_bit_for_bit(uvbg, grid):
    g = W.uniform_grid(6, seed=3) if grid == "uniform" else W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4)
    n = g["level"].size
    uvb = uvbg["uvb"] * 1e-3
    eta = np.random.default_rng(1).uniform(0.0, 1e-45, size=(3, n))
    for e in (None, eta):
        ref = emission_oracle.grid(g)
        if e is not None:
            ref.set_emission(e)
        want = ref.diffuse(uvb, uvbg["beta"])
        sg = scattering_oracle.grid(g)
        if e is not None:
            sg.set_emission(e)
        sg.set_scattering(np.zeros((3, n)))
        o = sg.diffuse(uvb, uvbg["beta"])
        assert o["status"] == 0 and o["nseg"] == want["nseg"]
        assert np.array_equal(o["J"], want["J"])
        # the solve sweeps with the threaded oracle, whose sum over the threads' directions has an order of its own
        want_mt = ref.diffuse_mt(uvb, uvbg["beta"], np.arange(NDIR), nthreads=4)
        s = sg.solve(uvb, uvbg["beta"], e, np.zeros((3, n)), 50, 1e-9, nthreads=4)
        assert s["iterations"] == 2 and s["residual"] == 0.0
        assert np.array_equal(s["J"], want_mt["J"])


@pytest.mark.parametrize("K", [1, 2, 5, 12])
def test_single_cell_follows_the_closed_form(uvbg, K):
    g = W.uniform_grid(1, seed=2)
    kap = _kappa(g, uvbg["beta"])[:, 0]
    sigma = np.array([[0.3], [0.7], [0.9]]) * kap[:, None]   # albedo 0.23 .. 0.47
    eta_th = np.array([[3.0e-44], [1.0e-45], [4.0e-46]])
    # b = dJ / deta of the cell, from two emissive sweeps with the extinction kappa + sigma (uvb = 0)
    sg = scattering_oracle.grid(g)
    sg.set_scattering(sigma)
    sg.set_emission(eta_th)
    J1 = sg.diffuse(np.zeros(3), uvbg["beta"])["J"][:, 0]
    sg.set_emission(2.0 * eta_th)
    J2 = sg.diffuse(np.zeros(3), uvbg["beta"])["J"][:, 0]
    b = (J2 - J1) / eta_th[:, 0]
    q = sigma[:, 0] * b
    want = J1 * (1.0 - q ** K) / (1.0 - q)
    s = scattering_oracle.grid(g).solve(np.zeros(3), uvbg["beta"], eta_th, sigma, K, 0.0)
    assert s["status"] == 0 and s["iterations"] == K
    err = float(np.max(np.abs(s["J"][:, 0] - want) / want))
    assert err < 1e-13, err


def conservative_case(n=4):
    """no absorber, sigma = 1 / box (box tau = 1): J = uvb * NDIR * WEIGHT everywhere at the fixed point"""
    g = W.uniform_grid(n, seed=8)
    g["HI"][:] = 0.0; g["HeI"][:] = 0.0; g["HeII"][:] = 0.0
    sigma = np.full((3, g["level"].size), 1.0 / g["box_size"])
    return g, sigma


def equilibrium_case(uvbg, n=4, seed=9):
    """absorber kappa_abs varying per cell, eta_th = S kappa_abs, uvb = S: J = S * NDIR * WEIGHT at the fixed point"""
    g = W.uniform_grid(n, seed=seed, tau_lo=0.05, tau_hi=0.5)
    kap = _kappa(g, uvbg["beta"])
    S = uvbg["uvb"] * 1e-3
    rng = np.random.default_rng(seed)
    sigma = kap * rng.uniform(0.1, 9.0, size=kap.shape)   # albedo 0.1 .. 0.9
    return g, S, S[:, None] * kap, sigma


def test_conservative_box_converges_to_the_boundary(uvbg):
    g, sigma = conservative_case()
    s = scattering_oracle.grid(g).solve(uvbg["uvb"], uvbg["beta"], None, sigma, 400, 1e-12)
    assert s["status"] == 0 and s["residual"] <= 1e-12, (s["iterations"], s["residual"])
    want = uvbg["uvb"][:, None] * (NDIR * WEIGHT)
    err = float(np.max(np.abs(s["J"] - want) / want))
    print(f"conservative box: {s['iterations']} iterations, err {err:.3e}")
    assert err < FIXED_POINT_BAR, err


def test_thermal_and_scattering_equilibrium(uvbg):
    g, S, eta_th, sigma = equilibrium_case(uvbg)
    s = scattering_oracle.grid(g).solve(S, uvbg["beta"], eta_th, sigma, 400, 1e-12)
    assert s["status"] == 0 and s["residual"] <= 1e-12, (s["iterations"], s["residual"])
    want = S[:, None] * (NDIR * WEIGHT)
    err = float(np.max(np.abs(s["J"] - want) / want))
    print(f"equilibrium: {s['iterations']} iterations, err {err:.3e}")
    assert err < FIXED_POINT_BAR, err


def test_residual_definition():
    J = np.array([[1.0, 0.0, 2.0], [4.0, 0.0, 5.0]])
    assert scattering_oracle.residual(J, J.copy()) == 0.0
    assert scattering_oracle.residual(J, J * 0.5) == 0.5
    P = J.copy(); P[0, 1] = 1e-300
    assert scattering_oracle.residual(J, P) == np.inf


def test_scattering_entry_points_reject_bad_arguments_without_a_device(build_product):
    from radiativetransfer_b200 import _lib
    L = _lib.lib()
    s = np.zeros(3)
    it, r = C.c_int32(0), C.c_double(0)
    assert L.rtb200_grid_set_scattering(None, s.ctypes.data_as(C.c_void_p), 10, 1e-9) == 12   # RTB200_ERR_ARG
    assert L.rtb200_grid_set_scattering(None, None, 1, 0.0) == 12
    assert L.rtb200_last_scattering(None, C.byref(it), C.byref(r)) == 12
