"""CPU checks of the accelerated source iteration (DESIGN.md 4.9) restated in numpy over oracle sweeps
(tests/ng_oracle.py): without acceleration it is the plain solve bit for bit, Ng is exact on a cell with two error
modes, Ng converges to the plain answer with far fewer sweeps, a warm start saves sweeps after a small change of sigma,
and the new entry points reject a NULL handle without a device."""
import ctypes as C

import numpy as np
import pytest

import ng_oracle
import scattering_oracle
from radiativetransfer_b200 import workloads as W

NTHREADS = 8


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


def _case(name):
    """the two grids of DESIGN.md 4.9's table: (grid, uvb scale); the nested one inside the refined-leaf intensity guard"""
    if name == "uniform":
        return W.uniform_grid(8, seed=3), 1.0
    return W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4), 1e-3


def test_without_acceleration_it_is_the_plain_solve_bit_for_bit(uvbg):
    g = W.uniform_grid(4, seed=5)
    sigma = _kappa(g, uvbg["beta"])   # albedo 0.5
    eta = np.random.default_rng(2).uniform(0.0, 1e-45, size=sigma.shape)
    want = scattering_oracle.grid(g).solve(uvbg["uvb"], uvbg["beta"], eta, sigma, 200, 1e-9, nthreads=NTHREADS)
    got = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvbg["uvb"], uvbg["beta"], eta, sigma, 200, 1e-9,
                                      ng=False, nthreads=NTHREADS)
    assert got["iterations"] == want["iterations"] and got["extrapolations"] == 0
    assert got["history"] == want["history"]
    assert np.array_equal(got["J"], want["J"])


@pytest.mark.parametrize("frac", [(0.3, 0.7, 0.0), (0.9, 0.5, 0.0)])
def test_two_error_modes_extrapolate_to_the_closed_form_limit(uvbg, frac):
    # one thick cell, two scattering groups: the error of plain iteration is two geometric modes, which Ng removes exactly
    g = W.uniform_grid(1, seed=2, tau_lo=5.0, tau_hi=5.0)
    kap = _kappa(g, uvbg["beta"])[:, 0]
    sigma = np.array(frac)[:, None] * kap[:, None]
    eta_th = np.array([[3.0e-44], [1.0e-45], [4.0e-46]])
    sg = scattering_oracle.grid(g)
    sg.set_scattering(sigma)
    sg.set_emission(eta_th)
    J1 = sg.diffuse(np.zeros(3), uvbg["beta"])["J"][:, 0]
    sg.set_emission(2.0 * eta_th)
    J2 = sg.diffuse(np.zeros(3), uvbg["beta"])["J"][:, 0]
    b = (J2 - J1) / eta_th[:, 0]
    want = J1 / (1.0 - sigma[:, 0] * b)
    s = ng_oracle.solve_accelerated(scattering_oracle.grid(g), np.zeros(3), uvbg["beta"], eta_th, sigma, 5, 0.0,
                                    nthreads=1)
    assert s["status"] == 0 and s["iterations"] == 5 and s["extrapolations"] == 1
    err = float(np.max(np.abs(s["J"][:, 0] - want) / want))
    assert err <= 1e-10, err
    # without Ng five sweeps are far from it
    p = ng_oracle.solve_accelerated(scattering_oracle.grid(g), np.zeros(3), uvbg["beta"], eta_th, sigma, 5, 0.0,
                                    ng=False, nthreads=1)
    assert float(np.max(np.abs(p["J"][:, 0] - want) / want)) > 1e-3


@pytest.mark.parametrize("albedo,ratio", [(0.5, 0.7), (0.9, 0.4)])
@pytest.mark.parametrize("grid", ["uniform", "nested"])
def test_ng_converges_to_the_plain_answer_in_fewer_sweeps(uvbg, grid, albedo, ratio):
    g, scale = _case(grid)
    sigma = albedo / (1.0 - albedo) * _kappa(g, uvbg["beta"])
    uvb = scale * uvbg["uvb"]
    plain = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, uvbg["beta"], None, sigma, 600, 1e-9, ng=False,
                                        nthreads=NTHREADS)
    ng = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, uvbg["beta"], None, sigma, 600, 1e-9,
                                     nthreads=NTHREADS)
    assert plain["residual"] <= 1e-9 and ng["residual"] <= 1e-9
    diff = float(np.max(np.abs(ng["J"] - plain["J"]) / plain["J"]))
    print(f"{grid} albedo {albedo}: plain {plain['iterations']} sweeps, Ng {ng['iterations']} "
          f"({ng['extrapolations']} extrapolations), max rel diff {diff:.2e}")
    assert diff <= 1e-6, diff
    assert ng["extrapolations"] >= 1
    assert ng["iterations"] <= ratio * plain["iterations"], (ng["iterations"], plain["iterations"])


@pytest.mark.parametrize("grid", ["uniform", "nested"])
def test_warm_start(uvbg, grid):
    g, scale = _case(grid)
    sigma = _kappa(g, uvbg["beta"])   # albedo 0.5
    uvb = scale * uvbg["uvb"]
    first = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, uvbg["beta"], None, sigma, 600, 1e-9,
                                        nthreads=NTHREADS)
    # unchanged inputs: the stored J is already the answer
    same = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, uvbg["beta"], None, sigma, 600, 1e-8,
                                       x0=first["J"], nthreads=NTHREADS)
    assert same["iterations"] <= 2, same["iterations"]
    # one outer step's worth of change: sigma within +-1 %
    pert = sigma * np.random.default_rng(7).uniform(0.99, 1.01, size=sigma.shape)
    for ng in (False, True):
        cold = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, uvbg["beta"], None, pert, 600, 1e-8, ng=ng,
                                           nthreads=NTHREADS)
        warm = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, uvbg["beta"], None, pert, 600, 1e-8, ng=ng,
                                           x0=first["J"], nthreads=NTHREADS)
        print(f"{grid} ng={ng}: cold {cold['iterations']} warm {warm['iterations']} sweeps")
        assert warm["iterations"] <= 0.7 * cold["iterations"], (warm["iterations"], cold["iterations"])


def test_ng_coefficients_skip_a_singular_system():
    I = np.full((3, 4), 2.0)
    assert ng_oracle.ng_coefficients(I, I, I, I) is None     # converged: every difference is 0
    rng = np.random.default_rng(3)
    I0, I1, I2, I3 = (rng.uniform(1.0, 2.0, size=(3, 4)) for _ in range(4))
    assert ng_oracle.ng_coefficients(I0, I1, I2, I3) is not None


def test_acceleration_entry_points_reject_a_null_handle_without_a_device(build_product):
    from radiativetransfer_b200 import _lib
    L = _lib.lib()
    n, w = C.c_int32(0), C.c_int32(0)
    assert L.rtb200_grid_set_scattering_acceleration(None, 0) == 12   # RTB200_ERR_ARG
    assert L.rtb200_grid_set_scattering_acceleration(None, 3) == 12
    assert L.rtb200_last_scattering_acceleration(None, C.byref(n), C.byref(w)) == 12
