"""CPU checks of the emission extension (DESIGN.md 4.6) on the oracle with emission (tests/emission_oracle.py): an
independent numpy evaluation of one cell, eta = 0 is the unmodified oracle's sweep bit for bit, the equilibrium S = eta / kappa is reproduced, linearity in (uvb, eta),
exact scaling without opacity, and the new entry points reject bad arguments without a device."""
import ctypes as C
import math

import numpy as np
import pytest

import emission_oracle
from radiativetransfer_b200 import workloads as W

NDIR = 192
WEIGHT = float(np.float32(1.0) / np.float32(NDIR))   # equiSources.f90:1386, single-precision division


def _og(oracle, g):
    return emission_oracle.grid(g)


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


def _phi(tau):
    if tau < 1e-2:
        return 0.5 + tau * (-1 / 6 + tau * (1 / 24 + tau * (-1 / 120 + tau * (1 / 720 + tau * (-1 / 5040 + tau / 40320)))))
    return (tau - (1.0 - math.exp(-tau))) / (tau * tau)


def _one_cell_J(pattern_row, box, kappa, eta, uvb):
    """J of the single cell of an n = 1 grid for one direction: every segment is fed by the boundary"""
    lens = [pattern_row[2], pattern_row[5], pattern_row[8]]   # xy, xz, yz: the reference's order
    J = np.zeros(3)
    for g in range(3):
        js = []
        for ln in lens:
            if ln <= 0.0:
                continue
            d = float(box) * float(ln)
            tau = float(kappa[g]) * d
            a = math.exp(-tau)   # the C library's exp / log (numpy's vectorised ones may differ in the last bit)
            Iin, Iatt = float(uvb[g]), float(uvb[g]) * a
            L = (Iin - Iatt) / math.log(Iin / Iatt) if Iatt < Iin else 0.5 * (Iin + Iatt)
            js.append(L + float(eta[g]) * d * _phi(tau))
        J[g] = sum(js) / len(js) * WEIGHT
    return J


@pytest.mark.parametrize("opacity", ["kappa>0", "kappa=0"])
def test_single_cell_matches_numpy_for_every_direction(oracle, uvbg, opacity):
    from radiativetransfer_b200 import _lib
    L = _lib.lib()
    g = W.uniform_grid(1, seed=2)
    if opacity == "kappa=0":
        g["HI"][:] = 0.0; g["HeI"][:] = 0.0; g["HeII"][:] = 0.0
    og = _og(oracle, g)
    eta = np.array([[3.0e-44], [1.0e-45], [4.0e-46]])
    og.set_emission(eta)
    kap = _kappa(g, uvbg["beta"])[:, 0]
    pat = np.zeros((1, 12))
    worst = 0.0
    for ray in range(NDIR):
        assert L.rtb200_patterns(3, ray, 1, pat.ctypes.data_as(C.c_void_p)) == 0
        o = og.diffuse(uvbg["uvb"], uvbg["beta"], ray_begin=ray, ray_end=ray + 1)
        assert o["status"] == 0
        ref = _one_cell_J(pat[0], g["box_size"], kap, eta[:, 0], uvbg["uvb"])
        worst = max(worst, float(np.max(np.abs(o["J"][:, 0] - ref) / np.abs(ref))))
    assert worst < 1e-14, worst


@pytest.mark.parametrize("grid", ["uniform", "nested"])
def test_zero_emission_is_the_emission_free_sweep_bit_for_bit(oracle, uvbg, grid):
    g = W.uniform_grid(6, seed=3) if grid == "uniform" else W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4)
    uvb = uvbg["uvb"] * 1e-3
    ref = oracle.OracleGrid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"]).diffuse(uvb, uvbg["beta"])
    og = _og(oracle, g)
    assert np.array_equal(og.diffuse(uvb, uvbg["beta"])["J"], ref["J"])
    og.set_emission(np.zeros((3, g["level"].size)))
    o = og.diffuse(uvb, uvbg["beta"])
    assert o["status"] == 0 and o["nseg"] == ref["nseg"]
    assert np.array_equal(o["J"], ref["J"])


def equilibrium_case(g, uvbg):
    """uniform opacity and uvb_g = S_g = eta_g / kappa_g: I = S on every path, J = S * ndir * weight everywhere"""
    n = g["level"].size
    g = dict(g, HI=np.full(n, 1.0e-4), HeI=np.zeros(n), HeII=np.zeros(n))
    kap = _kappa(g, uvbg["beta"])
    S = uvbg["uvb"] * 1e-3
    eta = S[:, None] * kap
    return g, S, eta, S[:, None] * (NDIR * WEIGHT)


@pytest.mark.parametrize("grid", ["uniform", "nested"])
def test_equilibrium_source_function(oracle, uvbg, grid):
    g = W.uniform_grid(6, seed=5) if grid == "uniform" else W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4)
    g, S, eta, want = equilibrium_case(g, uvbg)
    og = _og(oracle, g)
    og.set_emission(eta)
    o = og.diffuse(S, uvbg["beta"])
    assert o["status"] == 0
    err = float(np.max(np.abs(o["J"] - want) / want))
    assert err < 1e-12, err


def linearity_case(uvbg, seed=11):
    # per-cell tau >= 0.1: the reference's log-mean carries ~1e-16 / tau rounding noise per segment, and corner clips make
    # segments far shorter than a cell (at tau_cell >= 1e-3 that noise alone reaches 3e-11 of a cell's J)
    g = W.uniform_grid(8, seed=seed, tau_lo=0.1)
    kap = _kappa(g, uvbg["beta"])
    rng = np.random.default_rng(seed)
    ratio = 10.0 ** rng.uniform(-3.0, 3.0, size=kap.shape)   # S / uvb from 1e-3 to 1e3
    eta = ratio * uvbg["uvb"][:, None] * kap
    return g, eta


def test_linearity_in_boundary_intensity_and_emission(oracle, uvbg):
    g, eta = linearity_case(uvbg)
    og = _og(oracle, g)
    og.set_emission(eta)
    both = og.diffuse(uvbg["uvb"], uvbg["beta"])["J"]
    only_eta = og.diffuse(np.zeros(3), uvbg["beta"])["J"]
    og.set_emission(None)
    only_uvb = og.diffuse(uvbg["uvb"], uvbg["beta"])["J"]
    err = float(np.max(np.abs(both - (only_uvb + only_eta)) / np.abs(both)))
    assert err < 1e-12, err


def test_scaling_without_opacity_is_exact(oracle, uvbg):
    g = W.uniform_grid(5, seed=6)
    g["HI"][:] = 0.0; g["HeI"][:] = 0.0; g["HeII"][:] = 0.0
    rng = np.random.default_rng(3)
    eta = rng.uniform(0.0, 1e-44, size=(3, g["level"].size))
    og = _og(oracle, g)
    og.set_emission(eta)
    one = og.diffuse(np.zeros(3), uvbg["beta"])["J"]
    og.set_emission(2.0 * eta)
    two = og.diffuse(np.zeros(3), uvbg["beta"])["J"]
    assert np.array_equal(two, 2.0 * one)


def test_emission_entry_points_reject_bad_arguments_without_a_device(build_product):
    from radiativetransfer_b200 import _lib
    L = _lib.lib()
    eta = np.zeros(3)
    assert L.rtb200_grid_set_emission(None, eta.ctypes.data_as(C.c_void_p)) == 12       # RTB200_ERR_ARG
    assert L.rtb200_grid_set_emission(None, None) == 12
    assert L.rtb200_grid_set_emission_device(None, eta.ctypes.data_as(C.c_void_p), None) == 12
    assert L.rtb200_grid_set_emission_device(None, None, None) == 12
