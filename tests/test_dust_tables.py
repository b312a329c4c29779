"""CPU checks of the dust inputs of the diffuse sweep (DESIGN.md 4.8): the band-mean dust cross-sections of
rtb200_uvb_dust_beta against an independent numpy evaluation and a constant fit, their argument checks, the numpy
restatement of the per-leaf dust opacity (tests/dust_oracle.py) against a scalar one, and the dust oracle's iteration
against the scattering oracle's."""
import ctypes as C

import numpy as np
import pytest

import dust_oracle
import scattering_oracle
from radiativetransfer_b200 import _lib
from radiativetransfer_b200 import workloads as W

f32 = lambda x: float(np.float32(x))
FREQDEL = f32(0.02)


def _numpy_dust_beta(alpha, a_dust, nfreq=400, freqdel=FREQDEL):
    """the band sum written independently: vectorised bins, numpy power, the fit of dustModule.f90:36-50"""
    e = 10.0 ** (np.arange(nfreq) * freqdel)
    nu = np.array([W.NU1, W.NU2, W.NU3])
    lam_um = f32(2.99792458e10) / (e * W.EV_TO_HZ) * f32(1e8) / f32(1e4)
    a = np.asarray(a_dust, dtype=np.float64)
    fit = sum(a[t, 1] / ((lam_um / a[t, 0]) ** a[t, 3] + (lam_um / a[t, 0]) ** (-a[t, 4]) + a[t, 2]) for t in range(7))
    sD = f32(1.1) * fit * f32(0.9210340372) * f32(1e-22)
    out = np.zeros(3)
    for g in range(3):
        i = np.arange(1, nfreq)
        f = e[i]
        band = (f >= nu[g]) & (f <= nu[g + 1]) if g < 2 else f >= nu[2]
        dt = (f / nu[g]) ** (-alpha[g]) * (e[i] - e[i - 1])
        shape = (1 - (nu[g + 1] / nu[g]) ** (1 - alpha[g])) / (alpha[g] - 1) if g < 2 else 1 / (alpha[g] - 1)
        out[g] = np.sum((dt * sD[i])[band]) / (shape * nu[g])
    return out


def test_dust_beta_against_numpy(uvbg):
    a_dust = W.synthetic_spectra()["a_dust"]
    got = W.uvb_dust_beta(uvbg["alpha"], a_dust)
    want = _numpy_dust_beta(uvbg["alpha"], a_dust)
    err = float(np.max(np.abs(got - want) / want))
    print(f"betaDust {got}, rel err {err:.2e}")
    assert np.all(got > 0) and err <= 1e-13, err


def test_constant_fit_gives_the_weight_sum(uvbg):
    # one row with p = q = 0 is a / (1 + 1 + b) at every wavelength, the other rows have a = 0
    a_dust = np.array([[1.0, 0.0, 0.0, 1.0, 1.0]] * 7)
    a_dust[3] = [0.5, 3.0, 1.0, 0.0, 0.0]
    sigma = f32(1.1) * (3.0 / 3.0) * f32(0.9210340372) * f32(1e-22)
    alpha = uvbg["alpha"]
    got = W.uvb_dust_beta(alpha, a_dust)
    e = 10.0 ** (np.arange(400) * FREQDEL)
    nu = np.array([W.NU1, W.NU2, W.NU3])
    for g in range(3):
        f = e[1:]
        band = (f >= nu[g]) & (f <= nu[g + 1]) if g < 2 else f >= nu[2]
        dt = (f / nu[g]) ** (-alpha[g]) * np.diff(e)
        shape = (1 - (nu[g + 1] / nu[g]) ** (1 - alpha[g])) / (alpha[g] - 1) if g < 2 else 1 / (alpha[g] - 1)
        want = sigma * np.sum(dt[band]) / (shape * nu[g])
        assert abs(got[g] - want) <= 1e-13 * want, (g, got[g], want)


def test_dust_beta_argument_checks(uvbg):
    L = _lib.lib()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    al, ad, out = np.ascontiguousarray(uvbg["alpha"]), np.ones((7, 5)), np.zeros(3)
    assert L.rtb200_uvb_dust_beta(400, FREQDEL, p(al), p(ad), p(out)) == 0
    for args in ((1, FREQDEL, p(al), p(ad), p(out)), (400, FREQDEL, None, p(ad), p(out)),
                 (400, FREQDEL, p(al), None, p(out)), (400, FREQDEL, p(al), p(ad), None)):
        assert L.rtb200_uvb_dust_beta(*args) == 12
    with pytest.raises(Exception):
        W.uvb_dust_beta(uvbg["alpha"], ad, nfreq=1)


@pytest.mark.parametrize("mode", [1, 2])
def test_numpy_kd_is_the_scalar_formula(mode):
    g = W.uniform_grid(6, seed=5)
    g["abun2"] = np.random.default_rng(3).uniform(1e-3, 2.0, g["level"].size)
    bd = [2.1e-21, 7.3e-22, 3.3e-22]
    kd = dust_oracle.dust_kd(g, bd, mode)
    for i in range(0, g["level"].size, 7):
        for k in range(3):
            if mode == 1:
                want = ((float(g["HI"][i]) * bd[k]) * float(g["abun2"][i])) / f32(0.2)
            else:
                want = ((((f32(0.76) * float(g["rho"][i])) / f32(1.6726231e-24)) * bd[k]) * float(g["abun2"][i])) / f32(0.2)
            assert kd[k, i] == want
    assert np.array_equal(dust_oracle.dust_kd(g, bd, 0), np.zeros((3, g["level"].size)))


def test_albedo_one_is_the_scattering_oracle(uvbg):
    g = W.uniform_grid(4, seed=7)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    kd = dust_oracle.dust_kd(g, [3e-21, 1e-21, 5e-22], 1)
    a = dust_oracle.grid(g).solve(uvb, beta, None, kd, 1.0 * kd, 4, 0.0, nthreads=4)
    b = scattering_oracle.grid(g).solve(uvb, beta, None, kd, 4, 0.0, nthreads=4)
    assert a["status"] == 0 and a["iterations"] == 4 and np.array_equal(a["J"], b["J"])
    c = dust_oracle.grid(g).solve(uvb, beta, None, kd, 0.3 * kd, 4, 0.0, nthreads=4)
    assert np.all(c["J"] < a["J"]) and np.all(c["J"] > 0)
