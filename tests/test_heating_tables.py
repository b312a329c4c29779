"""CPU checks of the inputs and the definition of the heating pass (DESIGN.md 4.10): the band widths of
rtb200_uvb_band_width against an independent numpy evaluation, the dust band integral betaDust * W against a numpy sum
over the 400 bins, the argument checks, workloads.uvb_heating, and the numpy restatement of the pass
(tests/heating_oracle.py) against a scalar hand computation."""
import ctypes as C

import numpy as np
import pytest

import heating_oracle
from radiativetransfer_b200 import _lib
from radiativetransfer_b200 import workloads as W

f32 = lambda x: float(np.float32(x))
FREQDEL = f32(0.02)
NU = np.array([W.NU1, W.NU2, W.NU3])


def _numpy_width(alpha):
    shape = [(1 - (NU[1] / NU[0]) ** (1 - alpha[0])) / (alpha[0] - 1),
             (1 - (NU[2] / NU[1]) ** (1 - alpha[1])) / (alpha[1] - 1), 1 / (alpha[2] - 1)]
    return np.array([shape[g] * NU[g] * W.EV_TO_HZ for g in range(3)])


def _numpy_dust_band_integral(alpha, a_dust, nfreq=400, freqdel=FREQDEL):
    """sum over the in-band bins of (e/nu_g)^-alpha_g sigma_d(e) de, de in Hz: vectorised bins, the fit of
    dustModule.f90:36-50"""
    e = 10.0 ** (np.arange(nfreq) * freqdel)
    lam_um = f32(2.99792458e10) / (e * W.EV_TO_HZ) * f32(1e8) / f32(1e4)
    a = np.asarray(a_dust, dtype=np.float64)
    fit = sum(a[t, 1] / ((lam_um / a[t, 0]) ** a[t, 3] + (lam_um / a[t, 0]) ** (-a[t, 4]) + a[t, 2]) for t in range(7))
    sD = f32(1.1) * fit * f32(0.9210340372) * f32(1e-22)
    out = np.zeros(3)
    i = np.arange(1, nfreq)
    f = e[i]
    for g in range(3):
        band = (f >= NU[g]) & (f <= NU[g + 1]) if g < 2 else f >= NU[2]
        out[g] = np.sum(((f / NU[g]) ** (-alpha[g]) * (e[i] - e[i - 1]) * W.EV_TO_HZ * sD[i])[band])
    return out


def test_band_width_against_numpy(uvbg):
    gamma, width = W.uvb_heating(uvbg["table"], uvbg["alpha"])
    want = _numpy_width(uvbg["alpha"])
    err = float(np.max(np.abs(width - want) / want))
    print(f"band widths {width} Hz, rel err {err:.2e}")
    assert np.all(width > 0) and err <= 1e-13, err
    assert np.array_equal(gamma, np.asarray(uvbg["table"])[:, 16:19])


def test_dust_band_integral_against_numpy(uvbg):
    a_dust = W.synthetic_spectra()["a_dust"]
    _, width = W.uvb_heating(uvbg["table"], uvbg["alpha"])
    got = W.uvb_dust_beta(uvbg["alpha"], a_dust) * width
    want = _numpy_dust_band_integral(uvbg["alpha"], a_dust)
    err = float(np.max(np.abs(got - want) / want))
    print(f"betaDust * W {got} cm^2 Hz per H, rel err {err:.2e}")
    assert np.all(got > 0) and err <= 1e-13, err


def test_band_width_argument_checks(uvbg):
    L = _lib.lib()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    al, out = np.ascontiguousarray(uvbg["alpha"]), np.zeros(3)
    assert L.rtb200_uvb_band_width(p(al), p(out)) == 0 and np.all(out > 0)
    assert L.rtb200_uvb_band_width(None, p(out)) == 12    # RTB200_ERR_ARG
    assert L.rtb200_uvb_band_width(p(al), None) == 12
    assert L.rtb200_last_heating(None, p(out)) == 12
    assert L.rtb200_grid_set_heating(None, None, None) == 12


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_numpy_pass_is_the_scalar_formula(mode):
    g = W.uniform_grid(5, seed=13)
    N = g["level"].size
    g["abun2"] = np.random.default_rng(4).uniform(1e-3, 0.05, N)
    rng = np.random.default_rng(mode)
    J = 10.0 ** rng.uniform(-24.0, -20.0, (3, N))
    gamma = 10.0 ** rng.uniform(-30.0, -26.0, (3, 3))
    width = np.array([2.1e15, 4.4e15, 1.9e16])
    bd, albedo = [2.1e-21, 7.3e-22, 3.3e-22], (0.3, 0.0, 0.7)
    H = heating_oracle.heating(J, g, gamma, width, mode, bd, albedo)
    four_pi = 4.0 * f32(3.141592654)
    for i in range(0, N, 3):
        t = [four_pi * float(J[k, i]) for k in range(3)]
        G = [((t[0] * gamma[0][s]) + (t[1] * gamma[1][s])) + (t[2] * gamma[2][s]) for s in range(3)]
        gas = ((float(g["HI"][i]) * G[0]) + (float(g["HeI"][i]) * G[1])) + (float(g["HeII"][i]) * G[2])
        dust = 0.0
        if mode:
            col = float(g["HI"][i]) if mode == 1 else (f32(0.76) * float(g["rho"][i])) / f32(1.6726231e-24)
            u = [((1.0 - albedo[k]) * (((col * bd[k]) * float(g["abun2"][i])) / f32(0.2))) * (t[k] * width[k])
                 for k in range(3)]
            dust = (u[0] + u[1]) + u[2]
        assert [H[f, i] for f in range(5)] == G + [gas, dust], i
    if mode == 0:
        assert np.array_equal(H[4], np.zeros(N))
