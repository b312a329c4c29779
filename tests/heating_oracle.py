"""TEST INFRASTRUCTURE ONLY -- the heating pass (DESIGN.md 4.10) restated in numpy float64.

Every numpy operation below is one rounded IEEE operation (no FMA), in the order the definition writes, so that it
reproduces the device's fields bit for bit from the same J and species.  The dust opacity is dust_oracle.dust_kd, the
numpy restatement of the opacity the sweep uses.
"""
import numpy as np

import dust_oracle

FOUR_PI = 4.0 * float(np.float32(3.141592654))   # 4 * kPi of the library


def heating(J, g, gamma, width, mode=0, beta_dust=None, albedo=(0.0, 0.0, 0.0)):
    """[5, n] = Gamma_HI, Gamma_HeI, Gamma_HeII, H_gas, H_dust of J [3, n] and the grid dict g (HI, HeI, HeII, rho,
    abun2 of the same n leaves); gamma [3, 3] = [group][gammaHI, gammaHeI, gammaHeII], width[3] in Hz; mode / beta_dust /
    albedo as Transport.set_dust"""
    J = np.asarray(J, dtype=np.float64).reshape(3, -1)
    gam = np.asarray(gamma, dtype=np.float64).reshape(3, 3)
    w = np.asarray(width, dtype=np.float64).reshape(3)
    t = FOUR_PI * J
    G = [((t[0] * gam[0, s]) + (t[1] * gam[1, s])) + (t[2] * gam[2, s]) for s in range(3)]
    HI, HeI, HeII = (np.asarray(g[k], dtype=np.float64) for k in ("HI", "HeI", "HeII"))
    gas = ((HI * G[0]) + (HeI * G[1])) + (HeII * G[2])
    dust = np.zeros(J.shape[1])
    if mode:
        kd = dust_oracle.dust_kd(dict(g, level=HI), beta_dust, mode)
        u = [((1.0 - float(albedo[k])) * kd[k]) * (t[k] * w[k]) for k in range(3)]
        dust = (u[0] + u[1]) + u[2]
    return np.array([G[0], G[1], G[2], gas, dust])


def fields(d):
    """the [5, n] array of a Transport.last_heating() dict"""
    return np.array([d["gamma_HI"], d["gamma_HeI"], d["gamma_HeII"], d["gas"], d["dust"]])
