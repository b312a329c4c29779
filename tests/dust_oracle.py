"""TEST INFRASTRUCTURE ONLY -- dust in the diffuse sweep (DESIGN.md 4.8) on the oracle with scattering.

The dust opacity kd of a leaf is an extinction increment like the per-leaf sigma of tests/scattering_oracle.py, so the
oracle needs no edit of its own: kd goes into its `ksca` slot (added last to each kappa line, rounded once, as the
device adds it), and the source iteration runs in numpy with albedo * kd as the scattering source.  `dust_kd` restates
the definition operation for operation in numpy float64 (one rounding per operation, no FMA), so it reproduces the
device's kd bit for bit.
"""
import os

import numpy as np

import scattering_oracle

F02 = float(np.float32(0.2))
PSI = float(np.float32(0.76))
MH = float(np.float32(1.6726231e-24))


def dust_kd(g, beta_dust, mode):
    """kd[3, nleaf] in 1/cm: mode 1 ((HI * bd) * abun2) / 0.2f, mode 2 (((((0.76f * rho) / m_H) * bd) * abun2) / 0.2f"""
    N = g["level"].size
    if mode == 0:
        return np.zeros((3, N))
    col = np.asarray(g["HI"], dtype=np.float64) if mode == 1 else (PSI * np.asarray(g["rho"], dtype=np.float64)) / MH
    a = np.asarray(g["abun2"], dtype=np.float64)
    return np.array([((col * float(bd)) * a) / F02 for bd in beta_dust])


class DustOracleGrid(scattering_oracle.ScatteringOracleGrid):
    """ScatteringOracleGrid whose solve() takes the extinction increment and the scattering source separately"""

    def solve(self, uvb, beta, eta_th, kd, sigma_src, max_iter, tol, rays=None, nthreads=None, n_angular_level=3):
        """Source iteration with kappa = kappa_abs + kd and eta_k = eta_th + sigma_src * J_{k-1}: returns dict(J,
        iterations, residual, nseg, status, history).  sigma_src = 0 with max_iter = 1 is the absorbing sweep."""
        N = self.nleaf
        kd = np.ascontiguousarray(kd, dtype=np.float64).reshape(3, N)
        sigma_src = np.ascontiguousarray(sigma_src, dtype=np.float64).reshape(3, N)
        eta_th = np.zeros((3, N)) if eta_th is None else np.ascontiguousarray(eta_th, dtype=np.float64).reshape(3, N)
        if rays is None:
            rays = np.arange(12 << (2 * (n_angular_level - 1)), dtype=np.int32)
        nthreads = nthreads or min(16, os.cpu_count() or 1)
        self.set_scattering(kd)
        Jprev = np.zeros((3, N))
        eta = eta_th.copy()
        hist, nseg = [], 0
        for k in range(1, int(max_iter) + 1):
            self.set_emission(eta)
            o = self.diffuse_mt(uvb, beta, rays, n_angular_level=n_angular_level, nthreads=nthreads)
            if o["status"]:
                return dict(J=o["J"], iterations=k, residual=np.nan, nseg=nseg, status=o["status"], history=hist)
            J = o["J"]
            nseg += o["nseg"]
            r = scattering_oracle.residual(J, Jprev)
            hist.append(r)
            eta = eta_th + sigma_src * J   # numpy float64: one rounding each, no FMA
            Jprev = J
            if tol > 0 and r <= tol:
                break
        return dict(J=J, iterations=k, residual=r, nseg=nseg, status=0, history=hist)


def grid(g):
    """DustOracleGrid of a workloads.* grid dict"""
    return DustOracleGrid(g["nx"], g["level"], g["HI"], HeI=g["HeI"], HeII=g["HeII"], box_size=g["box_size"])

