"""TEST INFRASTRUCTURE ONLY -- the accelerated source iteration of DESIGN.md 4.9 restated in numpy over oracle sweeps.

x_{k-1} forms the source of sweep k (eta_k = eta_th + sigma * x_{k-1}), y_k = F(x_{k-1}) is what the sweep returns, the
residual is r_k = maxrel(y_k, x_{k-1}) and the call stops after the first k with r_k <= tol (tol > 0) or at max_iter,
returning y_k.  x_0 is the warm start (or 0).  With ng, after every fourth sweep counted from the start or from the last
attempted extrapolation, and never on the sweep that stops the call, Ng's order-2 step (Auer 1987) replaces x_k = y_k by
max(0, (1-a-b) y_k + a y_{k-1} + b y_{k-2}) when its 2x2 system is well conditioned.
"""
import os

import numpy as np

import scattering_oracle as S


def ng_coefficients(I0, I1, I2, I3):
    """(a, b) of Ng's order-2 step, or None when the step is skipped"""
    with np.errstate(divide="ignore", invalid="ignore"):
        w = np.where(I0 > 0, 1.0 / np.where(I0 > 0, I0, 1.0), 0.0)
    d0, d1, d2 = (I0 - I1) * w, (I1 - I2) * w, (I2 - I3) * w
    q1, q2 = d0 - d1, d0 - d2
    A11, A12, A22 = (q1 * q1).sum(), (q1 * q2).sum(), (q2 * q2).sum()
    c1, c2 = (d0 * q1).sum(), (d0 * q2).sum()
    det = A11 * A22 - A12 * A12
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        a = (c1 * A22 - c2 * A12) / det
        b = (c2 * A11 - c1 * A12) / det
    if not (det > 1e-14 * A11 * A22 and np.isfinite(a) and np.isfinite(b)):
        return None
    return a, b


def solve_accelerated(og, uvb, beta, eta_th, sigma, max_iter, tol, ng=True, x0=None, kext=None, rays=None,
                      nthreads=None, n_angular_level=3):
    """Accelerated source iteration on a ScatteringOracleGrid `og`.  sigma [3, nleaf] is the scattering source; kext
    (default sigma) is what joins the extinction (dust: kd, with sigma = albedo * kd).  x0 [3, nleaf] is the warm start
    (None: 0).  Returns dict(J, iterations, residual, history, extrapolations, nseg, status)."""
    N = og.nleaf
    sigma = np.ascontiguousarray(sigma, dtype=np.float64).reshape(3, N)
    kext = sigma if kext is None else np.ascontiguousarray(kext, dtype=np.float64).reshape(3, N)
    eta_th = np.zeros((3, N)) if eta_th is None else np.ascontiguousarray(eta_th, dtype=np.float64).reshape(3, N)
    if rays is None:
        rays = np.arange(12 << (2 * (n_angular_level - 1)), dtype=np.int32)
    nthreads = nthreads or min(16, os.cpu_count() or 1)
    og.set_scattering(kext)
    x = np.zeros((3, N)) if x0 is None else np.array(x0, dtype=np.float64).reshape(3, N)
    cycle, hist, nseg, nng = [], [], 0, 0
    y, r, k = None, np.nan, 0
    for k in range(1, int(max_iter) + 1):
        og.set_emission(eta_th + sigma * x)   # numpy float64: one rounding each, no FMA
        o = og.diffuse_mt(uvb, beta, rays, n_angular_level=n_angular_level, nthreads=nthreads)
        if o["status"]:
            return dict(J=o["J"], iterations=k, residual=np.nan, history=hist, extrapolations=nng, nseg=nseg,
                        status=o["status"])
        y = o["J"]
        nseg += o["nseg"]
        r = S.residual(y, x)
        hist.append(r)
        if tol > 0 and r <= tol:
            break
        cycle.append(y)
        x = y
        if ng and len(cycle) == 4 and k < max_iter:
            ab = ng_coefficients(cycle[3], cycle[2], cycle[1], cycle[0])
            if ab is not None:
                a, b = ab
                x = np.maximum(0.0, (1.0 - a - b) * cycle[3] + a * cycle[2] + b * cycle[1])
                nng += 1
            cycle = []
    return dict(J=y, iterations=k, residual=r, history=hist, extrapolations=nng, nseg=nseg, status=0)
