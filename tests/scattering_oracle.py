"""TEST INFRASTRUCTURE ONLY -- the CPU oracle with the scattering extension of DESIGN.md 4.7 applied.

On top of the emission oracle (tests/emission_oracle.py, whose EDITS this module reuses on a private copy) four edits
give every zone a scattering coefficient that joins the extinction, kappa_ext = kappa_abs + sigma, added last in the
order of the sweep's opacities.  The source iteration itself runs here in numpy over oracle sweeps:
    eta_k = eta_th + sigma * J_{k-1}   (two roundings, no FMA: numpy float64),  J_0 = 0,
    r_k   = max |J_k - J_{k-1}| / J_k  (0 where equal, +inf where J_k == 0 != J_{k-1}).
Each edit must match exactly once, so a change of the oracle shows up here as an error.

Edits (after the emission edits):
  * Zone gets ksca[3].
  * computeOpacities adds + z.ksca[g] to each kappa line.
  * diffuseSolveThreaded refreshes ksca in its per-thread octree copies.
  * ftte_grid_set_scattering(h, sigma[3][nleaf]) (NULL clears).
"""
import copy
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

import emission_oracle as EO
from oracle import ftte_oracle

EDITS = copy.deepcopy(EO.EDITS)
EDITS["ftte_common.h"].append((
    "  double eta[3];          // emission coefficient per group, uvb units per cm (0 = the reference)\n",
    "  double eta[3];          // emission coefficient per group, uvb units per cm (0 = the reference)\n"
    "  double ksca[3];         // scattering coefficient per group, 1/cm (0 = the reference)\n",
))
EDITS["ftte_diffuse.cpp"] += [
    ("      z.kappa[0] = z.HI * beta[0];\n", "      z.kappa[0] = z.HI * beta[0] + z.ksca[0];\n"),
    ("      z.kappa[1] = z.HI * beta[3] + z.HeI * beta[4];\n",
     "      z.kappa[1] = z.HI * beta[3] + z.HeI * beta[4] + z.ksca[1];\n"),
    ("      z.kappa[2] = z.HI * beta[6] + z.HeI * beta[7] + z.HeII * beta[8];\n",
     "      z.kappa[2] = z.HI * beta[6] + z.HeI * beta[7] + z.HeII * beta[8] + z.ksca[2];\n"),
    ("      for (int gI = 0; gI < 3; gI++) c.node[i].eta[gI] = g.node[i].eta[gI];\n",
     "      for (int gI = 0; gI < 3; gI++) c.node[i].eta[gI] = g.node[i].eta[gI];\n"
     "      for (int gI = 0; gI < 3; gI++) c.node[i].ksca[gI] = g.node[i].ksca[gI];\n"),
]
EDITS["ftte_capi.cpp"].append((
    "// Diffuse solve over directions",
    """int ftte_grid_set_scattering(void* h, const double* sigma) {
  Grid& g = *(Grid*)h;
  const size_t n = g.leafNode.size();
  for (size_t l = 0; l < n; l++) {
    Zone& z = g.node[g.leafNode[l]];
    for (int gI = 0; gI < 3; gI++) z.ksca[gI] = sigma ? sigma[gI * n + l] : 0.;
  }
  return OK;
}

// Diffuse solve over directions""",
))

_LIB = None


def _patched_sources():
    files = {}
    for f in sorted(os.listdir(EO.ORACLE)):
        if f.endswith((".cpp", ".h")):
            with open(os.path.join(EO.ORACLE, f)) as fh:
                files[f] = fh.read()
    for f, edits in EDITS.items():
        for old, new in edits:
            n = files[f].count(old)
            if n != 1:
                raise RuntimeError(f"scattering oracle: edit of oracle/{f} matches {n} times (the oracle changed?)")
            files[f] = files[f].replace(old, new)
    return files


def build():
    """compiles the patched oracle into a private temporary directory (keyed by the sources) and returns the library"""
    files = _patched_sources()
    key = hashlib.sha256("".join(f + files[f] for f in sorted(files)).encode()).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"rtb200-scattering-oracle-{os.getuid()}-{key}")
    so = os.path.join(out, "libftte_scattering.so")
    if os.path.exists(so):
        return so
    work = tempfile.mkdtemp(prefix="rtb200-scattering-oracle-")
    try:
        for f, text in files.items():
            with open(os.path.join(work, f), "w") as fh:
                fh.write(text)
        tmp_so = os.path.join(work, "libftte_scattering.so")
        subprocess.check_call([os.environ.get("CXX", "g++")] + EO.CXXFLAGS + ["-I", EO.ORACLE, "-shared", "-o", tmp_so]
                              + [os.path.join(work, s) for s in EO.SOURCES] + ["-lm", "-lpthread"])
        os.makedirs(out, exist_ok=True)
        os.replace(tmp_so, so)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        ref = ftte_oracle.lib()
        for name in ("ftte_grid_create", "ftte_grid_destroy", "ftte_grid_set_species", "ftte_diffuse", "ftte_diffuse_mt"):
            fn, r = getattr(L, name), getattr(ref, name)
            fn.restype, fn.argtypes = r.restype, r.argtypes
        for name in ("ftte_grid_set_emission", "ftte_grid_set_scattering"):
            getattr(L, name).restype = C.c_int
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


def residual(J, Jprev):
    """r = max over (group, leaf) of |J - Jprev| / J; 0 where equal, +inf where J == 0 != Jprev"""
    eq = J == Jprev
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(eq, 0.0, np.where(J == 0.0, np.inf, np.abs(J - Jprev) / J))
    return float(r.max())


class ScatteringOracleGrid(EO.EmissionOracleGrid):
    """EmissionOracleGrid on the scattering-patched oracle, with set_scattering(sigma [3, nleaf] or None) and solve()"""

    def __init__(self, *a, **k):
        # the constructor of EmissionOracleGrid, on the scattering library
        self.L = lib()
        nx, level, HI = a[0], a[1], a[2]
        HeI, HeII = k.get("HeI"), k.get("HeII")
        self.nx = int(nx)
        self.level = np.ascontiguousarray(level, dtype=np.int8)
        self.nleaf = int(self.level.size)
        arrs = [ftte_oracle._f64(x) for x in (HI, HeI, HeII, k.get("rho"), k.get("abun2"))]
        st = C.c_int(0)
        self.h = self.L.ftte_grid_create(self.nx, self.nleaf, ftte_oracle._p(self.level),
                                         *[ftte_oracle._p(x) for x in arrs], float(k.get("box_size", 1.0)), C.byref(st))
        if not self.h:
            raise RuntimeError(f"ftte_grid_create failed: status {st.value}")

    def set_scattering(self, sigma):
        s = None if sigma is None else np.ascontiguousarray(sigma, dtype=np.float64).reshape(3, self.nleaf)
        self._sigma = s
        self.L.ftte_grid_set_scattering(self.h, ftte_oracle._p(s))

    def solve(self, uvb, beta, eta_th, sigma, max_iter, tol, rays=None, nthreads=None, n_angular_level=3):
        """Source iteration (DESIGN.md 4.7) over oracle sweeps: returns dict(J, iterations, residual, nseg, status,
        history=[r_1, r_2, ...])."""
        N = self.nleaf
        sigma = np.ascontiguousarray(sigma, dtype=np.float64).reshape(3, N)
        eta_th = np.zeros((3, N)) if eta_th is None else np.ascontiguousarray(eta_th, dtype=np.float64).reshape(3, N)
        if rays is None:
            rays = np.arange(12 << (2 * (n_angular_level - 1)), dtype=np.int32)
        nthreads = nthreads or min(16, os.cpu_count() or 1)
        self.set_scattering(sigma)
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
            r = residual(J, Jprev)
            hist.append(r)
            eta = eta_th + sigma * J   # numpy float64: one rounding each, no FMA
            Jprev = J
            if tol > 0 and r <= tol:
                break
        return dict(J=J, iterations=k, residual=r, nseg=nseg, status=0, history=hist)


def grid(g):
    """ScatteringOracleGrid of a workloads.* grid dict"""
    return ScatteringOracleGrid(g["nx"], g["level"], g["HI"], HeI=g["HeI"], HeII=g["HeII"], box_size=g["box_size"])
