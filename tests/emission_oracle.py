"""TEST INFRASTRUCTURE ONLY -- the CPU oracle with the emission extension of DESIGN.md 4.6 applied.

There is no reference value of J for an emitting segment, so the checker is the oracle itself (oracle/, a restatement of
the reference) with `nemi = eta * dpath` in its segment update and the exact segment path average as its mean intensity.
The oracle's sources are left as they are: this module copies them to a private directory, applies the edits below
(each must match exactly once, so a change of the oracle shows up here as an error, not as a silently different
checker), compiles them with the oracle's flags and loads the result beside the unmodified oracle.

Edits:
  * Zone gets eta[3] (zero-initialised like every other field: value-initialised nodes).
  * transportLeaf: Iout = Iin*tmpabs + nemi*tmpemi/dpath with nemi = eta*dpath (the reference's own slot), and
    J_seg = computeCellIntensity(Iin, Iin*tmpabs) + nemi*phi(tau), phi = (tau - 1 + e^-tau)/tau^2 (series below
    tau = 1e-2).  With eta = 0 every operation of the original is repeated and the added terms are exact zeros.
  * diffuseSolveThreaded refreshes eta in its per-thread octree copies.
  * ftte_grid_set_emission(h, eta[3][nleaf]) (NULL clears).
"""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ftte_oracle  # noqa: E402

CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math"]   # oracle/Makefile
SOURCES = ["ftte_diffuse.cpp", "ftte_point.cpp", "ftte_chem.cpp", "ftte_uvb.cpp", "ftte_capi.cpp"]

EDITS = {
    "ftte_common.h": [(
        "  double Jmean[3];\n",
        "  double Jmean[3];\n"
        "  double eta[3];          // emission coefficient per group, uvb units per cm (0 = the reference)\n",
    )],
    "ftte_diffuse.cpp": [(
        """    double dpath = cellSize * len;
    for (int gI = 0; gI < 3; gI++) {
      double tau = z.kappa[gI] * dpath;
      double tmpabs = std::exp(-tau);
      // nemi = 0: Iout = Iin*tmpabs + 0.*tmpemi/dpath (transportRoutinesModule.f90:673-678)
      double tmpemi = (tau > (double)1.e-10f) ? (1. - tmpabs) / z.kappa[gI] : dpath;
      z.Iout[ray][gI] = Iin[gI] * tmpabs + 0. * tmpemi / dpath;
    }
""",
        """    double dpath = cellSize * len;
    double Jseg[3];
    for (int gI = 0; gI < 3; gI++) {
      double tau = z.kappa[gI] * dpath;
      double tmpabs = std::exp(-tau);
      double tmpemi = (tau > (double)1.e-10f) ? (1. - tmpabs) / z.kappa[gI] : dpath;
      const double nemi = z.eta[gI] * dpath;
      const double Iatt = Iin[gI] * tmpabs;
      z.Iout[ray][gI] = Iatt + nemi * tmpemi / dpath;
      Jseg[gI] = 0.;
      computeCellIntensity(Jseg[gI], Iin[gI], Iatt);
      double phi;
      if (tau < 1e-2) phi = 0.5 + tau * (-1. / 6. + tau * (1. / 24. + tau * (-1. / 120. + tau * (1. / 720. + tau * (-1. / 5040. + tau / 40320.)))));
      else phi = (tau - (1. - tmpabs)) / (tau * tau);
      Jseg[gI] = Jseg[gI] + nemi * phi;
    }
""",
    ), (
        "    for (int gI = 0; gI < 3; gI++) computeCellIntensity(Jm[gI], Iin[gI], z.Iout[ray][gI]);\n",
        "    for (int gI = 0; gI < 3; gI++) Jm[gI] = Jm[gI] + Jseg[gI];\n",
    ), (
        "      c.node[i].HI = g.node[i].HI; c.node[i].HeI = g.node[i].HeI; c.node[i].HeII = g.node[i].HeII;\n",
        "      c.node[i].HI = g.node[i].HI; c.node[i].HeI = g.node[i].HeI; c.node[i].HeII = g.node[i].HeII;\n"
        "      for (int gI = 0; gI < 3; gI++) c.node[i].eta[gI] = g.node[i].eta[gI];\n",
    )],
    "ftte_capi.cpp": [(
        "// Diffuse solve over directions",
        """int ftte_grid_set_emission(void* h, const double* eta) {
  Grid& g = *(Grid*)h;
  const size_t n = g.leafNode.size();
  for (size_t l = 0; l < n; l++) {
    Zone& z = g.node[g.leafNode[l]];
    for (int gI = 0; gI < 3; gI++) z.eta[gI] = eta ? eta[gI * n + l] : 0.;
  }
  return OK;
}

// Diffuse solve over directions""",
    )],
}

_LIB = None


def _patched_sources():
    files = {}
    for f in sorted(os.listdir(ORACLE)):
        if f.endswith((".cpp", ".h")):
            with open(os.path.join(ORACLE, f)) as fh:
                files[f] = fh.read()
    for f, edits in EDITS.items():
        for old, new in edits:
            n = files[f].count(old)
            if n != 1:
                raise RuntimeError(f"emission oracle: edit of oracle/{f} matches {n} times (the oracle changed?)")
            files[f] = files[f].replace(old, new)
    return files


def build():
    """compiles the patched oracle into a private temporary directory (keyed by the sources) and returns the library"""
    files = _patched_sources()
    key = hashlib.sha256("".join(f + files[f] for f in sorted(files)).encode()).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"rtb200-emission-oracle-{os.getuid()}-{key}")
    so = os.path.join(out, "libftte_emission.so")
    if os.path.exists(so):
        return so
    work = tempfile.mkdtemp(prefix="rtb200-emission-oracle-")
    try:
        for f, text in files.items():
            with open(os.path.join(work, f), "w") as fh:
                fh.write(text)
        tmp_so = os.path.join(work, "libftte_emission.so")
        # -I oracle/: the quoted include of csrc/portable_math.h is relative to the oracle's own directory
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-I", ORACLE, "-shared", "-o", tmp_so]
                              + [os.path.join(work, s) for s in SOURCES] + ["-lm", "-lpthread"])
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
        L.ftte_grid_set_emission.restype = C.c_int
        L.ftte_grid_set_emission.argtypes = [C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


class EmissionOracleGrid(ftte_oracle.OracleGrid):
    """OracleGrid on the patched oracle, with set_emission(eta [3, nleaf] or None)"""

    def __init__(self, nx, level, HI, HeI=None, HeII=None, rho=None, abun2=None, box_size=1.0):
        self.L = lib()
        self.nx = int(nx)
        self.level = np.ascontiguousarray(level, dtype=np.int8)
        self.nleaf = int(self.level.size)
        arrs = [ftte_oracle._f64(a) for a in (HI, HeI, HeII, rho, abun2)]
        st = C.c_int(0)
        self.h = self.L.ftte_grid_create(self.nx, self.nleaf, ftte_oracle._p(self.level),
                                         *[ftte_oracle._p(a) for a in arrs], float(box_size), C.byref(st))
        if not self.h:
            raise RuntimeError(f"ftte_grid_create failed: status {st.value}")

    def set_emission(self, eta):
        e = None if eta is None else np.ascontiguousarray(eta, dtype=np.float64).reshape(3, self.nleaf)
        self._eta = e   # the library reads the array during the call only; kept for inspection
        self.L.ftte_grid_set_emission(self.h, ftte_oracle._p(e))


def grid(g):
    """EmissionOracleGrid of a workloads.* grid dict"""
    return EmissionOracleGrid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])
