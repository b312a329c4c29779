"""Host-side mirror of the reference's hot-path call sites, on top of the C-ABI (include/rtb200.h).

The reference has no operator API: `program pointTransfer` runs, once per outer iteration,
    setZeroRates -> [point sources] -> computeOpacities + 192-direction diffuse sweep -> solveRateEquations
(equiSources.f90:1246-1831).  `Transport` keeps that shape: a grid in the reference's flattened leaf order goes in,
`diffuse()` returns Jmean1..3 per leaf exactly where the Fortran loop would have left them in `zoneType`.
"""
import ctypes as C

import numpy as np

from . import _lib

MATH_FAST, MATH_FAITHFUL = 0, 1


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def direction(n_angular_level, iray):
    """(izone, phi, theta) of one HEALPix direction -- equiSources.f90:1391-1454."""
    iz, phi, th = C.c_int32(0), C.c_double(0), C.c_double(0)
    st = _lib.lib().rtb200_direction(int(n_angular_level), int(iray), C.byref(iz), C.byref(phi), C.byref(th))
    _lib.check(st, "rtb200_direction")
    return iz.value, phi.value, th.value


def patterns(n_angular_level, iray, nx):
    out = np.zeros((nx, 12))
    _lib.check(_lib.lib().rtb200_patterns(int(n_angular_level), int(iray), int(nx), _ptr(out)), "rtb200_patterns")
    return out


def comm_unique_id():
    """128-byte id that joins the ranks of a one-process-per-GPU device group (rank 0 creates it, the launcher
    broadcasts it: e.g. torch.distributed.broadcast_object_list)"""
    _preload_nccl()
    buf = C.create_string_buffer(128)
    _lib.check(_lib.lib().rtb200_comm_unique_id(buf), "rtb200_comm_unique_id")
    return buf.raw


def _preload_nccl():
    """point the library's dlopen at the NCCL of the nvidia-nccl-cu12 wheel when no other one is configured"""
    import os
    if os.environ.get("RTB200_NCCL_LIB"):
        return
    try:
        import nvidia.nccl as _n
        for base in _n.__path__:
            p = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(p):
                os.environ["RTB200_NCCL_LIB"] = p
                return
    except Exception:
        pass


class Transport:
    """The transport engine behind one C-ABI handle:
        Transport(device=d)                      one GPU
        Transport(devices=[0, 1, ...])           one process driving several GPUs (rtb200_create_multi)
        Transport(device=d, comm=(nranks, rank, unique_id))   one process per GPU (rtb200_create_rank)
    Device groups accept the same set_grid / update_species / diffuse / point calls; the library shards the directions
    and sources and leaves / returns per-leaf results slab-wise (see include/rtb200.h)."""

    def __init__(self, device=0, math=MATH_FAST, devices=None, comm=None):
        self.L = _lib.lib()
        h = C.c_void_p()
        self.multi = devices is not None or comm is not None
        if devices is not None:
            _preload_nccl()
            d = np.ascontiguousarray(devices, dtype=np.int32)
            _lib.check(self.L.rtb200_create_multi(int(d.size), _ptr(d), C.byref(h)), "rtb200_create_multi")
        elif comm is not None:
            _preload_nccl()
            nranks, rank, uid = comm
            _lib.check(self.L.rtb200_create_rank(int(device), int(nranks), int(rank), uid, C.byref(h)),
                       "rtb200_create_rank")
        else:
            _lib.check(self.L.rtb200_create(int(device), C.byref(h)), "rtb200_create")
        self.h = h
        self.nleaf = 0
        self.nx = 0
        self.set_math(math)

    # ---- device groups -------------------------------------------------------------------------------------------
    def info(self):
        """dict(nranks, nlocal, first_rank, slab, reduce_mode): reduce_mode 1 = peer-memory kernel, 0 = NCCL, -1 = one GPU"""
        a, b, c, e = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
        d = C.c_int64(0)
        _lib.check(self.L.rtb200_multi_info(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e)),
                   "rtb200_multi_info")
        return dict(nranks=a.value, nlocal=b.value, first_rank=c.value, slab=d.value, reduce_mode=e.value)

    def shard(self, rank, n_angular_level=3):
        """HEALPix pixel numbers of the directions rank `rank` sweeps"""
        n = C.c_int32(0)
        cap = 12 * 4 ** (n_angular_level - 1)
        r = np.zeros(cap, dtype=np.int32)
        _lib.check(self.L.rtb200_multi_shard(self.h, int(n_angular_level), int(rank), _ptr(r), cap, C.byref(n)),
                   "rtb200_multi_shard")
        return r[:n.value].copy()

    def slab(self, local=0):
        """(offset, count, J_ptr, K_ptr, R_ptr) of local device `local`: device pointers to [3][slab], [3][slab], [6][slab]"""
        off, cnt = C.c_int64(0), C.c_int64(0)
        J, K, R = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _lib.check(self.L.rtb200_multi_slab(self.h, int(local), C.byref(off), C.byref(cnt), C.byref(J), C.byref(K),
                                            C.byref(R)), "rtb200_multi_slab")
        return off.value, cnt.value, J.value, K.value, R.value

    @staticmethod
    def _streams(streams):
        if streams is None:
            return None, None
        arr = (C.c_void_p * len(streams))(*[C.c_void_p(int(x)) for x in streams])
        return arr, arr

    def diffuse_resident(self, uvb, beta, ksi=None, chemistry=False, n_angular_level=3, streams=None):
        """resident step of a device group (asynchronous): sweep + reduce-scatter [+ photo-rates] [+ chemistry on the
        slab + all-gather]; returns this process's segment updates"""
        uvb, beta = _f64(uvb), _f64(np.asarray(beta).reshape(9))
        k = None if ksi is None else _f64(np.concatenate([np.ravel(x) for x in ksi]) if not isinstance(ksi, np.ndarray) else ksi)
        nseg = C.c_int64(0)
        keep, sp = self._streams(streams)
        st = self.L.rtb200_multi_diffuse_resident(self.h, int(n_angular_level), _ptr(uvb), _ptr(beta), _ptr(k),
                                                  int(bool(chemistry)), sp, C.byref(nseg))
        _lib.check(st, "rtb200_multi_diffuse_resident")
        return nseg.value

    def point_resident(self, spectra, src_leaf, src_weight, dust_approximation=0, max_pixel_level=6, streams=None,
                       diagnostics=False):
        keep, sa = self._spectra_args(spectra)
        leaf = np.ascontiguousarray(src_leaf, dtype=np.int32); wt = np.ascontiguousarray(src_weight, dtype=np.int32)
        ns = int(leaf.size)
        nseg = C.c_int64(0)
        rem = bnd = dust = spec = hpl = None
        if diagnostics:
            rem = np.zeros((ns, 7)); bnd = np.zeros((ns, 7)); dust = np.zeros(ns); spec = np.zeros((ns, 300))
            hpl = np.zeros(ns, dtype=np.int32)
        keeps, sp = self._streams(streams)
        st = self.L.rtb200_multi_point_resident(self.h, *sa, int(dust_approximation), int(max_pixel_level), ns, _ptr(leaf),
                                                _ptr(wt), sp, _ptr(rem), _ptr(bnd), _ptr(dust), _ptr(spec), _ptr(hpl),
                                                C.byref(nseg))
        _lib.check(st, "rtb200_multi_point_resident")
        if diagnostics:
            return nseg.value, dict(ndot_remaining=rem, ndot_boundary=bnd, ndot_dust=dust, ndot_spectrum=spec,
                                    highest_pixel_level=hpl)
        return nseg.value

    def sync(self):
        _lib.check(self.L.rtb200_multi_sync(self.h), "rtb200_multi_sync")

    def slab_get(self, local=0):
        """host copies (offset, count, J[3, count], K[3, count], R[6, count]) of a local device's slab results"""
        off, cnt, _, _, _ = self.slab(local)
        slab = self.info()["slab"]
        J, K, R = np.zeros((3, slab)), np.zeros((3, slab)), np.zeros((6, slab))
        _lib.check(self.L.rtb200_multi_slab_get(self.h, int(local), _ptr(J), _ptr(K), _ptr(R)), "rtb200_multi_slab_get")
        return off, cnt, J[:, :cnt].copy(), K[:, :cnt].copy(), R[:, :cnt].copy()

    def close(self):
        if getattr(self, "h", None):
            self.L.rtb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_math(self, mode):
        _lib.check(self.L.rtb200_set_math(self.h, int(mode)), "rtb200_set_math")

    def set_tuning(self, **kw):
        for k, v in kw.items():
            _lib.check(self.L.rtb200_set_tuning(self.h, k.encode(), float(v)), f"rtb200_set_tuning({k})")

    def set_grid(self, nx, level, HI, HeI=None, HeII=None, rho=None, abun2=None, box_size=1.0):
        level = np.ascontiguousarray(level, dtype=np.int8)
        arrs = [_f64(HI), _f64(HeI), _f64(HeII), _f64(rho), _f64(abun2)]
        for a in arrs:
            if a is not None and a.size != level.size:
                raise ValueError("per-leaf arrays must all have nleaf entries")
        st = self.L.rtb200_grid_set(self.h, int(nx), int(level.size), _ptr(level), *[_ptr(a) for a in arrs],
                                    float(box_size))
        _lib.check(st, "rtb200_grid_set")
        self.nleaf, self.nx = int(level.size), int(nx)

    def update_species(self, HI=None, HeI=None, HeII=None):
        a = [_f64(HI), _f64(HeI), _f64(HeII)]
        _lib.check(self.L.rtb200_grid_update_species(self.h, *[_ptr(x) for x in a]), "rtb200_grid_update_species")

    def set_emission(self, eta):
        """Emission coefficient per leaf and frequency group, [3, nleaf] in the units of uvb per cm (DESIGN.md 4.6);
        None clears it.  Negative, NaN or Inf entries raise and keep the previous emission."""
        if eta is None:
            _lib.check(self.L.rtb200_grid_set_emission(self.h, None), "rtb200_grid_set_emission")
            return
        e = np.ascontiguousarray(eta, dtype=np.float64)
        if e.size != 3 * self.nleaf:
            raise ValueError("eta must have 3 * nleaf entries ([3][nleaf])")
        _lib.check(self.L.rtb200_grid_set_emission(self.h, _ptr(e)), "rtb200_grid_set_emission")

    def set_emission_device(self, eta_ptr, stream=0):
        """The same from a device pointer to [3][nleaf] doubles (e.g. torch tensor .data_ptr()), copied and checked on
        `stream`; returns after synchronising it.  Single-GPU handles only."""
        st = self.L.rtb200_grid_set_emission_device(self.h, C.c_void_p(int(eta_ptr)), C.c_void_p(int(stream)))
        _lib.check(st, "rtb200_grid_set_emission_device")

    def set_scattering(self, sigma, max_iterations=100, tolerance=1e-9):
        """Isotropic scattering coefficient per leaf and frequency group, [3, nleaf] in 1/cm (DESIGN.md 4.7); None clears
        it.  The diffuse calls then solve by source iteration: at most `max_iterations` sweeps, stopping after the first
        whose largest relative change of J is <= `tolerance` (0: exactly `max_iterations` sweeps, no host round trip).
        Negative, NaN or Inf entries, a count < 1 or a negative tolerance raise and keep the previous state."""
        if sigma is None:
            _lib.check(self.L.rtb200_grid_set_scattering(self.h, None, 1, 0.0), "rtb200_grid_set_scattering")
            return
        s = np.ascontiguousarray(sigma, dtype=np.float64)
        if s.size != 3 * self.nleaf:
            raise ValueError("sigma must have 3 * nleaf entries ([3][nleaf])")
        st = self.L.rtb200_grid_set_scattering(self.h, _ptr(s), int(max_iterations), float(tolerance))
        _lib.check(st, "rtb200_grid_set_scattering")

    def set_dust(self, approximation, beta_dust=None, albedo=(0.0, 0.0, 0.0), max_iterations=100, tolerance=1e-9):
        """Dust in the diffuse sweep (DESIGN.md 4.8): `approximation` 1 (dust column from HI) or 2 (from rho) with the
        band-mean cross-sections `beta_dust[3]` of workloads.uvb_dust_beta, 0 clears it.  The opacity follows the current
        species in every diffuse call; an `albedo[3]` > 0 makes the dust scatter, solved by source iteration with
        `max_iterations` / `tolerance` as set_scattering.  Bad values, a missing rho / abun2, or scattering dust while a
        per-leaf sigma is set raise and keep the previous state."""
        bd = None if beta_dust is None else _f64(beta_dust)
        al = _f64(albedo)
        if (bd is not None and bd.size != 3) or al.size != 3:
            raise ValueError("beta_dust and albedo take one value per frequency group")
        st = self.L.rtb200_grid_set_dust(self.h, int(approximation), None if bd is None else _ptr(bd), _ptr(al),
                                         int(max_iterations), float(tolerance))
        _lib.check(st, "rtb200_grid_set_dust")

    def last_scattering(self):
        """Sweeps done and the last residual of the latest diffuse call: {"iterations", "residual"} (0 / 0 without
        scattering)."""
        it, r = C.c_int32(0), C.c_double(0)
        _lib.check(self.L.rtb200_last_scattering(self.h, C.byref(it), C.byref(r)), "rtb200_last_scattering")
        return {"iterations": it.value, "residual": r.value}

    def set_scattering_acceleration(self, ng=False, warm_start=False):
        """Acceleration of the source iteration of set_scattering / set_dust (DESIGN.md 4.9): `ng` extrapolates after
        every fourth sweep (Ng, order 2), `warm_start` starts from the J the previous completed solve returned instead
        of J = 0.  Both off is plain source iteration.  A device group sets it on every rank (collectively in rank mode).
        set_grid resets it."""
        flags = (1 if ng else 0) | (2 if warm_start else 0)
        _lib.check(self.L.rtb200_grid_set_scattering_acceleration(self.h, flags), "rtb200_grid_set_scattering_acceleration")

    def last_scattering_acceleration(self):
        """Of the latest diffuse call: {"extrapolations": Ng steps applied (skipped ones not counted), "warm_start": whether
        it started from the previous call's J}."""
        n, w = C.c_int32(0), C.c_int32(0)
        _lib.check(self.L.rtb200_last_scattering_acceleration(self.h, C.byref(n), C.byref(w)),
                   "rtb200_last_scattering_acceleration")
        return {"extrapolations": n.value, "warm_start": bool(w.value)}

    def set_heating(self, gamma, band_width=None):
        """Photo-heating and dust absorption per leaf (DESIGN.md 4.10): `gamma` [3, 3] = [group][gammaHI, gammaHeI,
        gammaHeII] and `band_width[3]` in Hz, as workloads.uvb_heating returns them; None clears the setting.  Every
        diffuse call then ends with one pass over the J it returns (read back with last_heating / heating_device).
        Negative, NaN or Inf entries raise and keep the previous state.  set_grid clears it."""
        if gamma is None:
            _lib.check(self.L.rtb200_grid_set_heating(self.h, None, None), "rtb200_grid_set_heating")
            return
        g, w = _f64(gamma), _f64(band_width)
        if g.size != 9 or w is None or w.size != 3:
            raise ValueError("gamma takes [3][3] values and band_width one per frequency group")
        _lib.check(self.L.rtb200_grid_set_heating(self.h, _ptr(g), _ptr(w)), "rtb200_grid_set_heating")

    def last_heating(self):
        """The heating fields of the latest diffuse call, each [nleaf]: {"gamma_HI", "gamma_HeI", "gamma_HeII"} in erg/s
        per absorber, {"gas", "dust"} in erg/s/cm^3 (a device group in rank mode fills its slab only, the rest is 0)."""
        H = np.zeros((5, self.nleaf))
        _lib.check(self.L.rtb200_last_heating(self.h, _ptr(H)), "rtb200_last_heating")
        return dict(gamma_HI=H[0], gamma_HeI=H[1], gamma_HeII=H[2], gas=H[3], dust=H[4])

    def heating_device(self, local=0):
        """(ptr, offset, count, stride): the library's device buffer [5][stride] of local device `local`, holding leaves
        [offset, offset + count); valid until the next diffuse call or setting change."""
        off, cnt, stride, H = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_void_p()
        _lib.check(self.L.rtb200_heating_device(self.h, int(local), C.byref(off), C.byref(cnt), C.byref(stride), C.byref(H)),
                   "rtb200_heating_device")
        return H.value, off.value, cnt.value, stride.value

    def diffuse(self, uvb, beta, n_angular_level=3, rays=None, out=None):
        """Host-buffer call (H2D of nothing but tables, D2H of J): returns (J[3, nleaf], nseg)."""
        uvb, beta = _f64(uvb), _f64(np.asarray(beta).reshape(9))
        J = out if out is not None else np.empty((3, self.nleaf))
        r = None if rays is None else np.ascontiguousarray(rays, dtype=np.int32)
        nseg = C.c_int64(0)
        st = self.L.rtb200_diffuse(self.h, int(n_angular_level), _ptr(uvb), _ptr(beta), _ptr(r),
                                   0 if r is None else int(r.size), _ptr(J[0]), _ptr(J[1]), _ptr(J[2]), C.byref(nseg))
        _lib.check(st, "rtb200_diffuse")
        return J, nseg.value

    def diffuse_device(self, uvb, beta, J_ptr, n_angular_level=3, rays=None, stream=0):
        """Resident call: J_ptr is a device pointer to [3][nleaf] doubles (e.g. torch tensor .data_ptr())."""
        uvb, beta = _f64(uvb), _f64(np.asarray(beta).reshape(9))
        r = None if rays is None else np.ascontiguousarray(rays, dtype=np.int32)
        nseg = C.c_int64(0)
        st = self.L.rtb200_diffuse_device(self.h, int(n_angular_level), _ptr(uvb), _ptr(beta), _ptr(r),
                                          0 if r is None else int(r.size), C.c_void_p(int(J_ptr)),
                                          C.c_void_p(int(stream)), C.byref(nseg))
        _lib.check(st, "rtb200_diffuse_device")
        return nseg.value

    def diffuse_rates_device(self, J_ptr, ksi24, ksi25, ksi26, k24_ptr, k25_ptr, k26_ptr, stream=0):
        a, b, c = _f64(ksi24), _f64(np.atleast_1d(ksi25)), _f64(ksi26)
        st = self.L.rtb200_diffuse_rates_device(self.h, C.c_void_p(int(J_ptr)), _ptr(a), _ptr(b), _ptr(c),
                                                C.c_void_p(int(k24_ptr)), C.c_void_p(int(k25_ptr)),
                                                C.c_void_p(int(k26_ptr)), C.c_void_p(int(stream)))
        _lib.check(st, "rtb200_diffuse_rates_device")

    # ---- point sources (equiSources.f90:1256-1370) ---------------------------------------------------------------
    @staticmethod
    def _spectra_args(spectra):
        wl = _f64(spectra["wavelength"]); lum = _f64(spectra["lum"]); met = _f64(spectra["metallicity"])
        ad = _f64(spectra["a_dust"])
        if lum.shape != (5, 2, wl.size) or met.size != 5 or ad.shape != (7, 5):
            raise ValueError("spectra: lum[5,2,nWave], metallicity[5], a_dust[7,5] expected")
        keep = (wl, lum, met, ad)
        return keep, [int(wl.size), _ptr(wl), _ptr(lum), _ptr(met), float(spectra["coef_spectrum"]), _ptr(ad)]

    def point(self, spectra, src_leaf, src_weight, dust_approximation=0, max_pixel_level=6, rates=None,
              trace_cap=0, inplace=False):
        """Host-buffer call.  `rates` [6, nleaf] (krate24, krate25, krate26, crate24, crate25, crate26) is accumulated
        like the reference's cell fields (zeros when None; `inplace=True` accumulates into the caller's C-contiguous
        fp64 array itself, e.g. a view of pinned memory, instead of a copy).  Returns dict(rates, ndot_remaining[nsrc,7],
        ndot_boundary[nsrc,7], ndot_dust[nsrc], ndot_spectrum[nsrc,300], highest_pixel_level[nsrc], nseg[, trace,
        trace_key])."""
        keep, sa = self._spectra_args(spectra)
        leaf = np.ascontiguousarray(src_leaf, dtype=np.int32); wt = np.ascontiguousarray(src_weight, dtype=np.int32)
        if leaf.size != wt.size:
            raise ValueError("src_leaf and src_weight differ in length")
        ns = int(leaf.size)
        if rates is None:
            R = np.zeros((6, self.nleaf))
        elif inplace:
            R = rates
            if not (isinstance(R, np.ndarray) and R.dtype == np.float64 and R.flags.c_contiguous
                    and R.shape == (6, self.nleaf)):
                raise ValueError("inplace rates must be a C-contiguous float64 array of shape (6, nleaf)")
        else:
            R = np.ascontiguousarray(rates, dtype=np.float64).copy()
        nseg = C.c_int64(0)
        out = dict(rates=R)
        if trace_cap:
            tr = np.zeros((int(trace_cap), 2), dtype=np.int64)
            tl = C.c_int64(0)
            st = self.L.rtb200_point_trace(self.h, *sa, int(dust_approximation), int(max_pixel_level), ns, _ptr(leaf),
                                           _ptr(wt), _ptr(R), C.byref(nseg), _ptr(tr), int(trace_cap), C.byref(tl))
            _lib.check(st, "rtb200_point_trace")
            if tl.value > trace_cap:
                raise RuntimeError(f"trace buffer too small: {tl.value} segments")
            tr = tr[:tl.value]
            order = np.argsort(tr[:, 1], kind="stable")
            out.update(trace=tr[order, 0].copy(), trace_key=tr[order, 1].copy())
        else:
            rem = np.zeros((ns, 7)); bnd = np.zeros((ns, 7)); dust = np.zeros(ns); spec = np.zeros((ns, 300))
            hpl = np.zeros(ns, dtype=np.int32)
            st = self.L.rtb200_point(self.h, *sa, int(dust_approximation), int(max_pixel_level), ns, _ptr(leaf),
                                     _ptr(wt), *[_ptr(R[i]) for i in range(6)], _ptr(rem), _ptr(bnd), _ptr(dust),
                                     _ptr(spec), _ptr(hpl), C.byref(nseg))
            _lib.check(st, "rtb200_point")
            out.update(ndot_remaining=rem, ndot_boundary=bnd, ndot_dust=dust, ndot_spectrum=spec,
                       highest_pixel_level=hpl)
        out["nseg"] = nseg.value
        return out

    def point_device(self, spectra, src_leaf, src_weight, rates_ptr, dust_approximation=0, max_pixel_level=6,
                     stream=0, diagnostics=False):
        """Resident call: rates_ptr = device pointer to [6][nleaf] doubles, accumulated.  Returns nseg (and the
        per-source diagnostics when asked)."""
        keep, sa = self._spectra_args(spectra)
        leaf = np.ascontiguousarray(src_leaf, dtype=np.int32); wt = np.ascontiguousarray(src_weight, dtype=np.int32)
        ns = int(leaf.size)
        nseg = C.c_int64(0)
        rem = bnd = dust = spec = hpl = None
        if diagnostics:
            rem = np.zeros((ns, 7)); bnd = np.zeros((ns, 7)); dust = np.zeros(ns); spec = np.zeros((ns, 300))
            hpl = np.zeros(ns, dtype=np.int32)
        st = self.L.rtb200_point_device(self.h, *sa, int(dust_approximation), int(max_pixel_level), ns, _ptr(leaf),
                                        _ptr(wt), C.c_void_p(int(rates_ptr)), C.c_void_p(int(stream)), _ptr(rem),
                                        _ptr(bnd), _ptr(dust), _ptr(spec), _ptr(hpl), C.byref(nseg))
        _lib.check(st, "rtb200_point_device")
        if diagnostics:
            return nseg.value, dict(ndot_remaining=rem, ndot_boundary=bnd, ndot_dust=dust, ndot_spectrum=spec,
                                    highest_pixel_level=hpl)
        return nseg.value

    def point_tables(self, spectra, i_metal, coef_metal):
        """the six (0:10)^4 tables of stellarBetaTable.f90 for one metallicity bracket: [6, 11^4]"""
        keep, sa = self._spectra_args(spectra)
        out = np.zeros((6, 11 ** 4))
        _lib.check(self.L.rtb200_point_tables(self.h, *sa, int(i_metal), float(coef_metal), _ptr(out)),
                   "rtb200_point_tables")
        return out

    # ---- chemistry (solveRateEquations, equiSources.f90:3459-3677) --------------------------------------------------
    def set_rate_tables(self, ktab):
        """ktab = dict(k[6, nratec] = k1a..k6a, logtem0, logtem9, dlogtem)"""
        k = _f64(ktab["k"])
        if k.ndim != 2 or k.shape[0] != 6:
            raise ValueError("k must have shape (6, nratec)")
        st = self.L.rtb200_chemistry_tables(self.h, int(k.shape[1]), float(ktab["logtem0"]), float(ktab["logtem9"]),
                                            float(ktab["dlogtem"]), *[_ptr(k[i]) for i in range(6)])
        _lib.check(st, "rtb200_chemistry_tables")

    def set_temperature(self, tgas):
        t = _f64(tgas)
        if t.size != self.nleaf:
            raise ValueError("tgas needs one value per leaf")
        _lib.check(self.L.rtb200_chemistry_temperature(self.h, _ptr(t)), "rtb200_chemistry_temperature")

    def chemistry_device(self, rates_ptr=0, J_ptr=0, ksi=None, uniform=None, stream=0, want_change=True):
        """One solveRateEquations pass over all leaves, in place on the device copies of HI, HeI, HeII.  rates_ptr /
        J_ptr: device pointers ([6][nleaf] / [3][nleaf]) or 0; ksi = (ksi24[3], ksi25, ksi26[2]) flattened; uniform =
        (add24, add25, add26, selfShieldingThreshold).  Returns the largest change of a species fraction."""
        k = None if ksi is None else _f64(np.concatenate([np.ravel(x) for x in ksi]) if not isinstance(ksi, np.ndarray) else ksi)
        u = None if uniform is None else _f64(uniform)
        mc = C.c_double(0)
        st = self.L.rtb200_chemistry_device(self.h, C.c_void_p(int(rates_ptr)) if rates_ptr else None,
                                            C.c_void_p(int(J_ptr)) if J_ptr else None, _ptr(k), _ptr(u),
                                            C.byref(mc) if want_change else None, C.c_void_p(int(stream)))
        _lib.check(st, "rtb200_chemistry_device")
        return mc.value

    def get_species(self):
        HI, HeI, HeII = np.empty(self.nleaf), np.empty(self.nleaf), np.empty(self.nleaf)
        _lib.check(self.L.rtb200_grid_get_species(self.h, _ptr(HI), _ptr(HeI), _ptr(HeII)), "rtb200_grid_get_species")
        return HI, HeI, HeII

    def compute_mass(self, stream=0):
        """(neutralHydrogenMass, totalHydrogenMass) in solar masses from the device copies of HI and rho: computeMass,
        equiSources.f90:4369-4393 (the driver prints their ratio after every chemistry pass, :1828-1836)."""
        a, b = C.c_double(0), C.c_double(0)
        _lib.check(self.L.rtb200_compute_mass(self.h, C.byref(a), C.byref(b), C.c_void_p(int(stream))),
                   "rtb200_compute_mass")
        return a.value, b.value

    def device_error(self):
        return self.L.rtb200_device_error(self.h)

    def neighbours(self, n_angular_level, iray):
        nb = np.full((3, self.nleaf), -9, dtype=np.int32)
        _lib.check(self.L.rtb200_neighbours(self.h, int(n_angular_level), int(iray), _ptr(nb)), "rtb200_neighbours")
        return nb

    def last_stats(self):
        ms, sms, n, sn, b = C.c_double(0), C.c_double(0), C.c_int64(0), C.c_int64(0), C.c_double(0)
        _lib.check(self.L.rtb200_last_stats(self.h, C.byref(ms), C.byref(sms), C.byref(n), C.byref(sn), C.byref(b)),
                   "rtb200_last_stats")
        return dict(device_ms=ms.value, sweep_ms=sms.value, launches=n.value, sweep_launches=sn.value,
                    algorithmic_bytes=b.value)
