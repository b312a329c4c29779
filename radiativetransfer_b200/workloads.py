"""Synthetic inputs of the shapes named in BASELINE.json (none of the reference's data files ship with it).

Grids are produced directly in the reference's flattened leaf order (`writeCell` pre-order,
equiSources.f90:4044-4079): base cells x outer / y / z inner, the 8 children of a refined cell x, y, z.
The UV-background amplitudes and group cross-sections come from the library's host-side restatement of the
reference set-up (rtb200_uvb_background; checked against the oracle and an independent numpy evaluation in
tests/test_uvb_tables.py).
"""
import numpy as np

# definitionsModule.f90:8-41 (single-precision literals widened)
_f = np.float32
PI = float(_f(3.141592654))
HP = float(_f(6.6260693e-27))
PC = float(_f(3.08568025e18))
KPC = 1.0e3 * PC
MP = float(_f(1.6726231e-24))
MN = float(_f(1.67492728e-24))
MHE = 2.0 * (MP + MN)
PSI = float(_f(0.76))
NU1, NU2, NU3 = float(_f(13.598)), float(_f(24.587)), float(_f(54.418))
EV_TO_ERG = 1.60217646e-12
EV_TO_HZ = EV_TO_ERG / HP


def _sigmas(nu):
    """HI, HeII, HeI photo-ionisation cross-sections (uvbBetaTable.f90:31-62)."""
    s24 = np.zeros_like(nu)
    s25 = np.zeros_like(nu)
    s26 = np.zeros_like(nu)
    m = nu > NU1
    d = np.sqrt(nu[m] / NU1 - 1)
    s24[m] = float(_f(6.3e-18)) * (NU1 / nu[m]) ** 4 * np.exp(4.0 - 4.0 * np.arctan(d) / d) / (1 - np.exp(-2.0 * PI / d))
    m = nu > NU3
    d = np.sqrt(nu[m] / NU3 - 1)
    s25[m] = float(_f(1.58e-18)) * (NU3 / nu[m]) ** 4 * np.exp(4.0 - 4.0 * np.arctan(d) / d) / (1 - np.exp(-2.0 * PI / d))
    m = nu > NU2
    s26[m] = float(_f(7.42e-18)) * (float(_f(1.66)) * (nu[m] / NU2) ** float(_f(-2.05)) - float(_f(0.66)) * (nu[m] / NU2) ** float(_f(-3.05)))
    return s24, s25, s26


def uvb_background(redshift=3.0, uvb_coefficient=1.0, nfreq=400, freqdel=None):
    """uvb[3], beta[3][3] = [group][beta24, beta26, beta25], ksi24[3], ksi25[1], ksi26[2], alpha[3], table[3][19] from the
    library's host-side restatement of the reference set-up (rtb200_uvb_background: equiSources.f90:198-246,
    :4985-5043, uvbBetaTable.f90:31-296).  nfreq / freqdel default to the reference's nfbins = 400 and
    frequencyBinWidth = 0.02 (a single-precision literal, definitionsModule.f90:239-241)."""
    import ctypes as C

    from . import _lib
    if freqdel is None:
        freqdel = float(_f(0.02))
    uvb, alpha, beta = np.zeros(3), np.zeros(3), np.zeros((3, 3))
    k24, k25, k26, tab = np.zeros(3), np.zeros(1), np.zeros(2), np.zeros((3, 19))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    st = _lib.lib().rtb200_uvb_background(float(redshift), float(uvb_coefficient), int(nfreq), float(freqdel), p(uvb),
                                          p(alpha), p(beta), p(k24), p(k25), p(k26), p(tab))
    _lib.check(st, "rtb200_uvb_background")
    return dict(uvb=uvb, beta=beta, alpha=alpha, ksi24=k24, ksi25=k25, ksi26=k26, table=tab)


def uvb_dust_beta(alpha, a_dust, nfreq=400, freqdel=None):
    """betaD[3]: band-mean dust cross-section of each frequency group [cm^2 per H] from the extinction fit a_dust[7, 5]
    with the weights of beta24 (rtb200_uvb_dust_beta, DESIGN.md 4.8), the input of Transport.set_dust.  alpha[3] are the
    background's effective slopes (uvb_background()["alpha"])."""
    import ctypes as C

    from . import _lib
    if freqdel is None:
        freqdel = float(_f(0.02))
    al = np.ascontiguousarray(alpha, dtype=np.float64).reshape(3)
    ad = np.ascontiguousarray(a_dust, dtype=np.float64).reshape(7, 5)
    out = np.zeros(3)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.lib().rtb200_uvb_dust_beta(int(nfreq), float(freqdel), p(al), p(ad), p(out)), "rtb200_uvb_dust_beta")
    return out


def uvb_heating(table, alpha):
    """(gamma9, width3), the inputs of Transport.set_heating (DESIGN.md 4.10): gamma9 [3, 3] = [group][gammaHI, gammaHeI,
    gammaHeII] from the background's table[3][19] (columns 16-18), width3[3] = the band widths in Hz of
    rtb200_uvb_band_width for the effective slopes alpha[3] (uvb_background()["table"], ["alpha"])."""
    import ctypes as C

    from . import _lib
    gamma = np.ascontiguousarray(np.asarray(table, dtype=np.float64).reshape(3, 19)[:, 16:19])
    al = np.ascontiguousarray(alpha, dtype=np.float64).reshape(3)
    width = np.zeros(3)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.lib().rtb200_uvb_band_width(p(al), p(width)), "rtb200_uvb_band_width")
    return gamma, width


# ------------------------------------------------------------------------------------------------------
# grids
# ------------------------------------------------------------------------------------------------------
def nested_leaves(n, refine, max_level):
    """Leaves of an octree over an n^3 base grid in reference leaf order.

    refine(level, x, y, z, size) -> bool mask, with x, y, z the cell CENTRES in box units [0,1) and `size` the cell
    edge; a cell for which it is true (and level < max_level) is replaced by its 8 children.
    Returns level[int8], and the leaf centres cx, cy, cz.
    """
    ix, iy, iz = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
    cur = (ix.ravel().astype(np.int64), iy.ravel().astype(np.int64), iz.ravel().astype(np.int64))
    done = []
    for lvl in range(max_level + 1):
        x, y, z = cur
        size = 1.0 / (n << lvl)
        if lvl < max_level and x.size:
            m = np.asarray(refine(lvl, (x + 0.5) * size, (y + 0.5) * size, (z + 0.5) * size, size), dtype=bool)
        else:
            m = np.zeros(x.size, dtype=bool)
        done.append((lvl, x[~m], y[~m], z[~m]))
        px, py, pz = x[m], y[m], z[m]
        off = np.arange(8)
        cur = ((2 * px[:, None] + (off >> 2)).ravel(), (2 * py[:, None] + ((off >> 1) & 1)).ravel(),
               (2 * pz[:, None] + (off & 1)).ravel())
    keys, lv, cx, cy, cz = [], [], [], [], []
    for lvl, x, y, z in done:
        if x.size == 0:
            continue
        bx, by, bz = x >> lvl, y >> lvl, z >> lvl
        key = (bx * n + by) * n + bz
        for d in range(lvl - 1, -1, -1):
            key = (key << 3) | ((((x >> d) & 1) << 2) | (((y >> d) & 1) << 1) | ((z >> d) & 1))
        key = key << (3 * (max_level - lvl))
        size = 1.0 / (n << lvl)
        keys.append(key); lv.append(np.full(x.size, lvl, dtype=np.int8))
        cx.append((x + 0.5) * size); cy.append((y + 0.5) * size); cz.append((z + 0.5) * size)
    keys = np.concatenate(keys)
    order = np.argsort(keys, kind="stable")
    cat = lambda a: np.concatenate(a)[order]
    return cat(lv), cat(cx), cat(cy), cat(cz)


def species_from_density(nH, xneu):
    """HI, HeI, HeII, rho as the reference initialises a leaf (equiSources.f90:1935-1944)."""
    rho = nH * MP / PSI
    HI = nH * xneu
    HeI = (1.0 - PSI) * rho / MHE
    return HI, HeI, np.zeros_like(HI), rho


def uniform_grid(n, seed=1, box_kpc=100.0, tau_lo=1e-3, tau_hi=20.0, beta24=2.0e-18, helium=True):
    """Config-2/4 style uniform grid: lognormal density (sigma_ln = 1) times a neutral fraction, rescaled so that the
    group-1 optical depth of one cell spans [tau_lo, tau_hi] (per-segment tau then lies in ~[1e-5, 30])."""
    rng = np.random.default_rng(seed)
    N = n ** 3
    box = box_kpc * KPC
    cell = box / n
    ln_tau = rng.uniform(np.log(tau_lo), np.log(tau_hi), N)
    HI = np.exp(ln_tau) / (beta24 * cell)
    nH = HI / 10.0 ** rng.uniform(-4.0, 0.0, N)  # implied total hydrogen density, neutral fraction 1e-4..1
    rho = nH * MP / PSI
    if helium:
        nHe = (1.0 - PSI) * rho / MHE
        f1 = rng.uniform(0.0, 1.0, N)
        HeI = nHe * f1 * (HI / nH)
        HeII = nHe * (1.0 - f1) * rng.uniform(0.0, 1.0, N) * (HI / nH)
    else:
        HeI = np.zeros(N)
        HeII = np.zeros(N)
    return dict(nx=n, level=np.zeros(N, dtype=np.int8), HI=HI, HeI=HeI, HeII=HeII, rho=rho,
                abun2=np.full(N, 0.02), box_size=box)


def nested_grid(n, max_level, refine, seed=1, box_kpc=100.0, tau_lo=1e-3, tau_hi=20.0, beta24=2.0e-18):
    """AMR grid (configs 3 and 5 style): same per-cell optical-depth distribution, measured per base-cell size
    divided by 2^level so that refined cells are not optically thinner on average."""
    level, cx, cy, cz = nested_leaves(n, refine, max_level)
    rng = np.random.default_rng(seed)
    N = level.size
    box = box_kpc * KPC
    cell = box / n / (1 << level.astype(np.int64))
    HI = np.exp(rng.uniform(np.log(tau_lo), np.log(tau_hi), N)) / (beta24 * cell)
    nH = HI / 10.0 ** rng.uniform(-4.0, 0.0, N)
    rho = nH * MP / PSI
    nHe = (1.0 - PSI) * rho / MHE
    f1 = rng.uniform(0.0, 1.0, N)
    HeI = nHe * f1 * (HI / nH)
    HeII = nHe * (1.0 - f1) * rng.uniform(0.0, 1.0, N) * (HI / nH)
    abun2 = 10.0 ** rng.uniform(np.log10(4e-4), np.log10(5e-2), N)
    return dict(nx=n, level=level, HI=HI, HeI=HeI, HeII=HeII, rho=rho, abun2=abun2, box_size=box,
                centres=(cx, cy, cz))


def central_box_refine(lo, hi, levels=1):
    """refine predicate: cells whose centre lies in [lo, hi)^3 (box units) down to `levels` levels"""
    def f(level, x, y, z, size):
        return (level < levels) & (x >= lo) & (x < hi) & (y >= lo) & (y < hi) & (z >= lo) & (z < hi)
    return f


def disc_refine(max_level, r0=0.28, h0=0.06):
    """refine predicate for a synthetic exponential disc (config 5): deeper levels closer to the mid-plane/centre"""
    def f(level, x, y, z, size):
        R = np.sqrt((x - 0.5) ** 2 + (y - 0.5) ** 2)
        s = 0.5 ** level
        return (level < max_level) & (R < r0 * s + size) & (np.abs(z - 0.5) < h0 * s + size)
    return f


# ------------------------------------------------------------------------------------------------------
# point sources
# ------------------------------------------------------------------------------------------------------
def synthetic_spectra(n_wave=1221, seed=0):
    """Stand-in for the starburst99 tables the reference reads (equiSources.f90:840-892; not shipped with it):
    blackbody-like spectra, hotter and brighter at lower metallicity, two time slices, on a log wavelength grid
    91 A .. 1.6e6 A; plus SMC-type extinction-fit parameters in the layout of smc_dust_parameters.dat
    (dustModule.f90:15-24: a(i,1)=lambda_i [micron], a(i,2)=a_i, a(i,3)=b_i, a(i,4)=p_i, a(i,5)=q_i)."""
    wl_A = np.logspace(np.log10(91.0), np.log10(1.6e6), n_wave)
    hc_over_k = 1.4387769e8  # Angstrom K
    lum = np.zeros((5, 2, n_wave))
    for m in range(5):
        for t in range(2):
            T = 4.5e4 * (1.0 - 0.05 * m) * (1.0 - 0.08 * t)
            x = hc_over_k / (wl_A * T)
            planck = 1.0 / (wl_A ** 5 * np.expm1(np.minimum(x, 600.0)))
            lum[m, t] = np.log10(planck / planck.max()) + 40.0 - 0.1 * m - 0.2 * t
    a_dust = np.array([[0.042, 185.0, 90.0, 2.0, 2.0], [0.08, 27.0, 5.5, 4.0, 4.0], [0.22, 0.005, -1.95, 2.0, 2.0],
                       [9.7, 0.010, -1.95, 2.0, 2.0], [18.0, 0.012, -1.8, 2.0, 2.0], [25.0, 0.030, 0.0, 2.0, 2.0],
                       [0.067, 10.0, 1.9, 4.0, 15.0]])
    return dict(wavelength=wl_A * 1.0e-8, lum=lum, metallicity=np.log10(np.array([0.0004, 0.004, 0.008, 0.020, 0.050])),
                coef_spectrum=0.37, a_dust=a_dust)


def point_workload(n, nsrc, seed=3, uniform=False, box_kpc=100.0):
    """Config-1/3 style point-source workload: n^3 base grid (optionally one refined level over the central (n/4)^3 base
    cells), tau_cell(nu_1) log-uniform in [1e-3, 1], metallicities log-uniform in [4e-4, 5e-2]; `nsrc` distinct source
    leaves inside the refined (central) region.  Returns (grid dict, src_leaf[int32])."""
    s24 = float(np.float32(6.3e-18))
    if uniform:
        g = uniform_grid(n, seed=seed, box_kpc=box_kpc, tau_lo=1e-3, tau_hi=1.0, beta24=s24)
        rng = np.random.default_rng(seed + 100)
        g["abun2"] = 10.0 ** rng.uniform(np.log10(4e-4), np.log10(5e-2), n ** 3)
        c = np.arange(n)
        central = np.where((c >= 3 * n // 8) & (c < 5 * n // 8))[0]
        ix = rng.choice(central, nsrc); iy = rng.choice(central, nsrc); iz = rng.choice(central, nsrc)
        leaves = np.unique(((ix * n + iy) * n + iz).astype(np.int64))
    else:
        g = nested_grid(n, 1, central_box_refine(0.375, 0.625, levels=1), seed=seed, box_kpc=box_kpc, tau_lo=1e-3,
                        tau_hi=1.0, beta24=s24)
        rng = np.random.default_rng(seed + 100)
        leaves = np.where(g["level"] == 1)[0]
    pick = rng.choice(leaves, size=min(nsrc, leaves.size), replace=False)
    if pick.size < nsrc:  # tiny grids: allow repeats
        pick = np.concatenate([pick, rng.choice(leaves, size=nsrc - pick.size)])
    return g, np.sort(pick).astype(np.int32)


# ------------------------------------------------------------------------------------------------------
# chemistry
# ------------------------------------------------------------------------------------------------------
def rate_tables(nratec=5000, temstart=1.0, temend=1.0e9):
    """Stand-in for the k1a..k6a tables of calc_rates.f (out of scope, SURVEY.md section 2): collisional ionisation and
    recombination coefficients of H and He in the analytic forms of Cen (1992), tabulated on the driver's log-T grid
    (equiSources.f90:174-176: dlogtem uses real(nratec-1), a single-precision divisor).  Workload parameters, fed
    identically to the GPU path and to the oracle."""
    logtem0, logtem9 = float(np.log(temstart)), float(np.log(temend))
    dlogtem = (logtem9 - logtem0) / float(np.float32(nratec - 1))
    T = np.exp(logtem0 + np.arange(nratec) * dlogtem)
    sq, t5 = np.sqrt(T), 1.0 / (1.0 + np.sqrt(T / 1.0e5))
    k = np.zeros((6, nratec))
    k[0] = 5.85e-11 * sq * np.exp(-157809.1 / T) * t5                      # HI  + e -> HII   + 2e
    k[1] = 8.4e-11 / sq * (T / 1.0e3) ** -0.2 / (1.0 + (T / 1.0e6) ** 0.7)  # HII + e -> HI
    k[2] = 2.38e-11 * sq * np.exp(-285335.4 / T) * t5                      # HeI + e -> HeII  + 2e
    k[3] = 1.5e-10 * T ** -0.6353                                          # HeII + e -> HeI
    k[4] = 5.68e-12 * sq * np.exp(-631515.0 / T) * t5                      # HeII + e -> HeIII + 2e
    k[5] = 3.36e-10 / sq * (T / 1.0e3) ** -0.2 / (1.0 + (T / 1.0e6) ** 0.7)  # HeIII + e -> HeII
    return dict(k=np.maximum(k, 1e-300), logtem0=logtem0, logtem9=logtem9, dlogtem=dlogtem)
