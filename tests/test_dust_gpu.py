"""GPU tests of dust in the diffuse sweep (DESIGN.md 4.8): mode 0, and dust set then cleared, give the dust-free bits on
every route; scattering dust of albedo 1 is bit for bit the per-leaf sigma = kd of rtb200_grid_set_scattering; absorbing
and scattering dust agree with the dust oracle (tests/dust_oracle.py); a conservative dust box reaches its fixed point;
the opacity follows the species of every call; the state is handled as documented; device groups of one and two GPUs
(threads and processes) agree with the single context."""
import os
import subprocess
import sys

import numpy as np
import pytest

import dust_oracle
from conftest import rel_err
from radiativetransfer_b200 import workloads as W
from test_scattering_oracle import NDIR, FIXED_POINT_BAR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"faithful": 1e-9, "fast": 1e-8}
K = 4
ALBEDO = (0.3, 0.5, 0.7)


@pytest.fixture(scope="module")
def rt(build_product):
    import radiativetransfer_b200 as rt
    return rt


@pytest.fixture()
def engine(rt):
    t = rt.Transport(device=0)
    yield t
    t.close()


def _set(t, g):
    t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])


def _mode(rt, name):
    return rt.MATH_FAITHFUL if name == "faithful" else rt.MATH_FAST


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


def _dusty(g, seed):
    """the grid with a seeded metallicity abun2 in [0.005, 0.04]"""
    g = dict(g)
    g["abun2"] = np.random.default_rng(seed).uniform(0.005, 0.04, g["level"].size)
    return g


def _beta_dust(g, uvbg, mode, scale="max"):
    """the band means of the synthetic fit, scaled so that the largest dust opacity of group 1 equals the gas's largest
    (scale="max") or the median dust opacity the gas's median (scale="median").
    "max" keeps every cell's optical depth within twice the grid's gas range (<= 71 here).  The dust still changes J by
    more than 1 % in 95-100 % of the cells.
    "median" makes mode 2, which follows rho and not HI, reach tau ~6600 in one cell.  That puts boundary rays whose Iout
    is a non-zero subnormal inside single segments (per-segment tau ~650-745), where FAST arithmetic departs from the
    reference formula by design (DESIGN.md 4.1); only test_thick_dust_vs_oracle uses it."""
    bd = W.uvb_dust_beta(uvbg["alpha"], W.synthetic_spectra()["a_dust"])
    kd = dust_oracle.dust_kd(g, bd, mode)
    pick = np.max if scale == "max" else np.median
    return bd * (pick(_kappa(g, uvbg["beta"])[0]) / pick(kd[0]))


def _eta(g, uvb, beta, seed):
    rng = np.random.default_rng(seed + 1000)
    kap = np.maximum(_kappa(g, beta), 1e-30)
    return 10.0 ** rng.uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap


BALANCED = _dusty(W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4), 4)


def _corner(level, x, y, z, size):
    return (level < 3) & (x < 0.26) & (y < 0.26) & (z > 0.74)


UNBALANCED = _dusty(W.nested_grid(4, 3, _corner, seed=6), 6)
GRIDS = {"u32": lambda: _dusty(W.uniform_grid(32, seed=32), 32), "u64": lambda: _dusty(W.uniform_grid(64, seed=64), 64),
         "balanced": lambda: BALANCED, "unbalanced": lambda: UNBALANCED,
         "u128-subset": lambda: _dusty(W.uniform_grid(128, seed=128), 128)}
SUBSET = np.array([3, 40, 77, 101, 150, 188], dtype=np.int32)   # directions of six zones
_CACHE = {}


def _grid(name):
    if name not in _CACHE:
        _CACHE[name] = GRIDS[name]()
    return _CACHE[name]


def _uvb(uvbg, g):
    return uvbg["uvb"] * (1.0 if g["level"].max() == 0 else 1e-3)   # nested grids: inside the refined-leaf guard


# routes: (name, tuning, group of one)
ROUTES = [("cells1-transpose0-graph1", dict(cells=1, transpose_z=0, graph=1), "u32"),
          ("cells2-transpose1-graph1", dict(cells=2, transpose_z=1, graph=1), "u32"),
          ("cells2-transpose1-graph0", dict(cells=2, transpose_z=1, graph=0), "u32"),
          ("amr_stream0", dict(amr_stream=0), "balanced"), ("amr_stream1", dict(amr_stream=1), "balanced"),
          ("group1", None, "u32"), ("group1-nested", None, "balanced")]


def _route_engine(rt, tuning, math=None):
    t = rt.Transport(devices=[0]) if tuning is None else rt.Transport(device=0)
    if tuning:
        t.set_tuning(**tuning)
    if math is not None:
        t.set_math(math)
    return t


# ---- 1. mode 0 and cleared dust are the dust-free sweep --------------------------------------------------------------
@pytest.mark.parametrize("route,tuning,grid", ROUTES, ids=[r[0] for r in ROUTES])
def test_mode0_and_cleared_dust_bit_for_bit(rt, uvbg, route, tuning, grid):
    g = _grid(grid)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    t = _route_engine(rt, tuning)
    try:
        _set(t, g)
        ref, n0 = t.diffuse(uvb, beta)
        t.set_dust(0)
        J, n = t.diffuse(uvb, beta)
        assert np.array_equal(J, ref) and n == n0
        bd = _beta_dust(g, uvbg, 2)
        t.set_dust(2, bd)
        Jd, _ = t.diffuse(uvb, beta)
        assert not np.array_equal(Jd, ref)
        t.set_dust(0)
        J, n = t.diffuse(uvb, beta)
        assert np.array_equal(J, ref) and n == n0
        t.set_dust(1, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
        t.diffuse(uvb, beta)
        assert t.last_scattering()["iterations"] == 3
        t.set_dust(0, None)
        J, n = t.diffuse(uvb, beta)
        assert np.array_equal(J, ref) and n == n0 and t.last_scattering() == {"iterations": 0, "residual": 0.0}
    finally:
        t.close()


# ---- 2. albedo 1 is the per-leaf sigma = kd --------------------------------------------------------------------------
@pytest.mark.parametrize("route,tuning,grid", ROUTES, ids=[r[0] for r in ROUTES])
@pytest.mark.parametrize("mode", [1, 2])
def test_albedo_one_is_the_per_leaf_sigma(rt, uvbg, route, tuning, grid, mode):
    g = _grid(grid)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    bd = _beta_dust(g, uvbg, mode)
    kd = dust_oracle.dust_kd(g, bd, mode)
    t = _route_engine(rt, tuning, rt.MATH_FAITHFUL if mode == 1 else rt.MATH_FAST)
    try:
        _set(t, g)
        t.set_emission(_eta(g, uvb, beta, 5))
        for max_iter, tol in ((3, 0.0), (100, 1e-9)):
            t.set_dust(mode, bd, albedo=(1.0, 1.0, 1.0), max_iterations=max_iter, tolerance=tol)
            Jd, nd = t.diffuse(uvb, beta)
            sd = t.last_scattering()
            t.set_dust(0)
            t.set_scattering(kd, max_iterations=max_iter, tolerance=tol)
            Js, ns = t.diffuse(uvb, beta)
            ss = t.last_scattering()
            t.set_scattering(None)
            assert sd == ss and nd == ns, (sd, ss)
            assert np.array_equal(Jd, Js), rel_err(Jd, Js)
    finally:
        t.close()


# ---- 3. / 4. against the dust oracle ---------------------------------------------------------------------------------
def _oracle(gname, g, uvbg, mode, albedo, max_iter, tol, rays=None, scale="max"):
    """the dust oracle's solve, once per case"""
    key = (gname, mode, tuple(albedo), max_iter, tol, scale)
    if key not in _CACHE:
        uvb, beta = _uvb(uvbg, g), uvbg["beta"]
        kd = dust_oracle.dust_kd(g, _beta_dust(g, uvbg, mode, scale), mode)
        o = dust_oracle.grid(g).solve(uvb, beta, None, kd, np.asarray(albedo)[:, None] * kd, max_iter, tol, rays=rays)
        assert o["status"] == 0
        _CACHE[key] = o
    return _CACHE[key]


@pytest.mark.parametrize("math", ["fast", "faithful"])
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("gname", ["u32", "u64", "balanced", "unbalanced", "u128-subset"])
def test_absorbing_dust_vs_oracle(rt, engine, uvbg, gname, mode, math):
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    rays = SUBSET if gname == "u128-subset" else None
    engine.set_math(_mode(rt, math))
    _set(engine, g)
    engine.set_dust(mode, _beta_dust(g, uvbg, mode))
    J, nseg = engine.diffuse(uvb, beta, rays=rays)
    o = _oracle(gname, g, uvbg, mode, (0.0, 0.0, 0.0), 1, 0.0, rays)
    err = rel_err(J, o["J"])
    print(f"absorbing dust {gname} mode {mode} {math}: rel err {err:.3e}")
    assert nseg == o["nseg"] and engine.last_scattering()["iterations"] == 0
    assert err < TOL[math], err


def test_thick_dust_vs_oracle(rt, engine, uvbg):
    """mode 2 at the median scaling: cells up to tau ~6600.  FAITHFUL follows the reference formula operation for
    operation, so it holds the 1e-9 bar there too.  FAST keeps its documented deviation where a segment's Iout is a
    non-zero subnormal: the reference's log(Iin/Iout) then has only a few significant bits, up to ln 2 absolute error on
    a log of ~280-745.  It stays well inside 1e-2."""
    g = _grid("u32")
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    bd = _beta_dust(g, uvbg, 2, scale="median")
    o = _oracle("u32", g, uvbg, 2, (0.0, 0.0, 0.0), 1, 0.0, scale="median")
    _set(engine, g)
    engine.set_dust(2, bd)
    out = {}
    for math in ("faithful", "fast"):
        engine.set_math(_mode(rt, math))
        J, nseg = engine.diffuse(uvb, beta)
        assert nseg == o["nseg"] and np.all(np.isfinite(J)) and np.all(J >= 0)
        out[math] = rel_err(J, o["J"])
    print(f"thick dust u32 mode 2: FAITHFUL {out['faithful']:.3e}, FAST {out['fast']:.3e}")
    assert out["faithful"] < TOL["faithful"], out
    assert out["fast"] < 1e-2, out


@pytest.mark.parametrize("math", ["fast", "faithful"])
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("gname", ["u32", "balanced"])
def test_scattering_dust_fixed_iterations_vs_oracle(rt, engine, uvbg, gname, mode, math):
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    engine.set_math(_mode(rt, math))
    _set(engine, g)
    engine.set_dust(mode, _beta_dust(g, uvbg, mode), albedo=ALBEDO, max_iterations=K, tolerance=0.0)
    J, nseg = engine.diffuse(uvb, beta)
    s = engine.last_scattering()
    o = _oracle(gname, g, uvbg, mode, ALBEDO, K, 0.0)
    err = rel_err(J, o["J"])
    print(f"scattering dust {gname} mode {mode} {math} K={K}: rel err {err:.3e}, residual {s['residual']:.3e} "
          f"(oracle {o['residual']:.3e})")
    assert s["iterations"] == K and nseg == o["nseg"]
    assert abs(s["residual"] - o["residual"]) <= 1e-4 * o["residual"]
    assert err < TOL[math], err


@pytest.mark.parametrize("mode", [1, 2])
def test_stopping_rule_takes_the_oracles_decision(rt, engine, uvbg, mode):
    g = _grid("u32")
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    hist = _oracle("u32", g, uvbg, mode, ALBEDO, 8, 0.0)["history"]
    k = 5
    tol = float(np.sqrt(hist[k - 1] * hist[k]))   # between the residuals of sweeps k and k + 1
    assert hist[k - 1] / tol > 1.01 and tol / hist[k] > 1.01, hist
    engine.set_math(_mode(rt, "faithful"))
    _set(engine, g)
    engine.set_dust(mode, _beta_dust(g, uvbg, mode), albedo=ALBEDO, max_iterations=60, tolerance=tol)
    J, _ = engine.diffuse(uvb, beta)
    s = engine.last_scattering()
    o = _oracle("u32", g, uvbg, mode, ALBEDO, 60, tol)
    print(f"stopping mode {mode}: residuals {['%.2e' % h for h in hist]}, tol {tol:.3e}, oracle {o['iterations']}, "
          f"GPU {s['iterations']}, err {rel_err(J, o['J']):.3e}")
    assert o["iterations"] == k + 1 and s["iterations"] == o["iterations"] and s["residual"] <= tol
    assert rel_err(J, o["J"]) < TOL["faithful"]


# ---- 5. conservative dust --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("math", ["fast", "faithful"])
def test_conservative_dust_box(rt, engine, uvbg, math):
    g = _dusty(W.uniform_grid(16, seed=8), 8)
    beta0 = np.zeros(9)                                  # no gas opacity: the dust alone, albedo 1
    col = g["HI"] * g["abun2"] / float(np.float32(0.2))
    bd = np.full(3, 1.0 / (np.mean(col) * g["box_size"]))   # box optical depth ~1
    engine.set_math(_mode(rt, math))
    _set(engine, g)
    engine.set_dust(1, bd, albedo=(1.0, 1.0, 1.0), max_iterations=400, tolerance=1e-12)
    J, _ = engine.diffuse(uvbg["uvb"], beta0)
    s = engine.last_scattering()
    want = uvbg["uvb"][:, None] * (NDIR * float(np.float32(1.0) / np.float32(NDIR)))
    err = float(np.max(np.abs(J - want) / want))
    print(f"conservative dust 16^3 {math}: {s['iterations']} iterations, residual {s['residual']:.3e}, err {err:.3e}")
    assert s["residual"] <= 1e-12 and np.all(np.isfinite(J))
    assert err < FIXED_POINT_BAR, err


# ---- 6. the opacity follows the species ------------------------------------------------------------------------------
def test_dust_follows_the_species(rt, uvbg):
    import torch
    g = _dusty(W.uniform_grid(24, seed=9), 9)
    N = g["level"].size
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    bd = _beta_dust(g, uvbg, 1)
    ktab = W.rate_tables(500)
    tgas = 10.0 ** np.random.default_rng(2).uniform(4.0, 4.1, N)
    ksi = np.concatenate([uvbg["ksi24"], uvbg["ksi25"], uvbg["ksi26"]])

    def fresh(HI, HeI, HeII):
        t = rt.Transport(device=0)
        _set(t, dict(g, HI=HI, HeI=HeI, HeII=HeII))
        t.set_dust(1, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
        J, _ = t.diffuse(uvb, beta)
        t.close()
        return J

    t = rt.Transport(device=0)
    try:
        _set(t, g)
        t.set_dust(1, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
        t.diffuse(uvb, beta)
        HI2 = g["HI"] * np.random.default_rng(10).uniform(0.2, 3.0, N)
        t.update_species(HI=HI2)
        J, _ = t.diffuse(uvb, beta)
        assert np.array_equal(J, fresh(HI2, g["HeI"], g["HeII"]))
        # one device-resident outer step: the sweep, then chemistry changes HI on the device
        t.set_rate_tables(ktab); t.set_temperature(tgas)
        Jd = torch.zeros((3, N), dtype=torch.float64, device="cuda:0")
        s = torch.cuda.current_stream().cuda_stream
        t.diffuse_device(uvb, beta, Jd.data_ptr(), stream=s)
        t.chemistry_device(0, Jd.data_ptr(), ksi=ksi, stream=s, want_change=False)
        t.diffuse_device(uvb, beta, Jd.data_ptr(), stream=s)
        torch.cuda.synchronize()
        HI3, HeI3, HeII3 = t.get_species()
        assert not np.array_equal(HI3, HI2)
        assert np.array_equal(Jd.cpu().numpy(), fresh(HI3, HeI3, HeII3))
    finally:
        t.close()


# ---- 7. state --------------------------------------------------------------------------------------------------------
def test_state_handling(rt, engine, uvbg):
    g = _dusty(W.uniform_grid(16, seed=71), 71)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    N = g["level"].size
    bd = _beta_dust(g, uvbg, 2)
    _set(engine, g)
    plain, n0 = engine.diffuse(uvb, beta)
    engine.set_dust(2, bd, albedo=ALBEDO, max_iterations=5, tolerance=0.0)
    J5, n5 = engine.diffuse(uvb, beta)
    assert n5 == 5 * n0 and engine.last_scattering()["iterations"] == 5
    sigma = np.full((3, N), 1e-25)
    nan3, inf3 = np.array([bd[0], np.nan, bd[2]]), np.array([bd[0], bd[1], np.inf])
    refused = [dict(approximation=3, beta_dust=bd), dict(approximation=-1, beta_dust=bd),
               dict(approximation=2, beta_dust=-bd), dict(approximation=2, beta_dust=nan3),
               dict(approximation=2, beta_dust=inf3), dict(approximation=2, beta_dust=bd, albedo=(0.5, -0.1, 0.5)),
               dict(approximation=2, beta_dust=bd, albedo=(0.5, 1.5, 0.5)),
               dict(approximation=2, beta_dust=bd, albedo=(np.nan, 0.5, 0.5)),
               dict(approximation=2, beta_dust=bd, albedo=ALBEDO, max_iterations=0),
               dict(approximation=2, beta_dust=bd, albedo=ALBEDO, tolerance=-1e-9),
               dict(approximation=2, beta_dust=bd, albedo=ALBEDO, tolerance=float("inf"))]
    for kw in refused:
        with pytest.raises(rt.RTB200Error):
            engine.set_dust(**kw)
        J, _ = engine.diffuse(uvb, beta)
        assert np.array_equal(J, J5) and engine.last_scattering()["iterations"] == 5, kw
    # scattering dust refuses a per-leaf sigma, and a direction subset
    with pytest.raises(rt.RTB200Error):
        engine.set_scattering(sigma, max_iterations=5, tolerance=0.0)
    with pytest.raises(rt.RTB200Error) as e:
        engine.diffuse(uvb, beta, rays=np.arange(10))
    assert e.value.status == 12
    J, _ = engine.diffuse(uvb, beta)
    assert np.array_equal(J, J5)
    # update_species keeps the dust, set_grid clears it
    engine.update_species(HI=g["HI"])
    J, _ = engine.diffuse(uvb, beta)
    assert np.array_equal(J, J5)
    _set(engine, g)
    J, n = engine.diffuse(uvb, beta)
    assert np.array_equal(J, plain) and n == n0
    # a per-leaf sigma refuses scattering dust; absorbing dust combines with it and with a direction subset
    engine.set_scattering(sigma, max_iterations=5, tolerance=0.0)
    Js, _ = engine.diffuse(uvb, beta)
    with pytest.raises(rt.RTB200Error):
        engine.set_dust(2, bd, albedo=ALBEDO, max_iterations=5, tolerance=0.0)
    J, _ = engine.diffuse(uvb, beta)
    assert np.array_equal(J, Js)
    engine.set_dust(2, bd)
    J, _ = engine.diffuse(uvb, beta)
    assert engine.last_scattering()["iterations"] == 5 and not np.array_equal(J, Js)
    engine.set_scattering(None)
    Jsub, _ = engine.diffuse(uvb, beta, rays=np.arange(10))
    assert np.all(np.isfinite(Jsub))
    # the modes need their fields
    t = rt.Transport(device=0)
    try:
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], None, None, g["box_size"])
        for m in (1, 2):
            with pytest.raises(rt.RTB200Error):
                t.set_dust(m, bd)
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], None, g["abun2"], g["box_size"])
        t.set_dust(1, bd)
        with pytest.raises(rt.RTB200Error):
            t.set_dust(2, bd)
    finally:
        t.close()


# ---- 8. device groups ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ndev", [1, 2])
@pytest.mark.parametrize("tol", [0.0, 1e-9])
def test_device_group_equals_plain_context(rt, uvbg, ndev, tol):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = _dusty(W.uniform_grid(24, seed=81), 81)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    bd, eta = _beta_dust(g, uvbg, 2), _eta(g, uvb, beta, 81)
    kd = dust_oracle.dust_kd(g, bd, 2)
    mi = K if tol == 0 else 100
    t = rt.Transport(device=0, math=rt.MATH_FAITHFUL)
    _set(t, g)
    t.set_emission(eta)
    t.set_dust(2, bd, albedo=ALBEDO, max_iterations=mi, tolerance=tol)
    ref, n0 = t.diffuse(uvb, beta)
    s0 = t.last_scattering()
    t.set_dust(1, bd)
    ref_abs, _ = t.diffuse(uvb, beta)
    t.close()
    m = rt.Transport(devices=list(range(ndev)), math=rt.MATH_FAITHFUL)
    try:
        _set(m, g)
        m.set_emission(eta)
        m.set_dust(2, bd, albedo=ALBEDO, max_iterations=mi, tolerance=tol)
        J, n1 = m.diffuse(uvb, beta)
        s1 = m.last_scattering()
        with pytest.raises(rt.RTB200Error):
            m.set_scattering(kd, max_iterations=mi, tolerance=tol)
        with pytest.raises(rt.RTB200Error):
            m.diffuse(uvb, beta, rays=np.arange(10))
        m.diffuse_resident(uvb, beta)
        m.sync()
        assert m.last_scattering()["iterations"] == s1["iterations"]
        for local in range(ndev):
            off, cnt, Js, _, _ = m.slab_get(local)
            assert np.array_equal(Js, J[:, off:off + cnt])
        # albedo 1 is the per-leaf sigma = kd, in the group too
        m.set_dust(2, bd, albedo=(1.0, 1.0, 1.0), max_iterations=mi, tolerance=tol)
        Jd, _ = m.diffuse(uvb, beta)
        m.set_dust(0)
        m.set_scattering(kd, max_iterations=mi, tolerance=tol)
        Jk, _ = m.diffuse(uvb, beta)
        assert np.array_equal(Jd, Jk)
        m.set_scattering(None)
        m.set_dust(1, bd)
        Ja, _ = m.diffuse(uvb, beta)
    finally:
        m.close()
    print(f"dust group of {ndev}, tol {tol}: {s1['iterations']} iterations (single {s0['iterations']}), "
          f"err {rel_err(J, ref):.3e}, absorbing err {rel_err(Ja, ref_abs):.3e}")
    assert n0 == n1 and s1["iterations"] == s0["iterations"]
    if ndev == 1:
        assert np.array_equal(J, ref) and s1["residual"] == s0["residual"] and np.array_equal(Ja, ref_abs)
    else:
        assert rel_err(J, ref) < 1e-12 and rel_err(Ja, ref_abs) < 1e-12


@pytest.mark.parametrize("ndev", [1, 2])
def test_resident_outer_steps_with_chemistry(rt, uvbg, ndev):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = _dusty(W.nested_grid(6, 2, W.central_box_refine(0.2, 0.7, levels=2), seed=5, tau_lo=1e-2, tau_hi=2.0), 5)
    N = g["level"].size
    uvb, beta = uvbg["uvb"] * 1e-3, uvbg["beta"]
    bd = _beta_dust(g, uvbg, 1)
    ktab = W.rate_tables(500)
    tgas = 10.0 ** np.random.default_rng(2).uniform(4.0, 4.1, N)
    ksi = np.concatenate([uvbg["ksi24"], uvbg["ksi25"], uvbg["ksi26"]])
    one = rt.Transport(device=0)
    _set(one, g)
    one.set_rate_tables(ktab); one.set_temperature(tgas)
    one.set_dust(1, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
    J = torch.zeros(3, N, dtype=torch.float64, device="cuda:0")
    s = torch.cuda.current_stream(0).cuda_stream
    for _ in range(2):
        one.diffuse_device(uvb, beta, J.data_ptr(), stream=s)
        one.chemistry_device(0, J.data_ptr(), ksi=ksi, stream=s, want_change=False)
    torch.cuda.synchronize()
    ref = one.get_species()
    one.close()
    grp = rt.Transport(devices=list(range(ndev)))
    try:
        _set(grp, g)
        grp.set_rate_tables(ktab); grp.set_temperature(tgas)
        grp.set_dust(1, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
        for _ in range(2):
            grp.diffuse_resident(uvb, beta, ksi=ksi, chemistry=True)
        grp.sync()
        assert grp.last_scattering()["iterations"] == 3
        got = grp.get_species()
    finally:
        grp.close()
    assert not np.array_equal(ref[0], g["HI"])
    for a, b in zip(got, ref):
        assert rel_err(a, b, floor=1e-300) < 1e-9


def test_one_process_per_gpu(rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(ROOT, "tests", "dust_rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:]); sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0
    assert r.stdout.count("RANK-OK") == 2
