"""GPU parity tests of the nested-grid diffuse sweep at the benchmarked sizes: bench.py's two nested grids (64^3 + 3
levels, 0.50 M leaves; 128^3 + 2 levels, 3.17 M leaves) and a strongly unbalanced grid of 1.15 M leaves, against the
oracle, on both default launch routes (DESIGN.md 4.4).

The sweep picks its route by the size of its waves: under 40 000 leaf-groups per wave the whole batch is one
`amr_stream_kernel` launch whose work items wait for their upstream records (64^3 + 3 levels), above it one
`amr_wave_kernel` launch per wave, FAST arithmetic with the 8-blocks register cap (128^3 + 2 levels).  The grids of
tests/test_diffuse_amr_gpu.py all have small waves, so only these sizes reach the per-wave FAST kernel of the
benchmark, put the streamed kernel's record polling under real contention, and show what the thin-segment rule buys.
Routes are forced with `amr_stream` only, and checked through the launch count of every sweep."""
import os

import numpy as np
import pytest

import emission_oracle
from conftest import rel_err
from radiativetransfer_b200 import workloads as W

pytestmark = pytest.mark.gpu
TOL = 1e-9
W192 = float(np.float32(1) / np.float32(192))   # the reference's weight of one direction (real*4)
ALL = np.arange(192, dtype=np.int32)


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


def _oracle_threads(nleaf, want):
    """host threads for the threaded oracle: every thread sweeps a private copy of the octree (~260 B per leaf)"""
    import psutil
    return int(max(1, min(want, os.cpu_count() or 1, (0.5 * psutil.virtual_memory().available) // (260.0 * nleaf))))


def _oracle(og, g, bg, rays):
    o = og.diffuse_mt(bg["uvb"], bg["beta"], rays, nthreads=_oracle_threads(g["level"].size, 64))
    assert o["status"] == 0
    return o


def _sweep(t, bg, rays=None):
    """(J, nseg, route) of one host-buffer sweep.  The route comes from the launch count: one streamed batch is at
    most 9 launches (one amr_stream_kernel launch with the copies, neighbour threading and merge around it), the
    per-wave scheme one launch per wave (568 at 64^3 + 3 levels, 879 at 128^3 + 2).  The bounds leave room for the
    few direction batches a card with less free memory cuts 192 directions into.  A streamed sweep that gave up on a
    record, or any other device-side guard, fails here."""
    J, nseg = t.diffuse(bg["uvb"], bg["beta"], rays=rays)
    assert t.device_error() == 0
    n = t.last_stats()["launches"]
    assert n < 40 or n > 200, f"{n} launches: neither route"
    return J, nseg, "streamed" if n < 40 else "per-wave"


def _combo(izone):
    """reflection combination of a zone (bit c: physical axis c reflected), rotateIndicesModule.f90:14-111 as
    csrc/geometry.cpp tabulates it"""
    b = (izone - 1) % 12
    refl = ((0, 0, 0), (0, 0, 1), (0, 1, 1), (0, 1, 0))[b // 3]
    return int(izone > 12) | refl[1] << 1 | refl[2] << 2


def _zones(rt):
    """zone -> its directions (HEALPix pixel numbers, ascending) at nAngularLevel = 3"""
    z = {}
    for r in range(192):
        z.setdefault(rt.direction(3, r)[0], []).append(r)
    return z


def _per_zone(rt, k):
    """the first k directions of every one of the 24 zones: all 24 zones and all 8 reflection combinations"""
    z = _zones(rt)
    rays = np.array(sorted(r for v in z.values() for r in v[:k]), dtype=np.int32)
    zones = {rt.direction(3, int(r))[0] for r in rays}
    assert len(zones) == 24 and rays.size == 24 * k
    assert {_combo(i) for i in zones} == set(range(8))
    return rays


def _bench_grid(name):
    import bench
    _, g, bg = bench.make_inputs(bench.WORKLOADS[name])
    return g, bg


@pytest.fixture(scope="module")
def g64():
    return _bench_grid("diffuse-64^3-amr3-192dir")


@pytest.fixture(scope="module")
def g128():
    return _bench_grid("diffuse-128^3-amr2-192dir")


@pytest.fixture(scope="module")
def gunb():
    """64^3 with a central box refined three levels at once: level 3 next to level 0 on every face of the box, 1.15 M
    leaves (the grid on which the round-1 flag-guarded scheme overflowed its deferred list, status 14)"""
    g = W.nested_grid(64, 3, W.central_box_refine(0.40625, 0.59375, levels=3), seed=5)
    assert g["level"].size == 1145152 and not np.any((g["level"] == 1) | (g["level"] == 2))
    return g, W.uvb_background(3.0)


@pytest.fixture(scope="module")
def rays48(rt):
    return _per_zone(rt, 2)


def _oracle_grid(oracle, g):
    return oracle.OracleGrid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])


@pytest.fixture(scope="module")
def o64(oracle, g64):
    g, bg = g64
    return _oracle(_oracle_grid(oracle, g), g, bg, ALL)


@pytest.fixture(scope="module")
def o128_48(oracle, g128, rays48):
    g, bg = g128
    return _oracle(_oracle_grid(oracle, g), g, bg, rays48)


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


def _eta(g, uvb, beta, seed):
    """seeded emission with source functions S = eta / kappa from 1e-3 to 1 of the boundary intensity"""
    rng = np.random.default_rng(seed)
    kap = np.maximum(_kappa(g, beta), 1e-30)
    return 10.0 ** rng.uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap


def _emission_oracle(g, bg, eta, rays):
    og = emission_oracle.grid(g)
    og.set_emission(eta)
    return _oracle(og, g, bg, rays)


@pytest.fixture(scope="module")
def e64(g64):
    g, bg = g64
    eta = _eta(g, bg["uvb"], bg["beta"], 64)
    return eta, _emission_oracle(g, bg, eta, ALL)


@pytest.fixture(scope="module")
def e128_48(g128, rays48):
    g, bg = g128
    eta = _eta(g, bg["uvb"], bg["beta"], 128)
    return eta, _emission_oracle(g, bg, eta, rays48)


# ---- 1. 64^3 + 3 levels: the default streamed route, all 192 directions ---------------------------------------------
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_64cube_amr3_all_directions_vs_oracle(rt, engine, g64, o64, mode):
    g, bg = g64
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    J, nseg, route = _sweep(engine, bg)
    err = rel_err(J, o64["J"])
    print(f"64^3 + 3 levels x 192 vs oracle, {mode}, {route}: rel L-inf {err:.3e}")
    assert route == "streamed"
    assert nseg == o64["nseg"]
    assert err < TOL


# ---- 2. 128^3 + 2 levels: the default per-wave route ----------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_128cube_amr2_two_directions_per_zone_vs_oracle(rt, engine, g128, rays48, o128_48, mode):
    """48 directions, two of every zone, make 24 groups: waves as large as the full solve's, so the same per-wave route.
    FAST is held to 1e-8 on the subset: the reference formula's own rounding noise (~1.1e-16 / tau per segment) does
    not average out over a few directions (test_diffuse_gpu.py::test_headline_256cube_direction_subset_vs_oracle)"""
    g, bg = g128
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    J, nseg, route = _sweep(engine, bg, rays=rays48)
    err = rel_err(J, o128_48["J"])
    print(f"128^3 + 2 levels x {rays48.size} vs oracle, {mode}, {route}: rel L-inf {err:.3e}")
    assert route == "per-wave"
    assert nseg == o128_48["nseg"]
    assert err < (TOL if mode == "faithful" else 1e-8)


def test_128cube_amr2_fast_vs_faithful_full_solve(rt, engine, g128):
    """the full 192-direction solve in both modes: the thin-segment rule (segments under 1e-3 of a cell in the
    reference's operation sequence) keeps FAST within 1e-9 of FAITHFUL; without it the two differ by 5.6e-9 here"""
    g, bg = g128
    _set(engine, g)
    engine.set_math(rt.MATH_FAITHFUL)
    Jf, nf, rf = _sweep(engine, bg)
    engine.set_math(rt.MATH_FAST)
    Jq, nq, rq = _sweep(engine, bg)
    err = rel_err(Jq, Jf)
    print(f"128^3 + 2 levels x 192, FAST ({rq}) vs FAITHFUL ({rf}): rel L-inf {err:.3e}")
    assert rf == rq == "per-wave"
    assert nf == nq
    assert err < TOL


@pytest.mark.skipif(not os.environ.get("RTB_SLOW_TESTS"), reason="~1 minute of host time: set RTB_SLOW_TESTS=1")
def test_128cube_amr2_all_directions_vs_oracle(rt, engine, oracle, g128):
    """the benchmarked nested-grid solve in full against the oracle on all host threads (1.1e9 segment updates on the
    CPU, ~20 s on 16 threads); the result of the last run is recorded in profiles/"""
    g, bg = g128
    o = _oracle(_oracle_grid(oracle, g), g, bg, ALL)
    _set(engine, g)
    for mode in ("fast", "faithful"):
        engine.set_math(_mode(rt, mode))
        J, nseg, route = _sweep(engine, bg)
        err = rel_err(J, o["J"])
        print(f"128^3 + 2 levels x 192 vs oracle, {mode}, {route}: rel L-inf {err:.3e}")
        assert route == "per-wave"
        assert nseg == o["nseg"]
        assert err < TOL


# ---- 3. routes, repeats, species updates, batches and shards: identical bits at size ------------------------------
@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("grid,default", [("g64", "streamed"), ("g128", "per-wave")])
def test_routes_and_repeats_bit_identical_at_size(rt, engine, request, grid, default, mode):
    """same arithmetic and summation order on every route: the other route, consecutive streamed sweeps (the records'
    sign alternates from sweep to sweep), a sweep on other opacities and back, direction batches; direction shards add
    up to the full solve"""
    g, bg = request.getfixturevalue(grid)
    name = {"g64": "64^3 + 3", "g128": "128^3 + 2"}[grid]
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    ref, nref, route = _sweep(engine, bg)
    assert route == default
    other = "per-wave" if default == "streamed" else "streamed"
    engine.set_tuning(amr_stream=int(other == "streamed"))
    J, n, route = _sweep(engine, bg)
    print(f"{name}, {mode}: {other} route vs default ({default}): identical {np.array_equal(J, ref)}, "
          f"rel L-inf {rel_err(J, ref):.3e}")
    assert route == other and n == nref and np.array_equal(J, ref)
    engine.set_tuning(amr_stream=1)
    for rep in range(3):
        J, n, route = _sweep(engine, bg)
        print(f"{name}, {mode}: streamed sweep {rep + 1} of 3: identical {np.array_equal(J, ref)}")
        assert route == "streamed" and n == nref and np.array_equal(J, ref), rep
    engine.set_tuning(amr_stream=-1)
    engine.update_species(HI=g["HI"] * 0.5)
    J2, _, _ = _sweep(engine, bg)
    engine.update_species(HI=g["HI"])
    J, _, route = _sweep(engine, bg)
    print(f"{name}, {mode}: half HI then back ({route}): identical {np.array_equal(J, ref)}")
    assert route == default
    assert not np.array_equal(J2, ref)
    assert np.array_equal(J, ref)
    engine.set_tuning(amr_batch=64)       # the 192 directions make 32 groups (<= 8 of one zone): 4 batches of 8
    J, n, route = _sweep(engine, bg)
    print(f"{name}, {mode}: amr_batch=64 ({route}): identical {np.array_equal(J, ref)}")
    assert n == nref and np.array_equal(J, ref)
    engine.set_tuning(amr_batch=0)
    a, na, _ = _sweep(engine, bg, rays=ALL[:96])
    b, nb, _ = _sweep(engine, bg, rays=ALL[96:])
    err = rel_err(a + b, ref)
    print(f"{name}, {mode}: directions 0-95 + 96-191 vs all: rel L-inf {err:.3e}")
    assert na + nb == nref
    assert err < 1e-13


# ---- 4. neighbour threading at size -------------------------------------------------------------------------------
@pytest.mark.parametrize("grid,combos", [("g64", (0, 1, 2, 3, 4, 5, 6, 7)), ("g128", (0, 3, 5, 6))])
def test_neighbour_threading_bit_exact_at_size(rt, engine, oracle, request, grid, combos):
    """the upstream leaf of every leaf and ray (xy, yz, xz) for one direction of each reflection combination named
    (128^3 + 2: every axis once reflected and once not), against the oracle's trace of the same direction"""
    g, bg = request.getfixturevalue(grid)
    _set(engine, g)
    og = _oracle_grid(oracle, g)
    first = {}
    for iz, rays in sorted(_zones(rt).items()):
        first.setdefault(_combo(iz), rays[0])
    for c in combos:
        ray = first[c]
        o = og.diffuse(bg["uvb"], bg["beta"], ray_begin=ray, ray_end=ray + 1, trace_ray=ray)
        assert o["status"] == 0
        nb = engine.neighbours(3, ray)
        assert engine.device_error() == 0
        diff = int(np.count_nonzero(nb != o["nb"]))
        print(f"{grid} neighbours, combination {c}, direction {ray}: {diff} entries differ")
        assert diff == 0, (grid, c, ray)


# ---- 5. emission at size ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_emission_64cube_amr3_all_directions_vs_oracle(rt, engine, g64, e64, mode):
    """the streamed kernel's emissive instantiation against the oracle with the emission definition applied"""
    g, bg = g64
    eta, o = e64
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    J, nseg, route = _sweep(engine, bg)
    err = rel_err(J, o["J"])
    print(f"emission 64^3 + 3 levels x 192 vs oracle, {mode}, {route}: rel L-inf {err:.3e}")
    assert route == "streamed"
    assert nseg == o["nseg"]
    assert err < TOL


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_emission_128cube_amr2_two_directions_per_zone_vs_oracle(rt, engine, g128, rays48, e128_48, mode):
    """the per-wave kernel's emissive instantiation (FAST: 8-blocks register cap); bars as without emission"""
    g, bg = g128
    eta, o = e128_48
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    J, nseg, route = _sweep(engine, bg, rays=rays48)
    err = rel_err(J, o["J"])
    print(f"emission 128^3 + 2 levels x {rays48.size} vs oracle, {mode}, {route}: rel L-inf {err:.3e}")
    assert route == "per-wave"
    assert nseg == o["nseg"]
    assert err < (TOL if mode == "faithful" else 1e-8)


def test_emission_128cube_amr2_streamed_equals_per_wave(rt, engine, g128):
    g, bg = g128
    _set(engine, g)
    engine.set_emission(_eta(g, bg["uvb"], bg["beta"], 129))
    for mode in ("fast", "faithful"):
        engine.set_math(_mode(rt, mode))
        engine.set_tuning(amr_stream=-1)
        Jw, nw, rw = _sweep(engine, bg)
        engine.set_tuning(amr_stream=1)
        Js, ns, rs = _sweep(engine, bg)
        print(f"emission 128^3 + 2 levels x 192, {mode}: {rs} vs {rw}: identical {np.array_equal(Js, Jw)}, "
              f"rel L-inf {rel_err(Js, Jw):.3e}")
        assert rw == "per-wave" and rs == "streamed"
        assert ns == nw and np.array_equal(Js, Jw)


# ---- 6. strongly unbalanced grid at size --------------------------------------------------------------------------
def test_strongly_unbalanced_grid_at_size(rt, engine, oracle, gunb):
    """waves by dependency depth on a grid that violates the 2:1 balance everywhere around the box: one direction of
    every zone against the oracle, and both routes over all 192 directions"""
    g, bg = gunb
    rays = _per_zone(rt, 1)
    o = _oracle(_oracle_grid(oracle, g), g, bg, rays)
    _set(engine, g)
    for mode in ("faithful", "fast"):
        engine.set_math(_mode(rt, mode))
        engine.set_tuning(amr_stream=-1)
        J, nseg, route = _sweep(engine, bg, rays=rays)
        err = rel_err(J, o["J"])
        print(f"unbalanced 64^3 + 3 levels x {rays.size} vs oracle, {mode}, {route}: rel L-inf {err:.3e}")
        assert nseg == o["nseg"]
        assert err < (TOL if mode == "faithful" else 1e-8)
        full, nfull, default = _sweep(engine, bg)
        res = {default: full}
        for stream in (0, 1):
            engine.set_tuning(amr_stream=stream)
            J, n, route = _sweep(engine, bg)
            assert route == ("streamed" if stream else "per-wave") and n == nfull
            res[route] = J
        print(f"unbalanced 64^3 + 3 levels x 192, {mode}: default route {default}, streamed vs per-wave identical "
              f"{np.array_equal(res['streamed'], res['per-wave'])}")
        assert np.array_equal(res["streamed"], res["per-wave"]) and np.array_equal(full, res["per-wave"])


# ---- 7. properties at size, no oracle -----------------------------------------------------------------------------
def test_128cube_amr2_properties(rt, engine, g128):
    g, bg = g128
    uvb = bg["uvb"]
    _set(engine, g)
    J, _, route = _sweep(engine, bg)
    assert route == "per-wave"
    assert np.isfinite(J).all() and (J >= 0).all()
    for gi in range(3):
        print(f"128^3 + 2 levels, group {gi}: max J / (uvb 192 w) = {J[gi].max() / (uvb[gi] * 192 * W192):.15f}")
        assert J[gi].max() <= uvb[gi] * 192 * W192 * (1 + 1e-12)        # absorption only: J <= background
    J2, _, _ = _sweep(engine, dict(bg, uvb=uvb * 0.25))
    print(f"128^3 + 2 levels, uvb / 4: identical to J / 4 {np.array_equal(J2, J * 0.25)}")
    assert np.array_equal(J2, J * 0.25)                                 # a power of two scales exactly
    z = np.zeros(g["level"].size)
    engine.update_species(z, z, z)
    for mode in ("fast", "faithful"):
        engine.set_math(_mode(rt, mode))
        J0, _, _ = _sweep(engine, bg)
        err = max(rel_err(J0[gi], np.full(J0.shape[1], uvb[gi] * 192 * W192)) for gi in range(3))
        print(f"128^3 + 2 levels, no absorber, {mode}: rel L-inf vs uvb 192 w {err:.3e}")
        assert err < 1e-13
