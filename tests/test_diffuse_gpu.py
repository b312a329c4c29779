"""GPU parity tests of the diffuse sweep: CUDA path through the C-ABI vs the CPU oracle on the same seeded inputs
(bit-exact traversal, <= 1e-9 relative on Jmean), plus size-independent properties at BASELINE.json sizes."""
import numpy as np
import pytest

from conftest import rel_err
from radiativetransfer_b200 import workloads as W

pytestmark = pytest.mark.gpu
TOL = 1e-9  # BASELINE.json north_star: relative L-infinity on per-cell mean intensity, fp64


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


def _oracle_J(oracle, g, bg, **kw):
    og = oracle.OracleGrid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])
    o = og.diffuse(bg["uvb"], bg["beta"], **kw)
    assert o["status"] == 0
    return o


@pytest.mark.parametrize("n,seed", [(1, 1), (2, 2), (5, 3), (16, 4), (31, 5), (32, 6), (33, 7), (48, 8)])
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_uniform_parity_vs_oracle(rt, engine, oracle, uvbg, n, seed, mode):
    g = W.uniform_grid(n, seed=seed)
    engine.set_math(rt.MATH_FAST if mode == "fast" else rt.MATH_FAITHFUL)
    _set(engine, g)
    J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    o = _oracle_J(oracle, g, uvbg)
    assert nseg == o["nseg"]                      # identical traversal: same number of ray-cell segments
    assert rel_err(J, o["J"]) < TOL, rel_err(J, o["J"])


@pytest.mark.parametrize("slots,graph,pdl", [(1, 0, 1), (5, 1, 1), (24, 1, 0), (2, 0, 0),
                                             (32, 1, 1), (0, 1, 0), (0, 0, 1), (7, 0, 0)])
def test_uniform_result_independent_of_launch_tuning(rt, engine, oracle, uvbg, slots, graph, pdl):
    g = W.uniform_grid(20, seed=11)
    _set(engine, g)
    engine.set_tuning(slots=slots, graph=graph, pdl=pdl)
    J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    J2, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])   # second call replays the cached plan / graph
    assert np.array_equal(J, J2)
    o = _oracle_J(oracle, g, uvbg)
    assert rel_err(J, o["J"]) < TOL


@pytest.mark.parametrize("n", [20, 31, 32, 33, 47, 48])
def test_cells_per_thread_and_block_size_do_not_change_a_bit(rt, engine, oracle, uvbg, n):
    """FAST arithmetic: one or two cells of a layer per thread (the upper cell takes the row hand-over from registers
    instead of recomputing it), 8 / 4 / 2 rows per block: identical bits, odd and even row counts, rows of exactly one
    31-cell strip (31), a last strip of one cell (32) and other ragged last strips"""
    g = W.uniform_grid(n, seed=n)
    _set(engine, g)
    ref = None
    for cells, warps in ((1, 8), (2, 8), (2, 4), (2, 2), (1, 2), (2, 8), (0, 0)):
        # dirs_per_task fixed: how the planner cuts zones into tasks (the summation order) may depend on the other knobs
        engine.set_tuning(cells=cells, block_warps=warps, dirs_per_task=8)
        J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        if ref is None:
            ref = J
            assert rel_err(J, _oracle_J(oracle, g, uvbg)["J"]) < TOL
        assert np.array_equal(J, ref), (cells, warps)
    # a direction shard (few zone tasks per launch) takes the automatic small blocks
    engine.set_tuning(cells=0, block_warps=0, dirs_per_task=0)
    rays = np.arange(40, 64, dtype=np.int32)
    Ja, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=rays)
    engine.set_tuning(cells=1, block_warps=8)
    Jb, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=rays)
    assert rel_err(Ja, Jb) < 1e-13        # the zone pieces (summation order) may be cut differently


def test_uniform_optically_thick_and_thin_extremes(rt, engine, oracle, uvbg):
    # optically thick: per-segment tau up to ~450, intensities underflow to zero deep inside
    g = W.uniform_grid(24, seed=12, tau_lo=1e-3, tau_hi=150.0)
    _set(engine, g)
    o = _oracle_J(oracle, g, uvbg)
    for mode in (rt.MATH_FAITHFUL, rt.MATH_FAST):
        engine.set_math(mode)
        J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        assert rel_err(J, o["J"], floor=1e-250) < TOL
    # per-segment tau up to ~900: Iout = Iin*exp(-tau) passes through the SUBNORMAL range, where the reference's
    # log(Iin/Iout) sees only the few bits Iout has left while Jseg ~ Iin/tau is still a normal number.  FAITHFUL
    # mode reproduces that artefact; FAST mode returns the smooth value (documented in segment_math.cuh), so it is
    # only held to the cells the artefact does not reach.
    g = W.uniform_grid(24, seed=12, tau_lo=1e-3, tau_hi=300.0)
    _set(engine, g)
    o = _oracle_J(oracle, g, uvbg)
    engine.set_math(rt.MATH_FAITHFUL)
    J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert rel_err(J, o["J"], floor=1e-250) < TOL
    engine.set_math(rt.MATH_FAST)
    J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert rel_err(J, o["J"], floor=1e-250) < 1e-5
    assert np.quantile(np.abs(J - o["J"]) / np.maximum(o["J"], 1e-250), 0.99) < TOL
    # optically thin: per-cell tau down to 1e-7, i.e. per-segment tau down to ~1e-12.  The reference's
    # (Iin-Iout)/log(Iin/Iout) amplifies a 1-ulp difference between two libm exp() implementations by
    # ~1.1e-16/tau_segment, so in this regime the reference value is itself only defined to ~1e-6 and neither
    # arithmetic mode can be expected to match to 1e-9 (SURVEY.md section 7, "ill-conditioned log-mean").
    g = W.uniform_grid(24, seed=13, tau_lo=1e-7, tau_hi=1e-2)
    _set(engine, g)
    o = _oracle_J(oracle, g, uvbg)
    for mode in (rt.MATH_FAITHFUL, rt.MATH_FAST):
        engine.set_math(mode)
        J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        print("thin-limit rel err", mode, rel_err(J, o["J"]))
        assert rel_err(J, o["J"]) < 1e-5


def test_zero_opacity_known_answer(rt, engine, uvbg):
    n = 40
    g = W.uniform_grid(n, seed=1)
    g["HI"][:] = 0; g["HeI"][:] = 0; g["HeII"][:] = 0
    _set(engine, g)
    w = float(np.float32(1) / np.float32(192))
    for mode in (rt.MATH_FAITHFUL, rt.MATH_FAST):
        engine.set_math(mode)
        J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        for gi in range(3):
            assert np.allclose(J[gi], uvbg["uvb"][gi] * 192 * w, rtol=1e-14, atol=0)


def test_direction_subsets_match_oracle_and_add_up(rt, engine, oracle, uvbg):
    g = W.uniform_grid(16, seed=13)
    _set(engine, g)
    from radiativetransfer_b200 import sharding
    shards = sharding.shard_directions(4, nx=16)
    total = np.zeros((3, 16 ** 3))
    for s in shards:
        J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=s)
        total += J
    full, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert np.allclose(total, full, rtol=1e-13, atol=0)
    # a contiguous shard against the oracle's ray range
    J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=np.arange(40, 75, dtype=np.int32))
    o = _oracle_J(oracle, g, uvbg, ray_begin=40, ray_end=75)
    assert nseg == o["nseg"] and rel_err(J, o["J"]) < TOL
    # an empty shard is legal and returns zeros
    J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=np.zeros(0, dtype=np.int32))
    assert nseg == 0 and not J.any()


def test_golden_fixture(rt, engine, uvbg):
    import os
    from conftest import ROOT
    f = np.load(os.path.join(ROOT, "tests", "golden", "diffuse_uniform_12.npz"))
    g = W.uniform_grid(12, seed=2024)
    assert np.array_equal(g["HI"], f["HI"])
    _set(engine, g)
    J, nseg = engine.diffuse(f["uvb"], f["beta"])
    assert nseg == int(f["nseg"])
    assert rel_err(J, f["J"]) < TOL


def test_full_size_properties_128(rt, engine, uvbg):
    # BASELINE config 2 size: 128^3 x 192 directions; properties that need no oracle run
    n = 128
    g = W.uniform_grid(n, seed=1)
    _set(engine, g)
    J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert nseg > 1.8 * n ** 3 * 192
    w = float(np.float32(1) / np.float32(192))
    assert (J >= 0).all() and np.isfinite(J).all()
    for gi in range(3):
        assert J[gi].max() <= uvbg["uvb"][gi] * 192 * w * (1 + 1e-12)   # absorption only: J <= background
    # linearity in the boundary intensity: scaling by a power of two is exact in fp64
    J2, _ = engine.diffuse(uvbg["uvb"] * 0.25, uvbg["beta"])
    assert np.array_equal(J2, J * 0.25)
    # faithful and fast arithmetic agree within the parity tolerance at full size
    engine.set_math(rt.MATH_FAITHFUL)
    Jf, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert rel_err(J, Jf) < TOL
    # update_species followed by a sweep equals a fresh grid with those species
    engine.set_math(rt.MATH_FAST)
    engine.update_species(HI=g["HI"] * 0.5)
    J3, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    g2 = dict(g); g2["HI"] = g["HI"] * 0.5
    _set(engine, g2)
    J4, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert np.array_equal(J3, J4)
    assert (J3 >= J - 1e-40).all()                                       # less absorber, more light


def test_device_resident_call_and_rates(rt, engine, uvbg):
    import torch
    g = W.uniform_grid(16, seed=21)
    _set(engine, g)
    Jh, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    Jd = torch.zeros(3, 16 ** 3, dtype=torch.float64, device="cuda:0")
    s = torch.cuda.current_stream().cuda_stream
    engine.diffuse_device(uvbg["uvb"], uvbg["beta"], Jd.data_ptr(), stream=s)
    torch.cuda.synchronize()
    assert engine.device_error() == 0
    assert np.array_equal(Jd.cpu().numpy(), Jh)
    k = torch.zeros(3, 16 ** 3, dtype=torch.float64, device="cuda:0")
    engine.diffuse_rates_device(Jd.data_ptr(), uvbg["ksi24"], uvbg["ksi25"], uvbg["ksi26"],
                                k[0].data_ptr(), k[1].data_ptr(), k[2].data_ptr(), stream=s)
    torch.cuda.synchronize()
    fp = 4.0 * W.PI
    k24 = fp * Jh[0] * uvbg["ksi24"][0] + fp * Jh[1] * uvbg["ksi24"][1] + fp * Jh[2] * uvbg["ksi24"][2]
    assert np.allclose(k[0].cpu().numpy(), k24, rtol=1e-14)
    assert np.allclose(k[1].cpu().numpy(), fp * Jh[2] * uvbg["ksi25"][0], rtol=1e-14)


def test_bad_arguments(rt, engine, uvbg):
    with pytest.raises(rt.RTB200Error):
        engine.diffuse(uvbg["uvb"], uvbg["beta"])                 # no grid yet
    g = W.uniform_grid(4, seed=1)
    with pytest.raises(rt.RTB200Error):
        engine.set_grid(4, g["level"][:-1], g["HI"][:-1])         # not n^3 leaves
    _set(engine, g)
    with pytest.raises(rt.RTB200Error):
        engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=np.array([192], dtype=np.int32))


def _oracle_threads(nleaf, want):
    """host threads for the threaded oracle: every thread sweeps a private copy of the octree (~260 B per leaf)"""
    import os
    import psutil
    return int(max(1, min(want, os.cpu_count() or 1, (0.5 * psutil.virtual_memory().available) // (260.0 * nleaf))))


def test_config2_full_128cube_192dir_vs_oracle(rt, engine, oracle, uvbg):
    """BASELINE config 2 at its full size against the oracle: 128^3 uniform grid (seed 1, the bench workload's grid),
    all 192 directions, both arithmetic modes.  The oracle runs on all host threads (each thread its own directions on a
    private octree; ~7.4e8 segment updates)."""
    n = 128
    g = W.uniform_grid(n, seed=1)
    og = oracle.OracleGrid(n, g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])
    o = og.diffuse_mt(uvbg["uvb"], uvbg["beta"], np.arange(192, dtype=np.int32), nthreads=_oracle_threads(n ** 3, 32))
    assert o["status"] == 0
    _set(engine, g)
    for mode in (rt.MATH_FAST, rt.MATH_FAITHFUL):
        engine.set_math(mode)
        J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        assert nseg == o["nseg"]
        err = rel_err(J, o["J"])
        print(f"128^3 x 192 vs oracle, math mode {mode}: rel L-inf {err:.3e}")
        assert err < TOL
    # the photo-rates that consume J (equiSources.f90:3546-3553), from the oracle's J with numpy
    import torch
    engine.set_math(rt.MATH_FAST)
    Jd = torch.zeros(3, n ** 3, dtype=torch.float64, device="cuda")
    K = torch.zeros(3, n ** 3, dtype=torch.float64, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    engine.diffuse_device(uvbg["uvb"], uvbg["beta"], Jd.data_ptr(), stream=s)
    engine.diffuse_rates_device(Jd.data_ptr(), uvbg["ksi24"], uvbg["ksi25"], uvbg["ksi26"], K[0].data_ptr(),
                                K[1].data_ptr(), K[2].data_ptr(), stream=s)
    torch.cuda.synchronize()
    fourpi = 4.0 * float(np.float32(3.141592654))
    Jo = o["J"]
    k24 = fourpi * Jo[0] * uvbg["ksi24"][0] + fourpi * Jo[1] * uvbg["ksi24"][1] + fourpi * Jo[2] * uvbg["ksi24"][2]
    k25 = fourpi * Jo[2] * uvbg["ksi25"][0]
    k26 = fourpi * Jo[1] * uvbg["ksi26"][0] + fourpi * Jo[2] * uvbg["ksi26"][1]
    Kh = K.cpu().numpy()
    assert rel_err(Kh[0], k24) < TOL and rel_err(Kh[1], k25) < TOL and rel_err(Kh[2], k26) < TOL


def test_headline_256cube_direction_subset_vs_oracle(rt, engine, oracle, uvbg):
    """The benchmarked configuration (256^3 uniform, seed 1 = bench.py's grid): a subset of directions that covers all
    three sweep axes and both signs, swept by the oracle and by the GPU (`rays=`).  Each direction is ~3.1e7 segment
    updates on the oracle.

    FAITHFUL (the reference's operation sequence) must meet the 1e-9 bar on the subset itself.  FAST evaluates the same
    quantity without the reference's exp -> divide -> log round trip, whose own rounding noise is ~1.1e-16 / tau per
    segment: in a sum over only 8 directions that noise of the REFERENCE shows in cells that one direction dominates
    (measured: 2.3e-9 in the worst cell), in the full 192-direction solve it averages out (1.3e-10 at 128^3, see
    test_config2_full_128cube_192dir_vs_oracle; 256^3 x 192: tests marked slow below).  So FAST is held to 1e-8 on the
    subset, and to 1e-9 against FAITHFUL on the full 192-direction solve at this size."""
    n = 256
    g = W.uniform_grid(n, seed=1)
    rays = np.array([0, 37, 74, 111, 148, 185, 30, 67], dtype=np.int32)
    zones = {rt.direction(3, int(r))[0] for r in rays}
    assert len(zones) >= 6
    og = oracle.OracleGrid(n, g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])
    o = og.diffuse_mt(uvbg["uvb"], uvbg["beta"], rays, nthreads=_oracle_threads(n ** 3, rays.size))
    assert o["status"] == 0
    del og
    _set(engine, g)
    errs = {}
    for name, mode in (("faithful", rt.MATH_FAITHFUL), ("fast", rt.MATH_FAST)):
        engine.set_math(mode)
        J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"], rays=rays)
        assert nseg == o["nseg"]
        errs[name] = rel_err(J, o["J"])
    print(f"256^3 x {rays.size} directions vs oracle: rel L-inf {errs}")
    assert errs["faithful"] < TOL
    assert errs["fast"] < 1e-8
    engine.set_math(rt.MATH_FAITHFUL)
    Jf, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    engine.set_math(rt.MATH_FAST)
    Jq, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    full = rel_err(Jq, Jf)
    print(f"256^3 x 192 directions, FAST vs FAITHFUL: rel L-inf {full:.3e}")
    assert full < TOL


@pytest.mark.skipif(not __import__("os").environ.get("RTB_SLOW_TESTS"), reason="~4 minutes of host time: set RTB_SLOW_TESTS=1")
def test_headline_256cube_full_192dir_vs_oracle(rt, engine, oracle, uvbg):
    """the benchmarked solve in full against the oracle on all host threads (5.96e9 segment updates on the CPU);
    the result of the last run is recorded in profiles/"""
    n = 256
    g = W.uniform_grid(n, seed=1)
    og = oracle.OracleGrid(n, g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])
    o = og.diffuse_mt(uvbg["uvb"], uvbg["beta"], np.arange(192, dtype=np.int32), nthreads=_oracle_threads(n ** 3, 32))
    assert o["status"] == 0
    del og
    _set(engine, g)
    for name, mode in (("fast", rt.MATH_FAST), ("faithful", rt.MATH_FAITHFUL)):
        engine.set_math(mode)
        J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        assert nseg == o["nseg"]
        err = rel_err(J, o["J"])
        print(f"256^3 x 192 vs oracle, {name}: rel L-inf {err:.3e}")
        assert err < TOL


def test_fast_exponential_error_budget(rt, engine):
    """FAST arithmetic's exponential (64-entry table, degree-4 polynomial) against libm in extended precision: the
    truncation error DESIGN.md 4.1 budgets (7.2e-12 of 1 - e^-tau, 3.9e-14 of e^-tau per segment), over the whole range
    of optical depths incl. the table's interval ends, tiny tau (no cancellation in 1 - e^-tau) and the clamp"""
    import ctypes as C
    rng = np.random.default_rng(5)
    tau = np.concatenate([10.0 ** rng.uniform(-12, 2.8, 200000), np.arange(0, 4096) * (np.log(2) / 128),
                          np.array([0.0, 1e-300, 5e-324, 700.0, 707.0, 1e4])])
    e, ome = np.empty_like(tau), np.empty_like(tau)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert engine.L.rtb200_debug_fast_exp(engine.h, int(tau.size), p(tau), p(e), p(ome)) == 0
    t = tau.astype(np.longdouble)
    ref_e, ref_ome = np.exp(-t), -np.expm1(-t)
    ok = tau <= 700.0                                   # beyond: clamped (e^-tau < 1e-304 multiplies an intensity)
    rel_e = np.abs((e[ok] - ref_e[ok]) / ref_e[ok]).astype(np.float64)
    nz = ok & (tau > 0)
    rel_ome = np.abs((ome[nz] - ref_ome[nz]) / ref_ome[nz]).astype(np.float64)
    assert rel_e.max() < 1e-13, rel_e.max()
    assert rel_ome.max() < 1e-11, rel_ome.max()
    assert ome[tau == 0.0][0] == 0.0 and e[tau == 0.0][0] == 1.0
    assert np.all(e[~ok] >= 0) and np.all(e[~ok] < 1e-300) and np.all(ome[~ok] == 1.0)
