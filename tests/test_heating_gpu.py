"""GPU tests of the heating pass (DESIGN.md 4.10): with heating set, J and nseg are those of the same call without it;
all five fields equal tests/heating_oracle.py applied to the returned J and the grid's species, bit for bit, on every
route (FAST / FAITHFUL, uniform / nested, emission, per-leaf sigma, dust modes with and without albedo, Ng and warm
start, a direction subset, the device call on a caller stream); the fields are linear in J; a transparent box gives the
closed form; the state is handled as documented; device groups of one and two GPUs (threads and processes) agree with
the oracle of their own J and with the single context."""
import os
import subprocess
import sys

import numpy as np
import pytest

import heating_oracle as HO
from conftest import rel_err
from radiativetransfer_b200 import workloads as W
from test_dust_gpu import ALBEDO, BALANCED, UNBALANCED, _beta_dust, _dusty, _eta, _uvb
from test_scattering_oracle import NDIR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUBSET = np.array([3, 40, 77, 101, 150, 188], dtype=np.int32)
_CACHE = {}


@pytest.fixture(scope="module")
def rt(build_product):
    import radiativetransfer_b200 as rt
    return rt


@pytest.fixture(scope="module")
def heat(uvbg):
    return W.uvb_heating(uvbg["table"], uvbg["alpha"])


@pytest.fixture()
def engine(rt):
    t = rt.Transport(device=0)
    yield t
    t.close()


def _grid(name):
    if name not in _CACHE:
        _CACHE[name] = {"u32": lambda: _dusty(W.uniform_grid(32, seed=32), 32), "balanced": lambda: BALANCED,
                        "unbalanced": lambda: UNBALANCED}[name]()
    return _CACHE[name]


def _set(t, g):
    t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])


# ---- 1. no effect on J -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gname", ["u32", "balanced", "unbalanced"])
def test_no_effect_on_J(rt, engine, uvbg, heat, gname):
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    _set(engine, g)
    for dust in (None, (2, ALBEDO)):
        if dust:
            engine.set_dust(dust[0], _beta_dust(g, uvbg, dust[0]), albedo=dust[1], max_iterations=3, tolerance=0.0)
        engine.set_heating(None)
        engine.diffuse(uvb, beta)   # the first call after a change of the grid or the medium builds the plans
        J0, n0 = engine.diffuse(uvb, beta)
        l0 = engine.last_stats()["launches"]
        engine.set_heating(*heat)
        J1, n1 = engine.diffuse(uvb, beta)
        l1 = engine.last_stats()["launches"]
        engine.set_heating(None)
        J2, n2 = engine.diffuse(uvb, beta)
        l2 = engine.last_stats()["launches"]
        assert np.array_equal(J1, J0) and np.array_equal(J2, J0) and n0 == n1 == n2
        assert l1 == l0 + 1 and l2 == l0, (l0, l1, l2)


# ---- 2. exact definition ---------------------------------------------------------------------------------------------
CASES = {
    "u32-fast": dict(grid="u32", math="fast"),
    "u32-faithful": dict(grid="u32", math="faithful"),
    "balanced-fast": dict(grid="balanced", math="fast"),
    "unbalanced-faithful": dict(grid="unbalanced", math="faithful"),
    "emission": dict(grid="u32", math="fast", emission=True),
    "sigma": dict(grid="balanced", math="fast", sigma=True),
    "dust1-absorbing": dict(grid="u32", math="faithful", dust=(1, (0.0, 0.0, 0.0))),
    "dust2-absorbing": dict(grid="balanced", math="fast", dust=(2, (0.0, 0.0, 0.0))),
    "dust1-albedo-ng-warm": dict(grid="u32", math="fast", dust=(1, ALBEDO), accel=True),
    "dust2-albedo-nested": dict(grid="balanced", math="faithful", dust=(2, ALBEDO)),
    "subset-dust1": dict(grid="u32", math="fast", dust=(1, (0.0, 0.0, 0.0)), rays=SUBSET),
}


@pytest.mark.parametrize("case", list(CASES))
def test_fields_are_the_definition(rt, engine, uvbg, heat, case):
    c = CASES[case]
    g = _grid(c["grid"])
    N = g["level"].size
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    engine.set_math(rt.MATH_FAITHFUL if c["math"] == "faithful" else rt.MATH_FAST)
    _set(engine, g)
    if c.get("emission"):
        engine.set_emission(_eta(g, uvb, beta, 3))
    if c.get("sigma"):
        engine.set_scattering(np.full((3, N), 1e-3 / g["box_size"]) * g["nx"], max_iterations=4, tolerance=0.0)
    mode, albedo, bd = 0, (0.0, 0.0, 0.0), None
    if "dust" in c:
        mode, albedo = c["dust"]
        bd = _beta_dust(g, uvbg, mode)
        engine.set_dust(mode, bd, albedo=albedo, max_iterations=9 if c.get("accel") else 3, tolerance=0.0)
    if c.get("accel"):
        engine.set_scattering_acceleration(ng=True, warm_start=True)
    engine.set_heating(*heat)
    for call in range(2 if c.get("accel") else 1):   # the second call starts warm
        J, _ = engine.diffuse(uvb, beta, rays=c.get("rays"))
        H = HO.fields(engine.last_heating())
        want = HO.heating(J, g, heat[0], heat[1], mode, bd, albedo)
        assert np.array_equal(H, want), [rel_err(H[f], want[f], floor=1e-300) for f in range(5)]
    if c.get("accel"):
        a = engine.last_scattering_acceleration()
        assert a["warm_start"] and a["extrapolations"] >= 1, a
    assert all(np.any(H[f] > 0) for f in range(4)) and (np.any(H[4] > 0) if mode else np.all(H[4] == 0))


def test_device_call_on_a_caller_stream(rt, engine, uvbg, heat):
    import torch
    g = _grid("u32")
    N = g["level"].size
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    bd = _beta_dust(g, uvbg, 2)
    _set(engine, g)
    engine.set_dust(2, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
    engine.set_heating(*heat)
    ptr, off, cnt, stride = engine.heating_device()
    assert (off, cnt, stride) == (0, N, N) and ptr
    Jd = torch.zeros((3, N), dtype=torch.float64, device="cuda:0")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        engine.diffuse_device(uvb, beta, Jd.data_ptr(), stream=s.cuda_stream)
        view = torch.as_tensor(_CudaArray(ptr, (5, stride)), device="cuda:0")
        H = view.clone()
    s.synchronize()
    J = Jd.cpu().numpy()
    want = HO.heating(J, g, heat[0], heat[1], 2, bd, ALBEDO)
    assert np.array_equal(H.cpu().numpy(), want)
    assert np.array_equal(HO.fields(engine.last_heating()), want)


class _CudaArray:
    """a zero-copy view of a library-owned device buffer of doubles"""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = dict(shape=shape, typestr="<f8", data=(int(ptr), False), version=2, strides=None)


# ---- 3. linearity ----------------------------------------------------------------------------------------------------
def test_direction_shards_add_up(rt, engine, uvbg, heat):
    g = _grid("u32")
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    _set(engine, g)
    engine.set_dust(1, _beta_dust(g, uvbg, 1))
    engine.set_heating(*heat)
    engine.diffuse(uvb, beta)
    full = HO.fields(engine.last_heating())
    a = np.arange(0, NDIR, 2, dtype=np.int32)
    engine.diffuse(uvb, beta, rays=a)
    Ha = HO.fields(engine.last_heating())
    engine.diffuse(uvb, beta, rays=np.setdiff1d(np.arange(NDIR, dtype=np.int32), a))
    Hb = HO.fields(engine.last_heating())
    err = rel_err(Ha + Hb, full, floor=1e-300)
    print(f"shards add up: rel err {err:.2e}")
    assert err < 1e-13, err


# ---- 4. transparent box ----------------------------------------------------------------------------------------------
def test_transparent_box(rt, engine, uvbg, heat):
    g = _dusty(W.uniform_grid(16, seed=21), 21)
    uvb = uvbg["uvb"]
    _set(engine, g)
    engine.set_heating(*heat)
    J, _ = engine.diffuse(uvb, np.zeros(9))
    H = HO.fields(engine.last_heating())
    Jw = uvb[:, None] * (NDIR * float(np.float32(1.0) / np.float32(NDIR)))
    gam = np.asarray(heat[0])
    for s in range(3):
        want = HO.FOUR_PI * sum(Jw[k] * gam[k, s] for k in range(3))
        err = rel_err(H[s], want, floor=1e-300)
        print(f"transparent box Gamma_{s}: rel err {err:.2e}")
        assert err < 1e-13, (s, err)
    assert np.array_equal(H[4], np.zeros(g["level"].size))


# ---- 5. state --------------------------------------------------------------------------------------------------------
def test_state_handling(rt, engine, uvbg, heat):
    import ctypes as C
    g = _dusty(W.uniform_grid(16, seed=31), 31)
    N = g["level"].size
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    gamma, width = heat
    _set(engine, g)
    with pytest.raises(rt.RTB200Error):
        engine.last_heating()                         # not set
    engine.set_heating(gamma, width)
    with pytest.raises(rt.RTB200Error) as e:
        engine.last_heating()                         # no call yet
    assert e.value.status == 12
    J, _ = engine.diffuse(uvb, beta)
    H0 = HO.fields(engine.last_heating())
    assert np.array_equal(H0, HO.heating(J, g, gamma, width))
    bad = []
    for v in (-1e-30, np.nan, np.inf):
        gm = np.array(gamma, dtype=np.float64).ravel(); gm[4] = v
        wd = np.array(width, dtype=np.float64); wd[2] = v
        bad += [(gm, width), (gamma, wd)]
    for gm, wd in bad:
        with pytest.raises(rt.RTB200Error):
            engine.set_heating(gm, wd)
        assert np.array_equal(HO.fields(engine.last_heating()), H0)   # the previous state stays
    gm = np.ascontiguousarray(gamma, dtype=np.float64)
    assert engine.L.rtb200_grid_set_heating(engine.h, gm.ctypes.data_as(C.c_void_p), None) == 12
    J, _ = engine.diffuse(uvb, beta)
    assert np.array_equal(HO.fields(engine.last_heating()), H0)
    # a failed call leaves no fields
    engine.set_dust(1, _beta_dust(g, uvbg, 1), albedo=ALBEDO, max_iterations=2, tolerance=0.0)
    with pytest.raises(rt.RTB200Error):
        engine.diffuse(uvb, beta, rays=SUBSET)
    with pytest.raises(rt.RTB200Error) as e:
        engine.last_heating()
    assert e.value.status == 12
    engine.set_dust(0)
    # update_species keeps the setting and the next call follows the new species
    HI2 = g["HI"] * np.random.default_rng(5).uniform(0.5, 2.0, N)
    engine.update_species(HI=HI2)
    J, _ = engine.diffuse(uvb, beta)
    assert np.array_equal(HO.fields(engine.last_heating()), HO.heating(J, dict(g, HI=HI2), gamma, width))
    # set_grid clears it
    plain = engine.last_stats()["launches"] - 1
    _set(engine, g)
    engine.diffuse(uvb, beta)
    engine.diffuse(uvb, beta)
    assert engine.last_stats()["launches"] == plain
    with pytest.raises(rt.RTB200Error):
        engine.last_heating()
    with pytest.raises(rt.RTB200Error):
        engine.heating_device()
    # clearing frees the buffer
    engine.set_heating(gamma, width)
    engine.set_heating(None)
    with pytest.raises(rt.RTB200Error):
        engine.heating_device()


# ---- 6. device groups ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gname", ["u32", "balanced"])
@pytest.mark.parametrize("ndev", [1, 2])
def test_device_group(rt, uvbg, heat, gname, ndev):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    bd = _beta_dust(g, uvbg, 2)
    out = {}
    for kind in ("single", "group"):
        t = rt.Transport(device=0) if kind == "single" else rt.Transport(devices=list(range(ndev)))
        try:
            _set(t, g)
            t.set_dust(2, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
            t.set_heating(*heat)
            J, _ = t.diffuse(uvb, beta)
            H = HO.fields(t.last_heating())
            out[kind] = (J, H)
            if kind == "group":
                assert np.array_equal(H, HO.heating(J, g, heat[0], heat[1], 2, bd, ALBEDO))
                slab = t.info()["slab"]
                for local in range(ndev):
                    ptr, off, cnt, stride = t.heating_device(local)
                    assert stride == slab and ptr
                with pytest.raises(rt.RTB200Error):
                    t.heating_device(ndev)
        finally:
            t.close()
    (J1, H1), (Jg, Hg) = out["single"], out["group"]
    if ndev == 1:
        assert np.array_equal(Jg, J1) and np.array_equal(Hg, H1)
    else:
        assert rel_err(Hg, H1, floor=1e-300) < 1e-13


@pytest.mark.parametrize("ndev", [1, 2])
def test_resident_call_with_chemistry_uses_the_swept_species(rt, uvbg, heat, ndev):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = _dusty(W.nested_grid(6, 2, W.central_box_refine(0.2, 0.7, levels=2), seed=5, tau_lo=1e-2, tau_hi=2.0), 5)
    N = g["level"].size
    uvb, beta = uvbg["uvb"] * 1e-3, uvbg["beta"]
    bd = _beta_dust(g, uvbg, 1)
    ksi = np.concatenate([uvbg["ksi24"], uvbg["ksi25"], uvbg["ksi26"]])
    grp = rt.Transport(devices=list(range(ndev)))
    try:
        _set(grp, g)
        grp.set_rate_tables(W.rate_tables(500))
        grp.set_temperature(10.0 ** np.random.default_rng(2).uniform(4.0, 4.1, N))
        grp.set_dust(1, bd, albedo=ALBEDO, max_iterations=3, tolerance=0.0)
        grp.set_heating(*heat)
        grp.diffuse_resident(uvb, beta, ksi=ksi, chemistry=True)
        grp.sync()
        H = HO.fields(grp.last_heating())
        J = np.zeros((3, N))
        for local in range(ndev):
            off, cnt, Js, _, _ = grp.slab_get(local)
            J[:, off:off + cnt] = Js
        assert not np.array_equal(grp.get_species()[0], g["HI"])   # chemistry changed HI after the pass
    finally:
        grp.close()
    assert np.array_equal(H, HO.heating(J, g, heat[0], heat[1], 1, bd, ALBEDO))


def test_one_process_per_gpu(rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", os.path.join(ROOT, "tests", "heating_rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:]); sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0
    assert r.stdout.count("RANK-OK") == 2
