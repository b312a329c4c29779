"""GPU tests of the accelerated source iteration (DESIGN.md 4.9): flags set and cleared again leave every route bit for
bit as before, Ng at a fixed sweep count agrees with the numpy restatement (tests/ng_oracle.py) on uniform and nested
grids, the stopping rule takes its decisions, the two-mode cell lands on its limit, the warm start follows its lifetime,
unknown flags are refused, the clamp keeps a thick dust grid's sources >= 0, accelerated scattering dust converges to the
dust oracle's answer, and device groups of one and two GPUs (threads, processes, the resident call with chemistry) agree
with the single context."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import dust_oracle
import ng_oracle
import scattering_oracle
from conftest import rel_err
from radiativetransfer_b200 import workloads as W
from test_dust_gpu import _beta_dust, _dusty
from test_scattering_gpu import BALANCED, UNBALANCED, _eta, _kappa, _mode, _set, _sigma

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"faithful": 1e-9, "fast": 1e-8}
_CACHE = {}


@pytest.fixture(scope="module")
def rt(build_product):
    import radiativetransfer_b200 as rt
    return rt


@pytest.fixture()
def engine(rt):
    t = rt.Transport(device=0)
    yield t
    t.close()


def _grid(name):
    return {"u16": lambda: W.uniform_grid(16, seed=16), "u33": lambda: W.uniform_grid(33, seed=33),
            "balanced": lambda: BALANCED, "unbalanced": lambda: UNBALANCED}[name]()


def _uvb(uvbg, g):
    return uvbg["uvb"] * (1.0 if g["level"].max() == 0 else 1e-3)   # nested grids: inside the refined-leaf guard


def _oracle(gname, g, uvb, beta, sigma, eta, max_iter, tol, ng=True):
    key = (gname, max_iter, tol, ng)
    if key not in _CACHE:
        o = ng_oracle.solve_accelerated(scattering_oracle.grid(g), uvb, beta, eta, sigma, max_iter, tol, ng=ng)
        assert o["status"] == 0
        _CACHE[key] = o
    return _CACHE[key]


# ---- 1. flags set and cleared are the plain solve --------------------------------------------------------------------
ROUTES = [("uniform-cells1", dict(cells=1, transpose_z=0), "u33", False), ("uniform-cells2", dict(cells=2), "u33", False),
          ("amr_stream0", dict(amr_stream=0), "balanced", False), ("amr_stream1", dict(amr_stream=1), "balanced", False),
          ("group1", None, "u33", True), ("group1-nested", None, "balanced", True)]


@pytest.mark.parametrize("route,tuning,gname,group", ROUTES, ids=[r[0] for r in ROUTES])
def test_flags_cleared_are_bit_for_bit_the_plain_solve(rt, uvbg, route, tuning, gname, group):
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    t = rt.Transport(devices=[0]) if group else rt.Transport(device=0)
    try:
        if tuning:
            t.set_tuning(**tuning)
        _set(t, g)
        t.set_emission(_eta(g, uvb, beta, 11))
        t.set_scattering(_sigma(g, beta, 11), max_iterations=9, tolerance=0.0)
        ref, n0 = t.diffuse(uvb, beta)
        t.set_scattering_acceleration(ng=True, warm_start=True)
        acc, _ = t.diffuse(uvb, beta)
        assert t.last_scattering_acceleration()["extrapolations"] >= 1 and not np.array_equal(acc, ref)
        t.set_scattering_acceleration()
        J, n = t.diffuse(uvb, beta)
        assert t.last_scattering_acceleration() == {"extrapolations": 0, "warm_start": False}
        assert np.array_equal(J, ref) and n == n0
    finally:
        t.close()


# ---- 2. against the numpy restatement at a fixed count ---------------------------------------------------------------
@pytest.mark.parametrize("K", [8, 9])
@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("gname,stream", [("u16", -1), ("u33", -1), ("balanced", 0), ("balanced", 1), ("unbalanced", -1)])
def test_fixed_count_vs_oracle(rt, engine, uvbg, gname, stream, mode, K):
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    sigma, eta = _sigma(g, beta, 21), _eta(g, uvb, beta, 21)
    engine.set_math(_mode(rt, mode))
    engine.set_tuning(amr_stream=stream)
    _set(engine, g)
    engine.set_emission(eta)
    engine.set_scattering(sigma, max_iterations=K, tolerance=0.0)
    engine.set_scattering_acceleration(ng=True)
    J, nseg = engine.diffuse(uvb, beta)
    acc = engine.last_scattering_acceleration()
    again, _ = engine.diffuse(uvb, beta)
    o = _oracle(gname, g, uvb, beta, sigma, eta, K, 0.0)
    err = rel_err(J, o["J"])
    print(f"Ng {gname} stream {stream} {mode} K={K}: {acc['extrapolations']} extrapolations (oracle "
          f"{o['extrapolations']}), rel err {err:.3e}")
    assert engine.last_scattering()["iterations"] == K and nseg == o["nseg"]
    assert acc == {"extrapolations": o["extrapolations"], "warm_start": False} and o["extrapolations"] == (K - 1) // 4
    assert np.array_equal(again, J)
    assert err < TOL[mode], err


@pytest.mark.parametrize("gname", ["u16", "balanced"])
def test_stopping_rule_takes_the_oracles_decision(rt, engine, uvbg, gname):
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    sigma, eta = _kappa(g, beta), _eta(g, uvb, beta, 31)   # albedo 0.5
    hist = _oracle(gname, g, uvb, beta, sigma, eta, 40, 0.0)["history"]
    # a tolerance at least 2x away from the residual that meets it and from every residual before it
    tol = next(float(np.sqrt(min(hist[:k]) * hist[k])) for k in range(5, len(hist)) if min(hist[:k]) >= 4.0 * hist[k])
    o = _oracle(gname, g, uvb, beta, sigma, eta, 100, tol)
    engine.set_math(rt.MATH_FAITHFUL)
    _set(engine, g)
    engine.set_emission(eta)
    engine.set_scattering(sigma, max_iterations=100, tolerance=tol)
    engine.set_scattering_acceleration(ng=True)
    J, _ = engine.diffuse(uvb, beta)
    s, acc = engine.last_scattering(), engine.last_scattering_acceleration()
    print(f"Ng stopping {gname}: tol {tol:.3e}, oracle {o['iterations']} sweeps / {o['extrapolations']} extrapolations, "
          f"GPU {s['iterations']} / {acc['extrapolations']}, err {rel_err(J, o['J']):.3e}")
    assert s["iterations"] == o["iterations"] and acc["extrapolations"] == o["extrapolations"]
    assert s["residual"] <= tol and rel_err(J, o["J"]) < 1e-9


def test_two_error_modes_land_on_the_limit(rt, engine, uvbg):
    g = W.uniform_grid(1, seed=2, tau_lo=5.0, tau_hi=5.0)
    kap = _kappa(g, uvbg["beta"])[:, 0]
    eta_th = np.array([[3.0e-44], [1.0e-45], [4.0e-46]])
    engine.set_math(rt.MATH_FAITHFUL)
    _set(engine, g)
    for frac in ((0.3, 0.7, 0.0), (0.9, 0.5, 0.0)):
        sigma = np.array(frac)[:, None] * kap[:, None]
        # b = dJ / deta of the cell from two emissive sweeps with the extinction kappa + sigma
        engine.set_scattering(sigma, max_iterations=1, tolerance=0.0)
        engine.set_scattering_acceleration()
        engine.set_emission(eta_th)
        J1 = engine.diffuse(np.zeros(3), uvbg["beta"])[0][:, 0]
        engine.set_emission(2.0 * eta_th)
        J2 = engine.diffuse(np.zeros(3), uvbg["beta"])[0][:, 0]
        want = J1 / (1.0 - sigma[:, 0] * (J2 - J1) / eta_th[:, 0])
        engine.set_emission(eta_th)
        engine.set_scattering(sigma, max_iterations=5, tolerance=0.0)
        engine.set_scattering_acceleration(ng=True)
        J, _ = engine.diffuse(np.zeros(3), uvbg["beta"])
        err = float(np.max(np.abs(J[:, 0] - want) / want))
        print(f"two-mode cell {frac}: {err:.3e}")
        assert engine.last_scattering_acceleration()["extrapolations"] == 1
        assert err <= 1e-10, err


# ---- 3. state -------------------------------------------------------------------------------------------------------
def test_warm_start_lifetime(rt, engine, uvbg):
    g = W.uniform_grid(16, seed=41)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    sigma = _kappa(g, beta)
    _set(engine, g)
    engine.set_scattering(sigma, max_iterations=200, tolerance=1e-8)
    cold, _ = engine.diffuse(uvb, beta)
    n_cold = engine.last_scattering()["iterations"]
    engine.set_scattering_acceleration(warm_start=True)
    J, _ = engine.diffuse(uvb, beta)   # the plain call before it stored its J
    assert engine.last_scattering_acceleration() == {"extrapolations": 0, "warm_start": True}
    assert engine.last_scattering()["iterations"] <= 2 and rel_err(J, cold) < 1e-7
    # update_species and new settings keep the stored J
    engine.update_species(HI=g["HI"])
    engine.set_scattering(sigma * 1.01, max_iterations=200, tolerance=1e-8)
    engine.diffuse(uvb, beta)
    n_warm = engine.last_scattering()["iterations"]
    assert engine.last_scattering_acceleration()["warm_start"] and n_warm < n_cold
    # a refused call drops it
    with pytest.raises(rt.RTB200Error):
        engine.diffuse(uvb, beta, rays=np.arange(10))
    engine.diffuse(uvb, beta)
    assert not engine.last_scattering_acceleration()["warm_start"]
    # clearing the scattering drops it
    engine.diffuse(uvb, beta)
    assert engine.last_scattering_acceleration()["warm_start"]
    engine.set_scattering(None)
    engine.set_scattering(sigma, max_iterations=200, tolerance=1e-8)
    J, _ = engine.diffuse(uvb, beta)
    assert not engine.last_scattering_acceleration()["warm_start"] and np.array_equal(J, cold)
    # set_grid resets the flags and drops the J
    _set(engine, g)
    engine.set_scattering(sigma, max_iterations=200, tolerance=1e-8)
    engine.diffuse(uvb, beta)
    engine.diffuse(uvb, beta)
    assert not engine.last_scattering_acceleration()["warm_start"]
    assert engine.last_scattering()["iterations"] == n_cold


def test_unknown_flags_are_refused_and_the_flags_stay(rt, engine, uvbg):
    g = W.uniform_grid(12, seed=42)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    _set(engine, g)
    engine.set_scattering(_kappa(g, beta), max_iterations=9, tolerance=0.0)
    engine.set_scattering_acceleration(ng=True)
    for bad in (4, 5, -1, 1 << 30):
        assert engine.L.rtb200_grid_set_scattering_acceleration(engine.h, bad) == 12   # RTB200_ERR_ARG
    engine.diffuse(uvb, beta)
    assert engine.last_scattering_acceleration() == {"extrapolations": 2, "warm_start": False}
    n, w = C.c_int32(-1), C.c_int32(-1)
    assert engine.L.rtb200_last_scattering_acceleration(engine.h, C.byref(n), C.byref(w)) == 0 and n.value == 2


def test_thick_dust_keeps_sources_non_negative(rt, engine, uvbg):
    g = _dusty(W.uniform_grid(32, seed=32), 32)
    _set(engine, g)
    engine.set_dust(2, _beta_dust(g, uvbg, 2, scale="median"), albedo=(0.9, 0.9, 0.9), max_iterations=60, tolerance=1e-8)
    engine.set_scattering_acceleration(ng=True, warm_start=True)
    for _ in range(2):
        J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        assert engine.device_error() == 0
        assert np.all(np.isfinite(J)) and np.all(J >= 0)
    print(f"thick dust albedo 0.9: {engine.last_scattering()}, {engine.last_scattering_acceleration()}")


def test_scattering_dust_converges_to_the_dust_oracle(rt, engine, uvbg):
    g = _dusty(BALANCED, 4)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    bd = _beta_dust(g, uvbg, 2)
    kd = dust_oracle.dust_kd(g, bd, 2)
    o = dust_oracle.grid(g).solve(uvb, beta, None, kd, 0.5 * kd, 300, 1e-11)
    assert o["status"] == 0
    _set(engine, g)
    engine.set_math(rt.MATH_FAITHFUL)
    engine.set_dust(2, bd, albedo=(0.5, 0.5, 0.5), max_iterations=300, tolerance=1e-11)
    engine.set_scattering_acceleration(ng=True, warm_start=True)
    J, _ = engine.diffuse(uvb, beta)
    s, acc = engine.last_scattering(), engine.last_scattering_acceleration()
    err = rel_err(J, o["J"])
    print(f"dust albedo 0.5: oracle {o['iterations']} plain sweeps, GPU {s['iterations']} with {acc['extrapolations']} "
          f"extrapolations, rel err {err:.3e}")
    assert acc["extrapolations"] >= 1 and s["iterations"] < o["iterations"]
    assert err < 1e-9, err


# ---- 4. device groups ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ndev", [1, 2])
@pytest.mark.parametrize("gname,tol", [("u33", 0.0), ("u33", 1e-9), ("balanced", 1e-9)])
def test_device_group_equals_plain_context(rt, uvbg, ndev, gname, tol):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = _grid(gname)
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    sigma, eta = _sigma(g, beta, 51), _eta(g, uvb, beta, 51)
    mi = 9 if tol == 0 else 200

    def run(t):
        _set(t, g)
        t.set_emission(eta)
        t.set_scattering(sigma, max_iterations=mi, tolerance=tol)
        t.set_scattering_acceleration(ng=True, warm_start=True)
        out = []
        for scale in (1.0, 1.01):   # the second call starts warm
            t.set_scattering(sigma * scale, max_iterations=mi, tolerance=tol)
            J, n = t.diffuse(uvb, beta)
            out.append((J, n, t.last_scattering()["iterations"], t.last_scattering_acceleration()))
        return out

    one = rt.Transport(device=0, math=rt.MATH_FAITHFUL)
    try:
        ref = run(one)
        J3, _ = one.diffuse(uvb, beta)
    finally:
        one.close()
    m = rt.Transport(devices=list(range(ndev)), math=rt.MATH_FAITHFUL)
    try:
        got = run(m)
        m.diffuse_resident(uvb, beta)   # a third warm call, resident: the single context's third J in the slabs
        m.sync()
        for local in range(ndev):
            off, cnt, Js, _, _ = m.slab_get(local)
            assert np.array_equal(Js, J3[:, off:off + cnt]) if ndev == 1 else rel_err(Js, J3[:, off:off + cnt]) < 1e-12
    finally:
        m.close()
    for (Jr, nr, ir, ar), (Jg, ng, ig, ag) in zip(ref, got):
        print(f"group of {ndev} {gname} tol {tol}: {ig} sweeps {ag} (single {ir} {ar}), err {rel_err(Jg, Jr):.3e}")
        assert nr == ng and ir == ig and ar == ag
        assert np.array_equal(Jg, Jr) if ndev == 1 else rel_err(Jg, Jr) < 1e-12
    assert ref[1][3]["warm_start"] and (tol == 0 or ref[1][2] < ref[0][2])


@pytest.mark.parametrize("ndev", [1, 2])
def test_device_group_failed_or_refused_call_starts_every_rank_cold(rt, uvbg, ndev):
    # a background 1e3 times too bright trips the refined-leaf intensity guard of the nested sweep in some directions,
    # i.e. on some members only; the next call must start cold on every rank alike (same collectives, same answer)
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = BALANCED
    uvb, beta = _uvb(uvbg, g), uvbg["beta"]
    sigma = _sigma(g, beta, 61)
    one = rt.Transport(device=0, math=rt.MATH_FAITHFUL)
    try:
        _set(one, g)
        one.set_scattering(sigma, max_iterations=200, tolerance=1e-9)
        cold, _ = one.diffuse(uvb, beta)
        n_cold = one.last_scattering()["iterations"]
    finally:
        one.close()
    m = rt.Transport(devices=list(range(ndev)), math=rt.MATH_FAITHFUL)
    try:
        _set(m, g)
        m.set_scattering(sigma, max_iterations=200, tolerance=1e-9)
        m.set_scattering_acceleration(warm_start=True)
        m.diffuse(uvb, beta)
        m.diffuse(uvb, beta)
        assert m.last_scattering_acceleration()["warm_start"]
        with pytest.raises(rt.RTB200Error) as e:
            m.diffuse(uvb * 1e6, beta)
        assert e.value.status == 7
        J, _ = m.diffuse(uvb, beta)
        assert m.last_scattering_acceleration() == {"extrapolations": 0, "warm_start": False}
        assert m.last_scattering()["iterations"] == n_cold
        assert np.array_equal(J, cold) if ndev == 1 else rel_err(J, cold) < 1e-12
        # a refused direction subset drops the stored J as well
        m.diffuse(uvb, beta)
        assert m.last_scattering_acceleration()["warm_start"]
        with pytest.raises(rt.RTB200Error):
            m.diffuse(uvb, beta, rays=np.arange(10))
        m.diffuse(uvb, beta)
        assert not m.last_scattering_acceleration()["warm_start"]
    finally:
        m.close()


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
    one.set_dust(1, bd, albedo=(0.5, 0.5, 0.5), max_iterations=9, tolerance=0.0)
    one.set_scattering_acceleration(ng=True, warm_start=True)
    J = torch.zeros(3, N, dtype=torch.float64, device="cuda:0")
    s = torch.cuda.current_stream(0).cuda_stream
    for _ in range(3):
        one.diffuse_device(uvb, beta, J.data_ptr(), stream=s)
        one.chemistry_device(0, J.data_ptr(), ksi=ksi, stream=s, want_change=False)
    torch.cuda.synchronize()
    acc1 = one.last_scattering_acceleration()
    ref = one.get_species()
    one.close()
    grp = rt.Transport(devices=list(range(ndev)))
    try:
        _set(grp, g)
        grp.set_rate_tables(ktab); grp.set_temperature(tgas)
        grp.set_dust(1, bd, albedo=(0.5, 0.5, 0.5), max_iterations=9, tolerance=0.0)
        grp.set_scattering_acceleration(ng=True, warm_start=True)
        for _ in range(3):
            grp.diffuse_resident(uvb, beta, ksi=ksi, chemistry=True)
        grp.sync()
        assert grp.last_scattering()["iterations"] == 9
        acc = grp.last_scattering_acceleration()
        got = grp.get_species()
    finally:
        grp.close()
    assert acc == acc1 and acc["warm_start"]
    assert not np.array_equal(ref[0], g["HI"])
    for a, b in zip(got, ref):
        assert rel_err(a, b, floor=1e-300) < 1e-9


def test_one_process_per_gpu(rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tests", "scattering_accel_rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:]); sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0
    assert r.stdout.count("RANK-OK") == 2
