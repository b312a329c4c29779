"""GPU tests of isotropic scattering by source iteration (DESIGN.md 4.7): sigma = 0 reproduces the plain sweep bit for
bit on every route, a fixed number of iterations agrees with the oracle's restatement (tests/scattering_oracle.py), the
stopping rule takes the oracle's decisions, the fixed points of a conservative box and of a thermal + scattering
equilibrium hold on the device, the launch routes agree bit for bit, the state is handled as the emission's, and device
groups of one and two GPUs (threads and processes) agree with the single context."""
import os
import subprocess
import sys

import numpy as np
import pytest

import scattering_oracle
from conftest import rel_err
from radiativetransfer_b200 import workloads as W
from test_scattering_oracle import NDIR, FIXED_POINT_BAR, conservative_case, equilibrium_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"faithful": 1e-9, "fast": 1e-8}
K = 4


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


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


def _sigma(g, beta, seed, lo=0.1, hi=0.9):
    """seeded scattering with albedo sigma / (kappa + sigma) from lo to hi per cell"""
    rng = np.random.default_rng(seed)
    kap = np.maximum(_kappa(g, beta), 1e-30)
    a = rng.uniform(lo, hi, size=kap.shape)
    return kap * a / (1.0 - a)


def _eta(g, uvb, beta, seed):
    rng = np.random.default_rng(seed + 1000)
    kap = np.maximum(_kappa(g, beta), 1e-30)
    return 10.0 ** rng.uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap


BALANCED = W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4)


def _corner(level, x, y, z, size):
    return (level < 3) & (x < 0.26) & (y < 0.26) & (z > 0.74)


UNBALANCED = W.nested_grid(4, 3, _corner, seed=6)


def _mode(rt, name):
    return rt.MATH_FAITHFUL if name == "faithful" else rt.MATH_FAST


# ---- 1. sigma = 0 is the plain sweep ---------------------------------------------------------------------------------
@pytest.mark.parametrize("emission", [False, True])
@pytest.mark.parametrize("cells,transpose,graph", [(1, 0, 1), (2, 1, 1), (2, 1, 0), (1, 1, 0)])
def test_zero_sigma_uniform_bit_for_bit(rt, engine, uvbg, cells, transpose, graph, emission):
    g = W.uniform_grid(40, seed=3)
    engine.set_tuning(cells=cells, transpose_z=transpose, graph=graph)
    _set(engine, g)
    if emission:
        engine.set_emission(_eta(g, uvbg["uvb"], uvbg["beta"], 3))
    ref, n0 = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    engine.set_scattering(np.zeros((3, g["level"].size)), max_iterations=50, tolerance=1e-9)
    J, n1 = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert engine.last_scattering() == {"iterations": 2, "residual": 0.0}
    assert n1 == 2 * n0 and np.array_equal(J, ref)


@pytest.mark.parametrize("emission", [False, True])
@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("stream", [0, 1])
@pytest.mark.parametrize("grid", ["balanced", "unbalanced"])
def test_zero_sigma_nested_bit_for_bit(rt, engine, uvbg, mode, stream, grid, emission):
    g = BALANCED if grid == "balanced" else UNBALANCED
    engine.set_math(_mode(rt, mode))
    engine.set_tuning(amr_stream=stream)
    _set(engine, g)
    uvb = uvbg["uvb"] * 1e-3
    if emission:
        engine.set_emission(_eta(g, uvb, uvbg["beta"], 4))
    ref, n0 = engine.diffuse(uvb, uvbg["beta"])
    engine.set_scattering(np.zeros((3, g["level"].size)), max_iterations=50, tolerance=1e-9)
    J, n1 = engine.diffuse(uvb, uvbg["beta"])
    assert engine.last_scattering() == {"iterations": 2, "residual": 0.0}
    assert n1 == 2 * n0 and np.array_equal(J, ref)


# ---- 2. / 3. against the oracle ---------------------------------------------------------------------------------------
def _vs_oracle(rt, engine, g, uvb, beta, sigma, eta, mode, max_iter, tol):
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    engine.set_scattering(sigma, max_iterations=max_iter, tolerance=tol)
    J, nseg = engine.diffuse(uvb, beta)
    s = engine.last_scattering()
    o = scattering_oracle.grid(g).solve(uvb, beta, eta, sigma, max_iter, tol)
    assert o["status"] == 0
    return J, nseg, s, o


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("n", [1, 16, 33, 48])
def test_uniform_fixed_iterations_vs_oracle(rt, engine, uvbg, mode, n):
    g = W.uniform_grid(n, seed=30 + n)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    J, nseg, s, o = _vs_oracle(rt, engine, g, uvb, beta, _sigma(g, beta, n), _eta(g, uvb, beta, n), mode, K, 0.0)
    err = rel_err(J, o["J"])
    print(f"scattering uniform n={n} {mode} K={K}: rel err {err:.3e}, residual {s['residual']:.3e} (oracle {o['residual']:.3e})")
    assert s["iterations"] == K and o["iterations"] == K
    assert nseg == o["nseg"]
    assert err < TOL[mode], err


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("grid", ["balanced", "unbalanced"])
def test_nested_fixed_iterations_vs_oracle(rt, engine, uvbg, mode, grid):
    g = BALANCED if grid == "balanced" else UNBALANCED
    uvb, beta = uvbg["uvb"] * 1e-3, uvbg["beta"]
    J, nseg, s, o = _vs_oracle(rt, engine, g, uvb, beta, _sigma(g, beta, 7), _eta(g, uvb, beta, 7), mode, K, 0.0)
    err = rel_err(J, o["J"])
    print(f"scattering nested {grid} {mode} K={K}: rel err {err:.3e}")
    assert s["iterations"] == K and nseg == o["nseg"]
    assert err < TOL[mode], err


@pytest.mark.parametrize("grid", ["uniform", "balanced"])
def test_stopping_rule_takes_the_oracles_decision(rt, engine, uvbg, grid):
    g = W.uniform_grid(12, seed=41) if grid == "uniform" else BALANCED
    uvb, beta = uvbg["uvb"] * (1.0 if grid == "uniform" else 1e-3), uvbg["beta"]
    # albedo 0.001 - 0.004: successive residuals fall by 200x or more, so a tolerance at the geometric mean of two of
    # them is 10x away from both and the decision is not borderline
    sigma, eta = _sigma(g, beta, 41, 0.001, 0.004), _eta(g, uvb, beta, 41)
    hist = scattering_oracle.grid(g).solve(uvb, beta, eta, sigma, 8, 0.0)["history"]
    k = next(i for i in range(2, len(hist)) if hist[i] < 1e-4)
    tol = float(np.sqrt(hist[k - 1] * hist[k]))
    assert hist[k - 1] / tol >= 10 and tol / hist[k] >= 10, hist
    J, _, s, o = _vs_oracle(rt, engine, g, uvb, beta, sigma, eta, "faithful", 60, tol)
    print(f"stopping {grid}: residuals {['%.2e' % h for h in hist]}, tol {tol:.3e}, oracle {o['iterations']} iterations, "
          f"GPU {s['iterations']}, residual {s['residual']:.3e} / {o['residual']:.3e}, err {rel_err(J, o['J']):.3e}")
    assert o["iterations"] == k + 1
    assert s["iterations"] == o["iterations"]
    assert s["residual"] <= tol
    assert rel_err(J, o["J"]) < 1e-9


# ---- 4. fixed points on the device -----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_conservative_box_on_the_device(rt, engine, uvbg, mode):
    g, sigma = conservative_case(n=16)
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_scattering(sigma, max_iterations=400, tolerance=1e-12)
    J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    s = engine.last_scattering()
    want = uvbg["uvb"][:, None] * (NDIR * float(np.float32(1.0) / np.float32(NDIR)))
    err = float(np.max(np.abs(J - want) / want))
    print(f"conservative box 16^3 {mode}: {s['iterations']} iterations, residual {s['residual']:.3e}, err {err:.3e}")
    assert s["residual"] <= 1e-12 and np.all(np.isfinite(J)) and np.all(J >= 0)
    assert err < FIXED_POINT_BAR, err


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_equilibrium_on_the_device(rt, engine, uvbg, mode):
    g, S, eta, sigma = equilibrium_case(uvbg, n=16)
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    engine.set_scattering(sigma, max_iterations=600, tolerance=1e-12)
    J, _ = engine.diffuse(S, uvbg["beta"])
    s = engine.last_scattering()
    want = S[:, None] * (NDIR * float(np.float32(1.0) / np.float32(NDIR)))
    err = float(np.max(np.abs(J - want) / want))
    print(f"equilibrium 16^3 {mode}: {s['iterations']} iterations, residual {s['residual']:.3e}, err {err:.3e}")
    assert s["residual"] <= 1e-12 and np.all(np.isfinite(J)) and np.all(J >= 0)
    assert err < FIXED_POINT_BAR, err


# ---- 5. scaling and linearity ----------------------------------------------------------------------------------------
def test_quarter_sources_give_a_quarter_and_linearity(rt, engine, uvbg):
    # per-cell tau >= 0.3: the reference log-mean's rounding on short corner-clip segments breaks linearity at the 1e-12
    # level for thinner cells, and the iteration carries it on (the oracle itself: 3.7e-12 at tau >= 0.1, K = 6)
    g = W.uniform_grid(20, seed=51, tau_lo=0.3)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    sigma, eta = _sigma(g, beta, 51), _eta(g, uvb, beta, 51)
    _set(engine, g)
    engine.set_math(_mode(rt, "faithful"))
    engine.set_scattering(sigma, max_iterations=200, tolerance=1e-10)
    engine.set_emission(eta)
    J, _ = engine.diffuse(uvb, beta)
    it = engine.last_scattering()["iterations"]
    engine.set_emission(eta * 0.25)
    Jq, _ = engine.diffuse(uvb * 0.25, beta)
    assert engine.last_scattering()["iterations"] == it
    assert np.array_equal(Jq, J * 0.25)
    engine.set_scattering(sigma, max_iterations=6, tolerance=0.0)
    engine.set_emission(eta)
    both, _ = engine.diffuse(uvb, beta)
    only_eta, _ = engine.diffuse(np.zeros(3), beta)
    engine.set_emission(None)
    only_uvb, _ = engine.diffuse(uvb, beta)
    err = float(np.max(np.abs(both - (only_uvb + only_eta)) / np.abs(both)))
    print(f"linearity K=6: {err:.3e}")
    assert err < 1e-12, err


# ---- 6. routes and repeats -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_uniform_routes_agree_bit_for_bit(rt, engine, uvbg, mode):
    g = W.uniform_grid(40, seed=61)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(_eta(g, uvb, beta, 61))
    engine.set_scattering(_sigma(g, beta, 61), max_iterations=3, tolerance=0.0)
    ref, _ = engine.diffuse(uvb, beta)
    for kw in (dict(cells=2), dict(graph=0), dict(pdl=0), dict(cells=1, graph=1, pdl=1)):
        engine.set_tuning(**kw)
        J, _ = engine.diffuse(uvb, beta)
        assert np.array_equal(J, ref), kw
    # without the z-major copy the zone tasks keep their order and the accumulators are summed in another order, which
    # changes the plain sweep's last bits too: the same to rounding (3.0e-13 measured, FAITHFUL, 3 iterations), and bit
    # for bit from one call to the next
    engine.set_tuning(transpose_z=0)
    a, _ = engine.diffuse(uvb, beta)
    b, _ = engine.diffuse(uvb, beta)
    print(f"transpose_z 0 vs 1, {mode}, K=3: {rel_err(a, ref):.3e}")
    assert np.array_equal(a, b) and rel_err(a, ref) < 1e-12, rel_err(a, ref)
    engine.set_tuning(transpose_z=1)
    # odd and even iteration counts, twice in a row
    for k in (3, 4):
        engine.set_scattering(_sigma(g, beta, 61), max_iterations=k, tolerance=0.0)
        a, _ = engine.diffuse(uvb, beta)
        b, _ = engine.diffuse(uvb, beta)
        assert np.array_equal(a, b)
    import torch
    d = torch.zeros((3, g["level"].size), dtype=torch.float64, device="cuda:0")
    engine.diffuse_device(uvb, beta, d.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert engine.last_scattering()["iterations"] == 4
    assert np.array_equal(d.cpu().numpy(), b)


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("grid", ["balanced", "unbalanced"])
def test_nested_routes_agree_bit_for_bit(rt, engine, uvbg, mode, grid):
    g = BALANCED if grid == "balanced" else UNBALANCED
    uvb, beta = uvbg["uvb"] * 1e-3, uvbg["beta"]
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(_eta(g, uvb, beta, 62))
    sigma = _sigma(g, beta, 62)
    outs = {}
    for k in (3, 4):   # the streamed sweep alternates the record sign sweep by sweep
        engine.set_scattering(sigma, max_iterations=k, tolerance=0.0)
        for stream in (0, 1):
            engine.set_tuning(amr_stream=stream, amr_batch=0)
            a, _ = engine.diffuse(uvb, beta)
            b, _ = engine.diffuse(uvb, beta)
            assert np.array_equal(a, b), (k, stream)
            outs[(k, stream)] = a
        engine.set_tuning(amr_stream=-1, amr_batch=64)
        c, _ = engine.diffuse(uvb, beta)
        engine.set_tuning(amr_batch=0)
        assert np.array_equal(outs[(k, 0)], outs[(k, 1)]), k
        assert np.array_equal(c, outs[(k, 0)]), k


# ---- 7. state ------------------------------------------------------------------------------------------------------
def test_state_handling(rt, engine, uvbg):
    g = W.uniform_grid(16, seed=71)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    N = g["level"].size
    _set(engine, g)
    plain, n0 = engine.diffuse(uvb, beta)
    assert engine.last_scattering() == {"iterations": 0, "residual": 0.0}
    sigma = _sigma(g, beta, 71)
    engine.set_scattering(sigma, max_iterations=5, tolerance=0.0)
    J5, n5 = engine.diffuse(uvb, beta)
    assert n5 == 5 * n0 and engine.last_scattering()["iterations"] == 5
    assert engine.last_stats()["algorithmic_bytes"] == 96.0 * N * NDIR * 5
    # refused: negative, NaN, Inf entries, a count < 1, a negative or NaN tolerance; the previous state stays
    for bad_s, mi, tol in ((-sigma, 5, 0.0), (np.where(np.arange(3 * N).reshape(3, N) == 7, np.nan, sigma), 5, 0.0),
                           (np.where(np.arange(3 * N).reshape(3, N) == 9, np.inf, sigma), 5, 0.0),
                           (sigma, 0, 0.0), (sigma, 5, -1e-9), (sigma, 5, float("nan"))):
        with pytest.raises(rt.RTB200Error):
            engine.set_scattering(bad_s, max_iterations=mi, tolerance=tol)
        J, _ = engine.diffuse(uvb, beta)
        assert np.array_equal(J, J5) and engine.last_scattering()["iterations"] == 5
    # a direction subset is refused while scattering is set
    with pytest.raises(rt.RTB200Error) as e:
        engine.diffuse(uvb, beta, rays=np.arange(10))
    assert e.value.status == 12
    # update_species keeps the scattering, set_grid clears it
    engine.update_species(HI=g["HI"])
    J, _ = engine.diffuse(uvb, beta)
    assert np.array_equal(J, J5)
    engine.set_scattering(None)
    J, n = engine.diffuse(uvb, beta)
    assert np.array_equal(J, plain) and n == n0 and engine.last_scattering()["iterations"] == 0
    engine.set_scattering(sigma, max_iterations=5, tolerance=0.0)
    _set(engine, g)
    J, n = engine.diffuse(uvb, beta)
    assert np.array_equal(J, plain) and n == n0


# ---- 8. device groups ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ndev", [1, 2])
@pytest.mark.parametrize("tol", [0.0, 1e-9])
def test_device_group_equals_plain_context(rt, uvbg, ndev, tol):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = W.uniform_grid(24, seed=81)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    sigma, eta = _sigma(g, beta, 81), _eta(g, uvb, beta, 81)
    t = rt.Transport(device=0, math=rt.MATH_FAITHFUL)
    _set(t, g)
    t.set_emission(eta)
    t.set_scattering(sigma, max_iterations=K if tol == 0 else 100, tolerance=tol)
    ref, n0 = t.diffuse(uvb, beta)
    s0 = t.last_scattering()
    t.close()
    m = rt.Transport(devices=list(range(ndev)), math=rt.MATH_FAITHFUL)
    try:
        _set(m, g)
        m.set_emission(eta)
        m.set_scattering(sigma, max_iterations=K if tol == 0 else 100, tolerance=tol)
        J, n1 = m.diffuse(uvb, beta)
        s1 = m.last_scattering()
        bad = sigma.copy(); bad[0, -1] = -1.0
        with pytest.raises(rt.RTB200Error):
            m.set_scattering(bad, max_iterations=K, tolerance=tol)
        with pytest.raises(rt.RTB200Error):
            m.diffuse(uvb, beta, rays=np.arange(10))
        # the resident call leaves the same J in the slabs
        m.diffuse_resident(uvb, beta)
        m.sync()
        assert m.last_scattering()["iterations"] == s1["iterations"]
        for local in range(ndev):
            off, cnt, Js, _, _ = m.slab_get(local)
            assert np.array_equal(Js, J[:, off:off + cnt])
        J2, _ = m.diffuse(uvb, beta)
    finally:
        m.close()
    print(f"group of {ndev}, tol {tol}: {s1['iterations']} iterations (single {s0['iterations']}), "
          f"residual {s1['residual']:.3e} / {s0['residual']:.3e}, err {rel_err(J, ref):.3e}")
    assert n0 == n1 and s1["iterations"] == s0["iterations"]
    assert (np.array_equal(J, ref) and s1["residual"] == s0["residual"]) if ndev == 1 else rel_err(J, ref) < 1e-12
    assert np.array_equal(J2, J)


def test_one_process_per_gpu(rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "scattering_rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:]); sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0
    assert r.stdout.count("RANK-OK") == 2


# ---- 9. the benchmark size -------------------------------------------------------------------------------------------
@pytest.mark.skipif(not os.environ.get("RTB_SLOW_TESTS"), reason="minutes of host time: set RTB_SLOW_TESTS=1")
def test_128cube_three_iterations_vs_oracle(rt, engine, uvbg):
    g = W.uniform_grid(128, seed=91)
    uvb, beta = uvbg["uvb"], uvbg["beta"]
    J, nseg, s, o = _vs_oracle(rt, engine, g, uvb, beta, _sigma(g, beta, 91), _eta(g, uvb, beta, 91), "fast", 3, 0.0)
    err = rel_err(J, o["J"])
    print(f"scattering 128^3 fast K=3: rel err {err:.3e}")
    assert nseg == o["nseg"] and err < TOL["fast"], err
