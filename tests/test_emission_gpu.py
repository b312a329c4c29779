"""GPU tests of the emission extension (DESIGN.md 4.6): eta = 0 reproduces the emission-free sweep bit for bit on every
route, random eta agrees with the oracle's restatement of the definition (tests/emission_oracle.py), the equilibrium
S = eta / kappa holds on the device, and the host setter, device setter, direction subsets, streamed nested sweep and
device groups agree."""
import numpy as np
import pytest

import emission_oracle
from conftest import rel_err
from radiativetransfer_b200 import workloads as W

pytestmark = pytest.mark.gpu
TOL = 1e-9


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


def _eta(g, uvb, beta, seed):
    """seeded emission with source functions S = eta / kappa from 1e-3 to 1 of the boundary intensity"""
    rng = np.random.default_rng(seed)
    kap = np.maximum(_kappa(g, beta), 1e-30)
    return 10.0 ** rng.uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap


BALANCED = W.nested_grid(6, 2, W.central_box_refine(0.3, 0.7, levels=2), seed=4)


def _corner(level, x, y, z, size):
    return (level < 3) & (x < 0.26) & (y < 0.26) & (z > 0.74)


UNBALANCED = W.nested_grid(4, 3, _corner, seed=6)


def _mode(rt, name):
    return rt.MATH_FAITHFUL if name == "faithful" else rt.MATH_FAST


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("cells,transpose,graph", [(1, 0, 1), (2, 1, 1), (2, 1, 0), (1, 1, 0)])
def test_zero_emission_uniform_bit_for_bit(rt, engine, uvbg, mode, cells, transpose, graph):
    g = W.uniform_grid(40, seed=3)
    engine.set_math(_mode(rt, mode))
    for k, v in (("cells", cells), ("transpose_z", transpose), ("graph", graph)):
        engine.set_tuning(**{k: v})
    _set(engine, g)
    ref, n0 = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    engine.set_emission(np.zeros((3, g["level"].size)))
    J, n1 = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert n0 == n1 and np.array_equal(J, ref)


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("stream", [0, 1])
@pytest.mark.parametrize("grid", ["balanced", "unbalanced"])
def test_zero_emission_nested_bit_for_bit(rt, engine, uvbg, mode, stream, grid):
    g = BALANCED if grid == "balanced" else UNBALANCED
    engine.set_math(_mode(rt, mode))
    engine.set_tuning(amr_stream=stream)
    _set(engine, g)
    uvb = uvbg["uvb"] * 1e-3
    ref, _ = engine.diffuse(uvb, uvbg["beta"])
    engine.set_emission(np.zeros((3, g["level"].size)))
    J, _ = engine.diffuse(uvb, uvbg["beta"])
    assert np.array_equal(J, ref)


def _vs_oracle(rt, engine, oracle, g, uvb, beta, eta, mode, rays=None):
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    J, nseg = engine.diffuse(uvb, beta, rays=rays)
    og = emission_oracle.grid(g)
    og.set_emission(eta)
    if rays is None:
        o = og.diffuse(uvb, beta)
        assert o["status"] == 0
        return rel_err(J, o["J"]), nseg, o["nseg"]
    Jo, no = np.zeros_like(J), 0
    for r in rays:
        o = og.diffuse(uvb, beta, ray_begin=int(r), ray_end=int(r) + 1)
        assert o["status"] == 0
        Jo += o["J"]; no += o["nseg"]
    return rel_err(J, Jo), nseg, no


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("n", [1, 5, 16, 33, 48])
def test_uniform_random_emission_vs_oracle(rt, engine, oracle, uvbg, mode, n):
    g = W.uniform_grid(n, seed=20 + n)
    err, nseg, no = _vs_oracle(rt, engine, oracle, g, uvbg["uvb"], uvbg["beta"], _eta(g, uvbg["uvb"], uvbg["beta"], n), mode)
    print(f"emission n={n} {mode}: rel err {err:.3e}")
    assert nseg == no and err < TOL, err


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("grid", ["balanced", "unbalanced"])
def test_nested_random_emission_vs_oracle(rt, engine, oracle, uvbg, mode, grid):
    g = BALANCED if grid == "balanced" else UNBALANCED
    uvb = uvbg["uvb"] * 1e-3
    err, nseg, no = _vs_oracle(rt, engine, oracle, g, uvb, uvbg["beta"], _eta(g, uvb, uvbg["beta"], 7), mode)
    print(f"emission nested {grid} {mode}: rel err {err:.3e}")
    assert nseg == no and err < TOL, err


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_ragged_direction_subset_vs_oracle(rt, engine, oracle, uvbg, mode):
    g = W.uniform_grid(12, seed=8)
    rays = np.array([0, 3, 17, 18, 19, 64, 101, 150, 191], dtype=np.int32)
    err, nseg, no = _vs_oracle(rt, engine, oracle, g, uvbg["uvb"], uvbg["beta"], _eta(g, uvbg["uvb"], uvbg["beta"], 9),
                               mode, rays=rays)
    assert nseg == no and err < TOL, err
    err, nseg, no = _vs_oracle(rt, engine, oracle, BALANCED, uvbg["uvb"] * 1e-3, uvbg["beta"],
                               _eta(BALANCED, uvbg["uvb"] * 1e-3, uvbg["beta"], 10), mode, rays=rays)
    assert nseg == no and err < TOL, err


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_config2_size_vs_oracle(rt, engine, oracle, uvbg, mode):
    g = W.uniform_grid(128, seed=1)
    eta = _eta(g, uvbg["uvb"], uvbg["beta"], 128)
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    og = emission_oracle.grid(g)
    og.set_emission(eta)
    import os
    o = og.diffuse_mt(uvbg["uvb"], uvbg["beta"], np.arange(192, dtype=np.int32), nthreads=os.cpu_count() or 1)
    assert o["status"] == 0 and o["nseg"] == nseg
    Jo = o["J"]
    err = rel_err(J, Jo)
    print(f"emission 128^3 x 192 {mode}: rel err {err:.3e}")
    assert err < TOL, err


def _equilibrium(g, uvbg):
    n = g["level"].size
    g = dict(g, HI=np.full(n, 1.0e-4), HeI=np.zeros(n), HeII=np.zeros(n))
    S = uvbg["uvb"] * 1e-3
    eta = S[:, None] * _kappa(g, uvbg["beta"])
    return g, S, eta, S[:, None] * (192 * float(np.float32(1.0) / np.float32(192)))


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("grid", ["uniform64", "nested"])
def test_equilibrium_on_the_device(rt, engine, uvbg, mode, grid):
    g, S, eta, want = _equilibrium(W.uniform_grid(64, seed=2) if grid == "uniform64" else BALANCED, uvbg)
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(eta)
    J, _ = engine.diffuse(S, uvbg["beta"])
    err = float(np.max(np.abs(J - want) / want))
    assert err < 1e-9, err


def test_host_and_device_setters_agree_and_bad_arrays_are_refused(rt, engine, uvbg):
    import torch
    g = W.uniform_grid(24, seed=4)
    _set(engine, g)
    eta = _eta(g, uvbg["uvb"], uvbg["beta"], 4)
    engine.set_emission(eta)
    Jh, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    d = torch.tensor(eta, dtype=torch.float64, device="cuda:0").contiguous()
    engine.set_emission_device(d.data_ptr(), torch.cuda.current_stream().cuda_stream)
    Jd, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert np.array_equal(Jh, Jd)
    for bad in (float("nan"), -1e-40, float("inf")):
        b = d.clone()
        b[1, 7] = bad
        with pytest.raises(rt.RTB200Error) as e:
            engine.set_emission_device(b.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert e.value.status == 12
        host = eta.copy(); host[2, 3] = bad
        with pytest.raises(rt.RTB200Error) as e:
            engine.set_emission(host)
        assert e.value.status == 12
    J2, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert np.array_equal(J2, Jh)          # the previous emission is still in place
    engine.set_emission(None)
    J0, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    engine.set_emission(np.zeros_like(eta))
    Jz, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert np.array_equal(J0, Jz)


@pytest.mark.parametrize("grid", ["uniform", "nested"])
def test_direction_subsets_add_up(rt, engine, uvbg, grid):
    g = W.uniform_grid(20, seed=5) if grid == "uniform" else BALANCED
    uvb = uvbg["uvb"] * (1.0 if grid == "uniform" else 1e-3)
    engine.set_math(rt.MATH_FAITHFUL)
    _set(engine, g)
    engine.set_emission(_eta(g, uvb, uvbg["beta"], 5))
    J, n = engine.diffuse(uvb, uvbg["beta"])
    parts, ns = np.zeros_like(J), 0
    for lo in range(0, 192, 48):
        Jp, nsp = engine.diffuse(uvb, uvbg["beta"], rays=np.arange(lo, lo + 48, dtype=np.int32))
        parts += Jp; ns += nsp
    assert ns == n and rel_err(parts, J) < 1e-12


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_streamed_and_wave_nested_sweeps_agree_with_emission(rt, engine, uvbg, mode):
    g = BALANCED
    uvb = uvbg["uvb"] * 1e-3
    engine.set_math(_mode(rt, mode))
    _set(engine, g)
    engine.set_emission(_eta(g, uvb, uvbg["beta"], 3))
    engine.set_tuning(amr_stream=0)
    Jw, _ = engine.diffuse(uvb, uvbg["beta"])
    engine.set_tuning(amr_stream=1)
    Js, _ = engine.diffuse(uvb, uvbg["beta"])
    Js2, _ = engine.diffuse(uvb, uvbg["beta"])
    assert np.array_equal(Jw, Js) and np.array_equal(Js, Js2)


def test_last_stats_count_the_emission_read(rt, engine, uvbg):
    g = W.uniform_grid(16, seed=6)
    _set(engine, g)
    engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert engine.last_stats()["algorithmic_bytes"] == 72.0 * g["level"].size * 192
    engine.set_emission(_eta(g, uvbg["uvb"], uvbg["beta"], 6))
    engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert engine.last_stats()["algorithmic_bytes"] == 96.0 * g["level"].size * 192


@pytest.mark.parametrize("ndev", [1, 2])
def test_device_group_equals_plain_context_with_emission(rt, uvbg, ndev):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    g = W.uniform_grid(24, seed=7)
    eta = _eta(g, uvbg["uvb"], uvbg["beta"], 7)
    t = rt.Transport(device=0, math=rt.MATH_FAITHFUL)
    _set(t, g)
    t.set_emission(eta)
    ref, n0 = t.diffuse(uvbg["uvb"], uvbg["beta"])
    t.close()
    m = rt.Transport(devices=list(range(ndev)), math=rt.MATH_FAITHFUL)
    try:
        _set(m, g)
        m.set_emission(eta)
        J, n1 = m.diffuse(uvbg["uvb"], uvbg["beta"])
        bad = eta.copy(); bad[0, -1] = -1.0
        with pytest.raises(rt.RTB200Error):
            m.set_emission(bad)
        J2, _ = m.diffuse(uvbg["uvb"], uvbg["beta"])
    finally:
        m.close()
    assert n0 == n1
    assert (np.array_equal(J, ref) if ndev == 1 else rel_err(J, ref) < 1e-12)
    assert np.array_equal(J2, J)
