"""Uniform sweep, lane packing: the layer positions run end to end across rows and warps, so a warp can span several
rows and a row can start mid-warp.  Grids whose rows are much shorter than a warp (n = 1, 2, 5, 7) put many row starts
in one warp; one- and two-cell threads and every block size must give the same bits, and those bits the oracle's
values, in FAST and (one-cell) FAITHFUL arithmetic, with and without emission."""
import numpy as np
import pytest

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


@pytest.mark.parametrize("n", [1, 2, 5, 7])
def test_short_rows_cells_and_block_size_do_not_change_a_bit(rt, engine, oracle, uvbg, n):
    g = W.uniform_grid(n, seed=100 + n)
    _set(engine, g)
    og = oracle.OracleGrid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], box_size=g["box_size"])
    o = og.diffuse(uvbg["uvb"], uvbg["beta"])
    assert o["status"] == 0
    ref = None
    for cells, warps in ((1, 8), (2, 8), (2, 2), (1, 2), (2, 4)):
        engine.set_tuning(cells=cells, block_warps=warps, dirs_per_task=8)
        J, nseg = engine.diffuse(uvbg["uvb"], uvbg["beta"])
        assert nseg == o["nseg"]
        if ref is None:
            ref = J
            assert rel_err(J, o["J"]) < TOL
        assert np.array_equal(J, ref), (cells, warps)
    engine.set_math(rt.MATH_FAITHFUL)
    J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert rel_err(J, o["J"]) < TOL


@pytest.mark.parametrize("n", [2, 5])
def test_short_rows_zero_emission_is_the_plain_sweep(rt, engine, uvbg, n):
    g = W.uniform_grid(n, seed=200 + n)
    _set(engine, g)
    J, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    engine.set_emission(np.zeros((3, n ** 3)))
    Je, _ = engine.diffuse(uvbg["uvb"], uvbg["beta"])
    assert np.array_equal(J, Je)
