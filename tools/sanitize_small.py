"""small end-to-end calls of every path for compute-sanitizer (memcheck): uniform sweep (one and two cells per thread,
block sizes, both math modes), nested-grid sweep (per-wave launches and the streamed
one-launch path, several sweeps), point sources (three deposition modes, trace), a device group of one, octree build"""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import radiativetransfer_b200 as rt
from radiativetransfer_b200 import workloads as W
bg = W.uvb_background(3.0)
sp = W.synthetic_spectra()
t = rt.Transport(device=0)
g = W.uniform_grid(33, seed=1)
t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
for mode in (rt.MATH_FAST, rt.MATH_FAITHFUL):
    t.set_math(mode)
    J, nseg = t.diffuse(bg["uvb"], bg["beta"], rays=list(range(0, 192, 5)))
    print("uniform", mode, nseg, float(J.sum()))
t.set_math(rt.MATH_FAST)
for kw in (dict(cells=1), dict(cells=2), dict(cells=2, block_warps=2)):
    t.set_tuning(cells=0, block_warps=0); t.set_tuning(**kw)
    J, nseg = t.diffuse(bg["uvb"], bg["beta"], rays=list(range(0, 192, 5)))
    print("uniform", kw, nseg, float(J.sum()), t.device_error())
t.set_tuning(cells=0, block_warps=0)
gb = W.nested_grid(8, 1, W.central_box_refine(0.25, 0.75), seed=3)      # 2:1 balanced: streamed path
t.set_grid(gb["nx"], gb["level"], gb["HI"], gb["HeI"], gb["HeII"], gb["rho"], gb["abun2"], gb["box_size"])
for stream in (1, 1, 1, 0, 1):
    for mode in (rt.MATH_FAST, rt.MATH_FAITHFUL):
        t.set_math(mode); t.set_tuning(amr_stream=stream)
        J, nseg = t.diffuse(bg["uvb"] * 1e-3, bg["beta"], rays=list(range(0, 192, 3)))
        print("amr balanced stream", stream, mode, nseg, float(J.sum()), t.device_error(), t.last_stats()["launches"])
t.set_tuning(amr_stream=-1)
g = W.nested_grid(6, 2, W.central_box_refine(0.2, 0.8, levels=2), seed=4, tau_lo=1e-3, tau_hi=0.5, beta24=6.3e-18)
t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
t.set_math(rt.MATH_FAST)
J, nseg = t.diffuse(bg["uvb"], bg["beta"], rays=list(range(0, 192, 7)))
print("amr", nseg, float(J.sum()), t.device_error())
for dep in (0, 1, 2, 2):
    for mode in (rt.MATH_FAST, rt.MATH_FAITHFUL):
        t.set_math(mode); t.set_tuning(point_deposit=dep)
        r = t.point(sp, [100, 2000], [1, 2], dust_approximation=2, max_pixel_level=4)
        print("point", dep, mode, r["nseg"], float(r["rates"].sum()))
t.set_tuning(point_deposit=0)
r = t.point(sp, [100], [1], max_pixel_level=3, trace_cap=100000)
print("trace", r["nseg"], r["trace"].size)
t.close()
# a device group of one runs the whole group path (slab copies, exchange buffers, reduce kernel, slab chemistry inputs)
grp = rt.Transport(devices=[0])
grp.set_grid(gb["nx"], gb["level"], gb["HI"], gb["HeI"], gb["HeII"], gb["rho"], gb["abun2"], gb["box_size"])
J, nseg = grp.diffuse(bg["uvb"] * 1e-3, bg["beta"])
r = grp.point(sp, [10, 200], [1, 2], max_pixel_level=3)
print("group of one", nseg, float(J.sum()), r["nseg"], float(r["rates"].sum()))
grp.close()
from radiativetransfer_b200 import formats as F
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from test_formats import _random_levels
levels = _random_levels(np.random.default_rng(11), 5, True, (60, 50, 40), (16.0, 9.0, 5.0))
for lv in levels:
    for k in lv:
        lv[k] = np.asarray(lv[k], dtype=np.float32)
got = F.build_leaves_device(levels, metals=True)
print("octree build on device:", got["level"].size, "leaves")
