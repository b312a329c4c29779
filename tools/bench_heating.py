"""Cost of the heating pass (DESIGN.md 4.10), FAST arithmetic, 192 directions, dust mode 2 (albedo 0), one process, every
shape warmed up first.  Prints one JSON line per case with the card's name and power limit (read through NVML):
  * step_ms / step_heating_ms: the whole diffuse call without and with heating, alternating call by call;
  * pass_ms: the pass alone, as the difference of an empty-shard call (opacities, no directions) with and without heating,
    alternating, over --pass-reps calls each; the pass's inputs and outputs (J, species, rho, abun2, the fields) are
    104 B per leaf, 1.7 GB at 256^3, far above the 126 MB of L2 (the opacity pass just before it leaves the last ~100 MB
    of the species in L2, so pass_gbs is an upper bound);
  * pass_gbs and pass_of_copy_peak: those bytes over pass_ms, and as a fraction of the copy rate of a 4 GB
    device-to-device torch copy (read + write bytes over time) measured in the same run.

    python tools/bench_heating.py [--reps 7] [--pass-reps 40] [--cases uniform256,nested128]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_scattering import card   # noqa: E402

PASS_BYTES_PER_LEAF = 24 + 24 + 8 + 8 + 40   # J, HI/HeI/HeII, rho, abun2 read; five fields written


def copy_peak_gbs(torch, s, e0, e1, nbytes=4 << 30, reps=10):
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda:0")
    b = torch.empty_like(a)
    b.copy_(a)
    ms = []
    for _ in range(reps):
        e0.record(s)
        b.copy_(a)
        e1.record(s)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    del a, b
    return 2 * nbytes / (float(np.median(ms)) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--pass-reps", type=int, default=40)
    ap.add_argument("--cases", default="uniform256,nested128")
    a = ap.parse_args()
    import torch

    import radiativetransfer_b200 as rt
    from radiativetransfer_b200 import workloads as W
    name, limit = card()
    bg = W.uvb_background(3.0)
    bd = W.uvb_dust_beta(bg["alpha"], W.synthetic_spectra()["a_dust"])
    gamma, width = W.uvb_heating(bg["table"], bg["alpha"])
    s = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    peak = copy_peak_gbs(torch, s, e0, e1)
    none = np.zeros(0, dtype=np.int32)
    for case in a.cases.split(","):
        nested = case == "nested128"
        g = W.nested_grid(128, 2, W.disc_refine(2), seed=5) if nested else W.uniform_grid(256, seed=1)
        N = g["level"].size
        uvb = bg["uvb"] * (1e-3 if nested else 1.0)   # nested grids: inside the refined-leaf intensity guard
        t = rt.Transport(device=0, math=rt.MATH_FAST)
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
        t.set_dust(2, bd)
        J = torch.empty((3, N), dtype=torch.float64, device="cuda:0")

        def call(heating, rays=None):
            t.set_heating(gamma, width) if heating else t.set_heating(None)
            e0.record(s)
            t.diffuse_device(uvb, bg["beta"], J.data_ptr(), rays=rays, stream=s.cuda_stream)
            e1.record(s)
            e1.synchronize()
            return e0.elapsed_time(e1)

        for h in (False, True):   # warm-up of every shape
            call(h)
            call(h, none)
        step = {False: [], True: []}
        for _ in range(a.reps):
            for h in (False, True):
                step[h].append(call(h))
        stats = t.last_stats()
        empty = {False: [], True: []}
        for _ in range(a.pass_reps):
            for h in (False, True):
                empty[h].append(call(h, none))
        pass_ms = float(np.median(empty[True]) - np.median(empty[False]))
        gbs = PASS_BYTES_PER_LEAF * N / (pass_ms * 1e-3) / 1e9
        st0, st1 = float(np.median(step[False])), float(np.median(step[True]))
        out = dict(case=case, n=g["nx"], levels=2 if nested else 0, nleaf=N, directions=192, math="fast", dust_mode=2,
                   device=name, power_limit=limit, reps=a.reps, pass_reps=a.pass_reps,
                   step_ms=st0, step_spread=[min(step[False]), max(step[False])],
                   step_heating_ms=st1, step_heating_spread=[min(step[True]), max(step[True])],
                   sweep_ms=stats["sweep_ms"], launches_with_heating=stats["launches"],
                   empty_ms=float(np.median(empty[False])), empty_heating_ms=float(np.median(empty[True])),
                   empty_spread=[min(empty[False]), max(empty[False])],
                   empty_heating_spread=[min(empty[True]), max(empty[True])],
                   pass_ms=pass_ms, pass_of_step=pass_ms / st0, pass_bytes=PASS_BYTES_PER_LEAF * N, pass_gbs=gbs,
                   copy_peak_gbs=peak, pass_of_copy_peak=gbs / peak)
        t.close()
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
