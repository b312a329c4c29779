"""Cost of dust in the diffuse sweep (DESIGN.md 4.8), FAST arithmetic, 192 directions, one process, every shape warmed up
first.  Prints one JSON line per case with the card's name and power limit (read through NVML):
  * absorb: the diffuse call without dust and with absorbing dust of modes 1 and 2 (albedo 0), the variants alternating
    call by call; the only added work is the opacity pass, so the difference is compared with the spread;
  * config4: 256^3, mode 2, albedo 0.5 in every group, tolerance 1e-8 (BASELINE.json config 4): iterations and time per
    call, and 10 device-resident outer steps of (dust-scattering solve + chemistry).
The band means are those of workloads.synthetic_spectra's extinction fit at z = 3, unscaled.

    python tools/bench_dust.py [--reps 7] [--cases absorb256,absorb_nested64,config4]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--cases", default="absorb256,absorb_nested64,config4")
    a = ap.parse_args()
    import torch

    import radiativetransfer_b200 as rt
    from radiativetransfer_b200 import workloads as W
    name, limit = card()
    bg = W.uvb_background(3.0)
    bd = W.uvb_dust_beta(bg["alpha"], W.synthetic_spectra()["a_dust"])
    s = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for case in a.cases.split(","):
        nested = case == "absorb_nested64"
        n = 64 if nested else 256
        g = W.nested_grid(64, 3, W.disc_refine(3), seed=5) if nested else W.uniform_grid(256, seed=1)
        N = g["level"].size
        uvb = bg["uvb"] * (1e-3 if nested else 1.0)   # nested grids: inside the refined-leaf intensity guard
        t = rt.Transport(device=0, math=rt.MATH_FAST)
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
        J = torch.empty((3, N), dtype=torch.float64, device="cuda:0")

        def call():
            e0.record(s)
            t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)
            e1.record(s)
            e1.synchronize()
            return e0.elapsed_time(e1)

        out = dict(case=case, n=n, levels=3 if nested else 0, nleaf=N, directions=192, math="fast",
                   beta_dust=bd.tolist(), device=name, power_limit=limit, reps=a.reps)
        if case.startswith("absorb"):
            variants = {"none": (0, (0.0, 0.0, 0.0)), "mode1": (1, (0.0, 0.0, 0.0)), "mode2": (2, (0.0, 0.0, 0.0))}
            ms = {k: [] for k in variants}
            for k, (mode, al) in variants.items():   # warm-up of every variant
                t.set_dust(mode, bd, albedo=al)
                call()
            for _ in range(a.reps):
                for k, (mode, al) in variants.items():
                    t.set_dust(mode, bd, albedo=al)
                    ms[k].append(call())
            for k in variants:
                out[f"{k}_ms"] = float(np.median(ms[k]))
                out[f"{k}_spread"] = [min(ms[k]), max(ms[k])]
        else:
            t.set_dust(2, bd, albedo=(0.5, 0.5, 0.5), max_iterations=500, tolerance=1e-8)
            call()
            ms = [call() for _ in range(a.reps)]
            sc = t.last_scattering()
            out.update(call_ms=float(np.median(ms)), call_spread=[min(ms), max(ms)], iterations=sc["iterations"],
                       residual=sc["residual"], ms_per_iteration=float(np.median(ms)) / sc["iterations"])
            # device-resident outer steps: the dust-scattering solve, then chemistry on the same stream
            t.set_rate_tables(W.rate_tables(5000))
            t.set_temperature(10.0 ** np.random.default_rng(2).uniform(4.0, 4.1, N))
            ksi = np.concatenate([bg["ksi24"], bg["ksi25"], bg["ksi26"]])
            t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)   # warm-up of the chemistry pass
            t.chemistry_device(0, J.data_ptr(), ksi=ksi, stream=s.cuda_stream, want_change=False)
            its = []
            e0.record(s)
            for _ in range(10):
                t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)
                its.append(t.last_scattering()["iterations"])
                t.chemistry_device(0, J.data_ptr(), ksi=ksi, stream=s.cuda_stream, want_change=False)
            e1.record(s)
            e1.synchronize()
            out.update(resident10_ms=e0.elapsed_time(e1), resident10_iterations=its)
        t.close()
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
