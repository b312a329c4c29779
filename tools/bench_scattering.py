"""Cost and convergence of scattering (source iteration, DESIGN.md 4.7), FAST arithmetic, 192 directions, one process,
every shape warmed up first.  Prints one JSON line per case with the card's name and power limit (read through NVML):
  * per-call and per-iteration device time with sigma = kappa_abs (albedo 0.5) and tolerance 1e-8, and the iterations;
  * the emissive sweep alone, and the calls with exactly 1 and 3 iterations (tolerance 0): the increment per iteration
    minus the sweep is the source pass, given as its share of an iteration;
  * iterations to converge (tolerance 1e-8) at albedo 0.1 / 0.5 / 0.9.

    python tools/bench_scattering.py [--reps 3] [--cases uniform256,uniform128,nested64]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = {
    "uniform256": dict(n=256, levels=0),
    "uniform128": dict(n=128, levels=0),
    "nested64": dict(n=64, levels=3),    # the grid of bench.py's iterate10-64^3-amr3-192dir workload
}


def card(index=0):
    """(name, enforced power limit in W) through NVML"""
    try:
        nv = C.CDLL("libnvidia-ml.so.1")
        assert nv.nvmlInit_v2() == 0
        h = C.c_void_p()
        assert nv.nvmlDeviceGetHandleByIndex_v2(index, C.byref(h)) == 0
        name = C.create_string_buffer(96)
        assert nv.nvmlDeviceGetName(h, name, 96) == 0
        mw = C.c_uint(0)
        assert nv.nvmlDeviceGetEnforcedPowerLimit(h, C.byref(mw)) == 0
        nv.nvmlShutdown()
        return name.value.decode(), f"{mw.value / 1000:.0f} W"
    except Exception as e:  # noqa: BLE001 -- the numbers are still worth printing, say why the card is unknown
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cases", default="uniform256,uniform128,nested64")
    a = ap.parse_args()
    import torch

    import radiativetransfer_b200 as rt
    from radiativetransfer_b200 import workloads as W
    name, limit = card()
    bg = W.uvb_background(3.0)
    for case in a.cases.split(","):
        spec = CASES[case]
        n = spec["n"]
        g = W.uniform_grid(n, seed=1) if spec["levels"] == 0 else W.nested_grid(n, spec["levels"], W.disc_refine(spec["levels"]), seed=5)
        N = g["level"].size
        uvb = bg["uvb"] * (1.0 if spec["levels"] == 0 else 1e-3)   # nested grids: inside the refined-leaf intensity guard
        b = np.asarray(bg["beta"]).reshape(9)
        kap = np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])
        eta = 10.0 ** np.random.default_rng(42).uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap
        t = rt.Transport(device=0, math=rt.MATH_FAST)
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
        t.set_emission(eta)
        J = torch.empty((3, N), dtype=torch.float64, device="cuda:0")
        s = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def timed(sigma, max_iter, tol):
            t.set_scattering(sigma, max_iterations=max_iter, tolerance=tol)
            t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)   # warm-up of this shape
            torch.cuda.synchronize()
            ms = []
            for _ in range(a.reps):
                e0.record(s)
                t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)
                e1.record(s)
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
            return float(np.median(ms)), [min(ms), max(ms)], t.last_scattering()

        sweep, sweep_spread, _ = timed(None, 1, 0.0)
        one, _, _ = timed(kap, 1, 0.0)
        three, _, _ = timed(kap, 3, 0.0)
        call, call_spread, sc = timed(kap, 500, 1e-8)
        inc = (three - one) / 2.0
        conv = {}
        for albedo in (0.1, 0.5, 0.9):
            t.set_scattering(kap * albedo / (1.0 - albedo), max_iterations=2000, tolerance=1e-8)
            t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)
            torch.cuda.synchronize()
            conv[str(albedo)] = t.last_scattering()
        t.close()
        print(json.dumps(dict(case=case, n=n, levels=spec["levels"], nleaf=N, directions=192, math="fast",
                              emissive_sweep_ms=sweep, emissive_sweep_spread=sweep_spread,
                              albedo05_tol1e8_call_ms=call, call_spread=call_spread, iterations=sc["iterations"],
                              residual=sc["residual"], ms_per_iteration=call / sc["iterations"],
                              call_1_iteration_ms=one, call_3_iterations_ms=three, increment_per_iteration_ms=inc,
                              source_pass_share=(inc - sweep) / inc, iterations_to_1e8_by_albedo=conv,
                              device=name, power_limit=limit, reps=a.reps)), flush=True)


if __name__ == "__main__":
    main()
