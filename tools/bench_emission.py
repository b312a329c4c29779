"""Cost of emission in the diffuse sweep: the same grid swept alternately without and with a seeded emission array, in
one process, every shape warmed up first.  Prints one JSON line per case with ms per sweep (device events around
rtb200_diffuse_device), segment updates per second, the on/off ratio, and the card's name and power limit.

    python tools/bench_emission.py [--reps 10] [--cases uniform256,nested64]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = {
    # bench.py's default workload (FAST arithmetic) and the grid of its iterate10-64^3-amr3-192dir workload
    "uniform256": dict(n=256, levels=0),
    "nested64": dict(n=64, levels=3),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001 -- the numbers are still worth printing, say why the card is unknown
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cases", default="uniform256,nested64")
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
        rng = np.random.default_rng(42)
        eta = 10.0 ** rng.uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap
        t = rt.Transport(device=0, math=rt.MATH_FAST)
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
        J = torch.empty((3, N), dtype=torch.float64, device="cuda:0")
        s = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = {"off": [], "on": []}
        nseg = 0
        for state in ("off", "on"):   # warm-up: plans, graphs and buffers of both shapes
            t.set_emission(None if state == "off" else eta)
            nseg = t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            for state in ("off", "on"):
                t.set_emission(None if state == "off" else eta)
                e0.record(s)
                t.diffuse_device(uvb, bg["beta"], J.data_ptr(), stream=s.cuda_stream)
                e1.record(s)
                e1.synchronize()
                times[state].append(e0.elapsed_time(e1))
        t.close()
        off, on = float(np.median(times["off"])), float(np.median(times["on"]))
        print(json.dumps(dict(case=case, n=n, levels=spec["levels"], nleaf=N, directions=192, math="fast", nseg=nseg,
                              ms_off=off, ms_on=on, ms_off_spread=[min(times["off"]), max(times["off"])],
                              ms_on_spread=[min(times["on"]), max(times["on"])], seg_per_s_off=nseg / (off * 1e-3),
                              seg_per_s_on=nseg / (on * 1e-3), ratio_on_off=on / off, device=name, power_limit=limit,
                              reps=a.reps)), flush=True)


if __name__ == "__main__":
    main()
