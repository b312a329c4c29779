"""GPU experiment driver: times the uniform diffuse sweep for a list of launch-tuning variants (device-resident call,
CUDA events inside the library)."""
import argparse
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import radiativetransfer_b200 as rt  # noqa: E402
from radiativetransfer_b200 import workloads as W  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, nargs="+", default=[128, 256])
# slots:math[:dirs_per_task:pdl]
ap.add_argument("--variants", nargs="+", default=["0:fast", "16:fast", "8:fast", "0:faithful"])
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
bg = W.uvb_background(3.0)
for n in args.n:
    g = W.uniform_grid(n, seed=1)
    t = rt.Transport(device=0)
    t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
    J = torch.zeros(3, n ** 3, dtype=torch.float64, device="cuda:0")
    s = torch.cuda.current_stream().cuda_stream
    for v in args.variants:
        f = v.split(":")
        slots, mode = f[:2]
        dpt = int(f[2]) if len(f) > 2 else 0
        pdl = int(f[3]) if len(f) > 3 else 0
        t.set_math(rt.MATH_FAST if mode == "fast" else rt.MATH_FAITHFUL)
        t.set_tuning(slots=int(slots), dirs_per_task=dpt, pdl=pdl)
        ms = []
        for rep in range(args.reps + 1):
            nseg = t.diffuse_device(bg["uvb"], bg["beta"], J.data_ptr(), stream=s)
            torch.cuda.synchronize()
            st = t.last_stats()
            ms.append(st["sweep_ms"])
        best = min(ms[1:])
        print(f"n={n} slots={slots} dpt={dpt} pdl={pdl} math={mode}: ms={['%.2f' % m for m in ms]} "
              f"seg/s={nseg / best * 1e3:.3e} alg GB/s={st['algorithmic_bytes'] / best / 1e6:.1f} "
              f"total_ms={st['device_ms']:.2f} launches={st['launches']}", flush=True)
    t.close()
