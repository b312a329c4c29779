"""GPU experiment: single-cell vs two-cells-per-thread uniform sweep (set_tuning cells), 256^3 and 128^3, with a
bit-for-bit comparison of the results"""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import radiativetransfer_b200 as rt
from radiativetransfer_b200 import workloads as W
bg = W.uvb_background(3.0)
for n in (255, 128, 256):
    g = W.uniform_grid(n, seed=1)
    t = rt.Transport(device=0)
    t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
    J = torch.zeros(3, n ** 3, dtype=torch.float64, device="cuda:0")
    s = torch.cuda.current_stream().cuda_stream
    ref = None
    for cells in (1, 2, 1, 2):
        t.set_tuning(cells=cells)
        ms = []
        for rep in range(5):
            nseg = t.diffuse_device(bg["uvb"], bg["beta"], J.data_ptr(), stream=s)
            torch.cuda.synchronize()
            st = t.last_stats()
            ms.append(st["sweep_ms"])
        Jh = J.cpu().numpy()
        if ref is None:
            ref = Jh
        same = bool(np.array_equal(Jh, ref))
        best = min(ms[1:])
        print(f"n={n} cells={cells}: sweep ms {['%.2f' % m for m in ms]} best {best:.2f} total {st['device_ms']:.2f} "
              f"alg GB/s {st['algorithmic_bytes'] / best / 1e6:.0f} identical_to_first={same}", flush=True)
    t.close()
