"""times every rank's direction shard of an N-GPU run on ONE GPU (the sweep of a shard does not depend on the other
ranks), for the zone-class cost factors of the sharding rule and the block size of small shards:
python tools/shard_times.py [world] [block_warps ...]"""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import radiativetransfer_b200 as rt
from radiativetransfer_b200 import sharding, workloads as W
n = 256
world = int(sys.argv[1]) if len(sys.argv) > 1 else 8
variants = sys.argv[2:] or ["0"]          # block_warps[:slots] or key=value,key=value (set_tuning keys)
bg = W.uvb_background(3.0)
g = W.uniform_grid(n, seed=1)
t = rt.Transport(device=0)
t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
J = torch.zeros(3, n ** 3, dtype=torch.float64, device="cuda:0")
s = torch.cuda.current_stream().cuda_stream
shards = sharding.shard_directions(world, n_angular_level=3, nx=n)
zone, cost = sharding.direction_costs(3, 64)
DEFAULTS = dict(block_warps=0, slots=0, cells=0, dirs_per_task=0)
for v in variants:
    if "=" in v:                 # k=v,k=v
        kv = {k: int(x) for k, x in (f.split("=") for f in v.split(","))}
    else:                        # block_warps[:slots]
        f = [int(x) for x in v.split(":")]
        kv = dict(zip(("block_warps", "slots"), f))
    cfg = dict(DEFAULTS); cfg.update(kv)
    t.set_tuning(**cfg)
    times, totals = [], []
    for rank in range(world):
        for rep in range(4):
            t.diffuse_device(bg["uvb"], bg["beta"], J.data_ptr(), rays=shards[rank], stream=s)
            torch.cuda.synchronize()
            st = t.last_stats()
        zs = sorted(set(int(zone[r]) for r in shards[rank]))
        times.append(st["sweep_ms"]); totals.append(st["device_ms"])
        print(f"world {world} block_warps {v} rank {rank} ndir {len(shards[rank])} zones {zs} segs/col {cost[shards[rank]].sum():.0f}: "
              f"sweep_ms {st['sweep_ms']:.3f} total_ms {st['device_ms']:.3f} launches {st['launches']}", flush=True)
    print(f"world {world} block_warps {v}: sweep max {max(times):.3f} mean {np.mean(times):.3f} max/mean {max(times) / np.mean(times):.4f}; "
          f"call (opacities + sweep + merge) max {max(totals):.3f}", flush=True)
t.close()
