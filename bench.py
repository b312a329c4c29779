#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: the per-direction diffuse-radiation sweep (and, as further
workloads, the point-source ray casting and the combined outer iteration on a nested grid).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torch.distributed.run)
    python bench.py --impl reference ...                      (CPU arm: the reference algorithm on the host cores)
    python bench.py ... --dump-outputs DIR                    (one GPU: the last timed step's outputs as DIR/*.npy)

One *step* of the default workload = one full diffuse solve (all 12*4**(nAngularLevel-1) = 192 directions) over one
synthetic grid: computeOpacities + sweep + merge + diffuse photo-rates; on N > 1 GPUs the directions are sharded inside
the library's device group (one process per GPU, rtb200_create_rank) and the per-leaf sums are reduce-scattered over
NVLink, so that every rank ends with its slab of Jmean1..3 and of the photo-rates ("strong" scaling: fixed total work).
Default workload: the configuration the metric's target is quoted on -- a 256^3 uniform grid, 192 directions.

Prints ONE JSON line (rank 0).  `value` = ray-cell segment updates per second with inputs resident in HBM; `e2e` = the
same metric through the host-buffer C-ABI calls (H2D of HI/HeI/HeII from pinned memory, D2H of Jmean1..3; slab-wise per
rank on N > 1 GPUs) inside the timed region; `roofline` = algorithmic bytes (72 B per leaf per direction, SURVEY.md 8d)
of the sweep kernel launches over their CUDA-event time, against the measured HBM copy bandwidth; `cpu_baseline` = the
CPU oracle (a port of the reference: the Fortran itself cannot be built here) on a bounded sample of the same workload,
one core; `parity` = the GPU result for exactly those sampled directions / sources against the oracle's, at the
benchmarked size; `secondary` = short runs of the nested-grid sweep, the point-source pass and the combined outer
iteration (BASELINE configs 5, 3, 5), each with its own roofline fraction and parity.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

REAL_STDOUT = 1
METRIC = "ray-cell segment updates/sec (diffuse sweep)"
METRIC_POINT = "ray-cell segment updates/sec (point-source ray casting + rate deposition)"
METRIC_COMBINED = "ray-cell segment updates/sec (point-source pass + diffuse sweep + ionisation equilibrium)"
UNIT = "segment-updates/s"

# DRAM traffic of the dominant kernel: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed
# `ncu --set full` summaries (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep export)
def ncu_traffic(workload):
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            e = json.load(f).get(workload)
        return (float(e["dram_read_bytes"]) + float(e["dram_write_bytes"])) if e else None
    except Exception:
        return None


WORKLOADS = {
    "diffuse-256^3-uniform-192dir": dict(kind="diffuse", n=256),
    "diffuse-128^3-uniform-192dir": dict(kind="diffuse", n=128),
    "diffuse-64^3-uniform-192dir": dict(kind="diffuse", n=64),
    "diffuse-32^3-uniform-192dir": dict(kind="diffuse", n=32),
    # config 4 style: the reference's outer loop, sweep -> ionisation equilibrium, 10 passes per step, all on the device
    "iterate10-256^3-uniform-192dir": dict(kind="iterate", n=256, iterations=10),
    "iterate10-64^3-uniform-192dir": dict(kind="iterate", n=64, iterations=10),
    "iterate10-64^3-amr3-192dir": dict(kind="iterate", n=64, iterations=10, levels=3),
    # config-5 style nested grid: n^3 base + refinement levels around a synthetic disc (general octree path)
    "diffuse-128^3-amr2-192dir": dict(kind="diffuse", n=128, levels=2),
    "diffuse-64^3-amr3-192dir": dict(kind="diffuse", n=64, levels=3),
    "diffuse-16^3-amr2-192dir": dict(kind="diffuse", n=16, levels=2),
    # point sources: n^3 base grid + one refined level over the central (n/4)^3 base cells, sources inside it
    "point-128^3-amr-100src": dict(kind="point", n=128, nsrc=100),
    "point-256^3-amr-1000src": dict(kind="point", n=256, nsrc=1000),
    "point-32^3-uniform-1src": dict(kind="point", n=32, nsrc=1, uniform=True),
    "point-16^3-amr-4src": dict(kind="point", n=16, nsrc=4),
    # config 5: one outer iteration on the nested grid = point-source pass + diffuse sweep + solveRateEquations
    "combined-64^3-amr3-192dir-64src": dict(kind="combined", n=64, levels=3, nsrc=64),
    "combined-16^3-amr2-192dir-4src": dict(kind="combined", n=16, levels=2, nsrc=4),
}


def make_inputs(spec, seed=1):
    """(n, grid dict, background) of a diffuse-type workload: uniform n^3 or a nested grid"""
    from radiativetransfer_b200 import workloads as W
    n = spec["n"]
    if spec.get("levels"):
        return n, W.nested_grid(n, spec["levels"], W.disc_refine(spec["levels"]), seed=5), W.uvb_background(3.0)
    return n, W.uniform_grid(n, seed=seed), W.uvb_background(3.0)


def point_inputs(spec):
    from radiativetransfer_b200 import workloads as W
    g, src = W.point_workload(spec["n"], spec["nsrc"], uniform=bool(spec.get("uniform")))
    return spec["n"], g, src, np.ones(src.size, dtype=np.int32), W.synthetic_spectra()


def combined_sources(g, nsrc, seed=11):
    """source leaves of the combined workload: the most refined leaves (the disc's mid-plane), seeded choice"""
    lv = g["level"]
    cand = np.where(lv == lv.max())[0]
    rng = np.random.default_rng(seed)
    return np.sort(rng.choice(cand, size=min(nsrc, cand.size), replace=False)).astype(np.int32)


def workload_temperature(N):
    """gas temperature per leaf of the chemistry workloads: 10^4.0 .. 10^4.1 K.  (The reference's equilibrium solver
    prints and stops when a fraction leaves [0, 1] (equiSources.f90:3634-3655), which random combinations of a hot
    cell, a high neutral fraction and a vanishing radiation field provoke; rtb200 reports the same condition as
    RTB200_ERR_CHEMISTRY.  The synthetic state stays clear of it; `device_status` in the JSON line is the check.)"""
    return 10.0 ** np.random.default_rng(2).uniform(4.0, 4.1, N)


def make_config(workload, world):
    """identical for the product arm and the reference arm: names the workload, nothing measured"""
    spec = WORKLOADS[workload]
    n = spec["n"]
    kind = spec["kind"]
    grid = f"{n}^3 uniform, lognormal tau" if not spec.get("levels") and kind != "point" else \
        (f"{n}^3 base + {spec['levels']} nested levels around a synthetic disc" if spec.get("levels") else
         (f"{n}^3 uniform" if spec.get("uniform") else f"{n}^3 base + one refined level over the central {n // 4}^3 cells"))
    cfg = {"workload": workload, "grid": grid, "frequency_groups": 3, "math": "fast", "gpus": world}
    if kind in ("diffuse", "iterate", "combined"):
        cfg.update(directions=192, n_angular_level=3)
    if kind in ("point", "combined"):
        cfg.update(sources=spec["nsrc"], max_pixel_level=6, dust_approximation=0)
    if kind == "iterate":
        cfg["outer_iterations_per_step"] = spec["iterations"]
    cfg["step"] = {
        "diffuse": "computeOpacities + 192-direction sweep + merge + diffuse photo-rates",
        "iterate": f"{spec.get('iterations', 0)} x (computeOpacities + 192-direction sweep + merge + solveRateEquations), "
                   "species re-uploaded at the start of the step",
        "point": "setZeroRates + ray casting of all sources + rate deposition",
        "combined": "species upload + setZeroRates + point-source pass + computeOpacities + 192-direction sweep + "
                    "solveRateEquations (one outer iteration of the reference driver without its I/O)",
    }[kind]
    cfg["parallelism"] = ("one GPU" if world == 1 else
                          f"device group of {world} GPUs (one process each): full grid per GPU, directions / sources "
                          "sharded in the library, reduce-scatter of the per-leaf sums over NVLink, results slab-wise")
    cfg["l2_policy"] = ("inputs larger than L2 (kappa + J + planes >> 126 MB)" if n >= 200 else
                        "working set comparable to L2; not flushed between steps")
    return cfg


# ------------------------------------------------------------------------------------------------------------------
CLOCK_PERIOD_S = float(os.environ.get("RTB_BENCH_CLOCK_PERIOD", "0.1"))   # seconds between NVML clock samples


def sample_clocks(stop, out, dev):
    """SM clock and throttle reasons of GPU `dev` every CLOCK_PERIOD_S until `stop` is set.  NVML in-process (nvidia_ml_py): a
    query costs microseconds and does not fork -- spawning nvidia-smi from a process with a CUDA context stalls the
    launching thread for milliseconds, which is visible in short timed regions.  nvidia-smi is the fallback."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(int(dev))
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        bits = [0x8, 0x40, 0x20, 0x4]          # hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap
        while True:
            r = int(reasons_fn(h))
            out.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx)] +
                       ["Active" if r & b else "Not Active" for b in bits])
            if stop.wait(CLOCK_PERIOD_S):
                break
        return
    except Exception:
        pass
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(dev)],
                               capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 6:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.2)


def clocks_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(float(s[0]) for s in samples if s[0].replace(".", "").isdigit())
    mx = [float(s[1]) for s in samples if s[1].replace(".", "").isdigit()]
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [nm for i, nm in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
            "samples": len(samples)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def rel_linf(a, b, floor=1e-290):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor))) if a.size else 0.0


DUMP_BYTES = 64 * 10 ** 6            # what --dump-outputs writes at most


def dump_outputs(path, arrays, nseg, nleaf, max_bytes=DUMP_BYTES, seed=0):
    """writes the per-leaf outputs `arrays` (name -> [rows, nleaf], torch tensor or numpy) as path/<name>.npy in float64,
    with segment_updates.npy = [nseg] and leaf_index.npy = the leaves written.  When all leaves would exceed `max_bytes`,
    every array is cut to the same seeded sample of leaves (sorted), identical from run to run for a given nleaf."""
    rows = sum(int(a.shape[0]) for a in arrays.values())
    count = min(nleaf, (max_bytes - 4096 * (len(arrays) + 2)) // (8 * (rows + 1)))     # 4 KiB per file for the header
    idx = np.arange(nleaf) if count == nleaf else \
        np.sort(np.random.default_rng(seed).choice(nleaf, size=count, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "leaf_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "segment_updates.npy"), np.array([nseg], dtype=np.float64))
    for name, a in arrays.items():
        if isinstance(a, np.ndarray):
            a = a[:, idx]
        else:
            import torch
            a = a[:, torch.from_numpy(idx).to(a.device)].cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------------------------
# CPU legs (the oracle is test infrastructure: it is the checker and the reported baseline, never the product path)
# ------------------------------------------------------------------------------------------------------------------
class CpuDiffuse:
    """CPU oracle of the diffuse sweep on the workload's grid; the octree (and the worker threads' private copies) is
    built once, every sample() sweeps a bounded number of directions and keeps what it swept for the parity check"""

    def __init__(self, n, grid, bg, threads):
        from oracle import ftte_oracle as fo
        self.og = fo.OracleGrid(n, grid["level"], grid["HI"], grid["HeI"], grid["HeII"], box_size=grid["box_size"])
        self.bg, self.n, self.threads = bg, n, threads
        self.order = (np.arange(192) * 37) % 192          # spread the sampled directions over the zones
        self.cursor = 0
        self.J = np.zeros((3, int(grid["level"].size)))    # sum over the directions swept so far
        self.rays = []
        self.nseg = 0
        if threads > 1:  # creates the worker threads' private octree copies (set-up, untimed)
            self.og.diffuse_mt(bg["uvb"], bg["beta"], self.order[:0], nthreads=threads)

    def sample(self, seconds, max_batches=None, keep=True):
        """sweeps batches of `threads` directions until `seconds` are used up (at least one batch)"""
        t0 = time.perf_counter()
        nseg, ndirs, batches = 0, 0, 0
        while True:
            rays = self.order[(self.cursor + np.arange(self.threads)) % 192]
            self.cursor = (self.cursor + self.threads) % 192
            o = self.og.diffuse_mt(self.bg["uvb"], self.bg["beta"], rays, nthreads=self.threads)
            assert o["status"] == 0
            nseg += o["nseg"]; ndirs += rays.size; batches += 1
            if keep and len(self.rays) + rays.size <= 192:
                self.J += o["J"]; self.rays += [int(r) for r in rays]; self.nseg += o["nseg"]
            dt = time.perf_counter() - t0
            if dt + dt / batches > seconds or (max_batches and batches >= max_batches):
                break
        self.last_seconds = dt
        return nseg / dt, (f"{ndirs} direction sweep(s) out of the workload's 192 (cycled), same {self.n}^3 grid, "
                           f"{dt:.1f} s, {self.threads} thread(s)")


def cpu_point_sample(g, src, wt, sp, seconds, threads, max_sources=None):
    """times the CPU oracle (libm, as the reference) on a bounded number of the workload's sources, one source per
    host thread at a time (each thread a private copy of the octree); returns (rate, description, parity data)"""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import ftte_oracle as fo
    n = g["nx"]
    grids = [fo.OracleGrid(n, g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
             for _ in range(threads)]
    results = {}

    def one(i):
        o = grids[i % threads].point(sp, src[i:i + 1], wt[i:i + 1])
        results[i] = o
        return o["nseg"]

    t0 = time.perf_counter()
    done, nseg = 0, 0
    limit = src.size if max_sources is None else min(src.size, max_sources)
    with ThreadPoolExecutor(threads) as ex:    # ctypes releases the GIL inside the oracle call
        while done < limit and (done == 0 or time.perf_counter() - t0 < seconds):
            chunk = list(range(done, min(done + threads, limit)))
            nseg += sum(ex.map(one, chunk))
            done += len(chunk)
    dt = time.perf_counter() - t0
    idx = sorted(results)
    par = dict(idx=np.array(idx, dtype=np.int64), rates=sum(results[i]["rates"] for i in idx),
               nseg=sum(results[i]["nseg"] for i in idx),
               diag={k: np.concatenate([results[i][k] for i in idx]) for k in
                     ("ndot_remaining", "ndot_boundary", "ndot_dust", "ndot_spectrum", "highest_pixel_level")})
    return nseg / dt, f"{done} of {src.size} sources of the same grid, {dt:.1f} s, {threads} thread(s)", par


def host_threads(nleaf, cap=32):
    import psutil
    cores = os.cpu_count() or 1
    per_copy = 260.0 * nleaf                                  # bytes per private octree copy
    return int(max(1, min(cores, cap, (0.5 * psutil.virtual_memory().available) // per_copy)))


def run_reference(args):
    """CPU arm: the reference algorithm (C++ oracle port; the Fortran cannot be compiled in this image) on all host
    cores, rank 0 only.  Each step is a bounded sample of the workload; the whole run is capped at ~150 s of sweeps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    spec = WORKLOADS[args.workload]
    budget_total = float(os.environ.get("RTB_BENCH_REFERENCE_SECONDS", "150"))
    t_start = time.perf_counter()
    if spec["kind"] == "point":
        n, g, src, wt, sp = point_inputs(spec)
        threads = args.cpu_threads or host_threads(int(g["level"].size))
        metric = METRIC_POINT
        vals, secs = [], []
        nsamples = max(2, min(args.warmup + args.steps, 6))
        for it in range(nsamples):
            v, desc, _ = cpu_point_sample(g, src, wt, sp, budget_total / nsamples, threads)
            if it >= 1 or nsamples == 1:
                vals.append(v)
            secs.append(budget_total / nsamples)
            if time.perf_counter() - t_start > budget_total:
                break
    else:
        n, grid, bg = make_inputs(spec)
        threads = args.cpu_threads or host_threads(int(grid["level"].size))
        metric = METRIC_COMBINED if spec["kind"] == "combined" else METRIC
        cpu = CpuDiffuse(n, grid, bg, threads)
        vals, secs = [], []
        v, desc = cpu.sample(0.0, max_batches=1, keep=False)          # warm-up batch, also the time of one batch
        batch_s = cpu.last_seconds
        nsamples = int(max(2, min(args.steps, (budget_total - batch_s) // max(batch_s, 1e-3))))
        for it in range(nsamples):
            v, desc = cpu.sample(0.0, max_batches=1, keep=False)
            vals.append(v); secs.append(cpu.last_seconds)
            if time.perf_counter() - t_start > budget_total:
                break
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": make_config(args.workload, world),
        "samples_measured": len(vals),
        "sample_note": "each step = a bounded sample of the workload's directions / sources (one batch of one per host "
                       "thread), scaled per segment update; the run is capped at RTB_BENCH_REFERENCE_SECONDS of sweeps",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------------------------
class Env:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the rtb200 path has no CPU fallback (use --impl reference)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.current_stream().cuda_stream

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values, op):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op))
        return [float(x) for x in t]

    def gather(self, value):
        t = self.torch.tensor([value], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(value)]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(x[0]) for x in out]

    def engine(self):
        """one GPU: a plain context; N GPUs: the library's device group, one process per GPU"""
        import radiativetransfer_b200 as rt
        if self.world == 1:
            return rt.Transport(device=self.local), "context"
        uid = [rt.comm_unique_id() if self.rank == 0 else None]
        self.dist.broadcast_object_list(uid, src=0)
        eng = rt.Transport(device=self.local, comm=(self.world, self.rank, uid[0]))
        if os.environ.get("RTB200_MULTI_REDUCE"):      # ablation: 0 = NCCL reduce-scatter instead of the peer-memory kernel
            eng.set_tuning(multi_reduce=int(os.environ["RTB200_MULTI_REDUCE"]))
        return eng, "group"

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def time_steps(env, step, warmup, steps, clock_samples=None):
    """W warm-ups, then exactly K steps between barrier + synchronize; CUDA events on the launch stream; max over ranks"""
    torch = env.torch
    out = None
    for _ in range(warmup):
        out = step()
    env.barrier()
    stop = threading.Event()
    th = None
    if clock_samples is not None and env.rank == 0:
        th = threading.Thread(target=sample_clocks, args=(stop, clock_samples, env.local), daemon=True)
        th.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    stop.set()
    env.barrier()
    return env.reduce([ms], "MAX")[0] / steps, out


def time_e2e(env, step, steps):
    step()
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    env.torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    return env.reduce([ms], "MAX")[0]


def set_grid(eng, g):
    eng.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])


def run_workload(env, workload, steps, warmup, cpu_seconds, with_clocks=True, faithful_too=False, e2e_steps=3,
                 dump_dir=None):
    """times one workload on the process group `env`; returns the dict of measured fields (rank 0 uses it).
    `dump_dir` (one process only): the outputs of the last timed step go there (dump_outputs)."""
    import radiativetransfer_b200 as rt
    from radiativetransfer_b200 import workloads as Wk
    torch = env.torch
    spec = WORKLOADS[workload]
    kind = spec["kind"]
    world, rank = env.world, env.rank
    W = max(warmup, 3 if kind in ("diffuse", "iterate") else 5)   # the point path sizes its scratch on the first passes
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    if kind == "point":
        n, g, src, wt, sp = point_inputs(spec)
        bg = None
    else:
        n, g, bg = make_inputs(spec)
        src = wt = sp = None
        if kind == "combined":
            src = combined_sources(g, spec["nsrc"]); wt = np.ones(src.size, dtype=np.int32); sp = Wk.synthetic_spectra()
    N = int(g["level"].size)
    uniform = not spec.get("levels") and kind != "point"
    eng, mode = env.engine()
    set_grid(eng, g)
    group = mode == "group"
    info = eng.info() if group else dict(nranks=1, slab=N, reduce_mode=-1)
    iterations = spec.get("iterations", 0)
    ksi_all = None if bg is None else np.concatenate([bg["ksi24"], bg["ksi25"], bg["ksi26"]])
    if kind in ("iterate", "combined"):
        eng.set_rate_tables(Wk.rate_tables(5000))
        eng.set_temperature(workload_temperature(N))
    hHI, hHeI, hHeII = pin(g["HI"]), pin(g["HeI"]), pin(g["HeII"])
    stream = env.stream
    if not group:
        J = torch.zeros(3, N, dtype=torch.float64, device=env.dev)
        K = torch.zeros(3, N, dtype=torch.float64, device=env.dev)
        R = torch.zeros(6, N, dtype=torch.float64, device=env.dev) if kind in ("point", "combined") else None

    # ---- resident steps ----
    def step_resident():
        if kind == "diffuse":
            if group:
                return eng.diffuse_resident(bg["uvb"], bg["beta"], ksi=ksi_all, streams=[stream])
            nseg = eng.diffuse_device(bg["uvb"], bg["beta"], J.data_ptr(), stream=stream)
            eng.diffuse_rates_device(J.data_ptr(), bg["ksi24"], bg["ksi25"], bg["ksi26"], K[0].data_ptr(), K[1].data_ptr(),
                                     K[2].data_ptr(), stream=stream)
            return nseg
        if kind == "iterate":
            # the reference's outer loop (equiSources.f90:1230-1843) without its I/O: sweep -> solveRateEquations,
            # `iterations` passes; HI, HeI, HeII, J never leave the device.  Every step starts from the same state
            # (update_species waits for the device before it overwrites the arrays).
            eng.update_species(hHI.numpy(), hHeI.numpy(), hHeII.numpy())
            total = 0
            for _ in range(iterations):
                if group:
                    total += eng.diffuse_resident(bg["uvb"], bg["beta"], ksi=ksi_all, chemistry=True, streams=[stream])
                else:
                    total += eng.diffuse_device(bg["uvb"], bg["beta"], J.data_ptr(), stream=stream)
                    eng.chemistry_device(0, J.data_ptr(), ksi=ksi_all, stream=stream, want_change=False)
            return total
        if kind == "point":
            if group:
                return eng.point_resident(sp, src, wt, streams=[stream])
            R.zero_()                                          # setZeroRates (equiSources.f90:1246)
            return eng.point_device(sp, src, wt, R.data_ptr(), stream=stream)
        # combined: one outer iteration of the driver (equiSources.f90:1246-1831) without its I/O
        eng.update_species(hHI.numpy(), hHeI.numpy(), hHeII.numpy())
        if group:
            a = eng.point_resident(sp, src, wt, streams=[stream])
            b = eng.diffuse_resident(bg["uvb"], bg["beta"], ksi=ksi_all, chemistry=True, streams=[stream])
            return a + b
        R.zero_()
        a = eng.point_device(sp, src, wt, R.data_ptr(), stream=stream)
        b = eng.diffuse_device(bg["uvb"], bg["beta"], J.data_ptr(), stream=stream)
        eng.chemistry_device(R.data_ptr(), J.data_ptr(), ksi=ksi_all, stream=stream, want_change=False)
        return a + b

    clock_samples = [] if with_clocks else None
    ms_per_step, nseg_rank = time_steps(env, step_resident, W, steps, clock_samples)
    if dump_dir is not None:
        # what a caller of the resident step holds after it: Jmean1..3 [3, N], the diffuse photo-rates k24, k25, k26
        # [3, N], the point-source rates in the order of rtb200_point [6, N], the species HI, HeI, HeII [3, N]
        outs = {} if kind == "point" else dict(jmean=J)
        if kind == "diffuse":
            # the rates call adds to K (rate fields the caller zeroes once per outer iteration) and the timed steps never
            # zero it: K holds the sum over all steps, so the last step's photo-rates are evaluated again from its J
            K.zero_()
            eng.diffuse_rates_device(J.data_ptr(), bg["ksi24"], bg["ksi25"], bg["ksi26"], K[0].data_ptr(), K[1].data_ptr(),
                                     K[2].data_ptr(), stream=stream)
            outs["photo_rates"] = K
        if kind in ("point", "combined"):
            outs["rates"] = R
        if kind in ("iterate", "combined"):
            outs["species"] = np.stack(eng.get_species())
        dump_outputs(dump_dir, outs, nseg_rank, N)
    if not with_clocks:   # secondary workloads (3 steps): a second pass, keep the better one (host jitter of a shared box)
        ms2, _ = time_steps(env, step_resident, 1, steps)
        ms_per_step = min(ms_per_step, ms2)
    st = eng.last_stats()                    # the library's own CUDA events (same stream), LAST sweep / pass of the step
    sweep_ms = st["sweep_ms"] if st["sweep_ms"] > 0 else st["device_ms"]
    nseg_total = env.reduce([float(nseg_rank)], "SUM")[0]
    rank_kernel_ms = env.gather(sweep_ms)
    value = nseg_total / (ms_per_step * 1e-3)

    # ---- end to end through the host-buffer C-ABI calls (pinned host arrays; slab-wise per rank in a group) ----
    hJ = torch.empty(3, N, dtype=torch.float64).pin_memory()
    hR = torch.zeros(6, N, dtype=torch.float64).pin_memory() if kind == "point" else None
    hS = [torch.empty(N, dtype=torch.float64).pin_memory() for _ in range(3)] if kind in ("iterate", "combined") else None
    off, cnt = (eng.slab(0)[:2] if group else (0, N))
    nsrc_mine = 0 if src is None else (len(range(rank, src.size, world)) if group else int(src.size))

    def step_e2e():
        if kind == "diffuse":
            eng.update_species(hHI.numpy(), hHeI.numpy(), hHeII.numpy())          # H2D (this rank's slab in a group)
            eng.diffuse(bg["uvb"], bg["beta"], out=hJ.numpy())                    # ... + D2H of J (slab) inside the call
            return float(hJ[0, off])
        if kind == "point":
            # the call ACCUMULATES into the caller's rate fields (H2D + D2H of the six fields, this rank's slab in a
            # group); zeroing them between passes is the driver's setZeroRates, not part of the call: the fields simply
            # grow from step to step here
            eng.point(sp, src, wt, rates=hR.numpy(), inplace=True)
            return float(hR[0, off])
        step_resident()                                                           # includes the species upload
        if group:
            eng.L.rtb200_grid_get_species(eng.h, *[x.numpy().ctypes.data for x in hS])
        else:
            eng.L.rtb200_grid_get_species(eng.h, *[x.numpy().ctypes.data for x in hS])
        return float(hS[0][off])

    e2e_ms = time_e2e(env, step_e2e, max(1, min(steps, e2e_steps)))
    if kind == "diffuse":
        h2d, d2h = 3 * cnt * 8, 3 * cnt * 8
    elif kind == "point":
        h2d, d2h = 6 * cnt * 8, 6 * cnt * 8 + nsrc_mine * 316 * 8
    else:
        h2d, d2h = 3 * cnt * 8, 3 * cnt * 8
    tot = env.reduce([float(h2d), float(d2h)], "SUM")

    status = eng.device_error() if not group else eng.L.rtb200_multi_sync(eng.h)
    status = int(env.reduce([float(status)], "MAX")[0])
    out = dict(workload=workload, kind=kind, N=N, n=n, uniform=uniform, ms_per_step=ms_per_step, value=value, device_status=status,
               nseg_total=nseg_total, e2e_ms=e2e_ms, e2e_value=nseg_total / (e2e_ms * 1e-3), h2d=int(tot[0]), d2h=int(tot[1]),
               launches=int(st["launches"]), sweep_launches=int(st["sweep_launches"]), sweep_ms=sweep_ms,
               alg_bytes_rank=st["algorithmic_bytes"], rank_kernel_ms=rank_kernel_ms, mode=mode, info=info,
               clocks=clocks_summary(clock_samples) if clock_samples is not None else None, warmup=W)

    # ---- the reference's own operation sequence (FAITHFUL) beside the benchmarked FAST arithmetic ----
    if faithful_too and kind == "diffuse":
        eng.set_math(rt.MATH_FAITHFUL)
        out["faithful_ms_per_step"], _ = time_steps(env, step_resident, 1, 2)
        eng.set_math(rt.MATH_FAST)

    # ---- CPU baseline (one core, bounded sample) and parity of the GPU result on exactly that sample ----
    if world == 1 and cpu_seconds > 0:
        try:
            if kind in ("diffuse", "iterate"):
                cpu = CpuDiffuse(n, g, bg, 1)
                v, desc = cpu.sample(cpu_seconds)
                out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc}
                eng.update_species(hHI.numpy(), hHeI.numpy(), hHeII.numpy())
                rays = np.array(cpu.rays, dtype=np.int32)
                Jg, nseg_g = eng.diffuse(bg["uvb"], bg["beta"], rays=rays)
                par = {"vs": "cpu oracle (libm), same grid, the sampled directions", "dirs": int(rays.size),
                       "rel_linf_J_fast": rel_linf(Jg, cpu.J), "nseg_equal": bool(nseg_g == cpu.nseg), "tolerance": 1e-9}
                eng.set_math(rt.MATH_FAITHFUL)
                Jf, _ = eng.diffuse(bg["uvb"], bg["beta"], rays=rays)
                Jf_full, _ = eng.diffuse(bg["uvb"], bg["beta"])
                eng.set_math(rt.MATH_FAST)
                Jq_full, _ = eng.diffuse(bg["uvb"], bg["beta"])
                par["rel_linf_J_faithful"] = rel_linf(Jf, cpu.J)
                par["rel_linf_J_fast_vs_faithful_all_192_directions"] = rel_linf(Jq_full, Jf_full)
                par["note"] = ("FAITHFUL = the reference's operation sequence: held to 1e-9 on the sampled directions.  FAST "
                               "(benchmarked) omits the reference's exp->divide->log round trip, whose rounding noise "
                               "(~1.1e-16/tau per segment) shows in sums over a few directions: held to 1e-8 on the sample and "
                               "to 1e-9 against FAITHFUL on the full 192-direction solve (tests/test_diffuse_gpu.py)")
                par["ok"] = bool(par["nseg_equal"] and par["rel_linf_J_faithful"] < 1e-9 and par["rel_linf_J_fast"] < 1e-8 and
                                 par["rel_linf_J_fast_vs_faithful_all_192_directions"] < 1e-9)
                out["parity"] = par
            elif kind == "point":
                v, desc, ref = cpu_point_sample(g, src, wt, sp, cpu_seconds, 1)
                out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc}
                out["parity"] = point_parity(eng, sp, g, src, wt, ref)
            else:
                out["cpu_baseline"], out["parity"] = combined_cpu_and_parity(eng, n, g, bg, sp, src, wt, ksi_all, cpu_seconds)
        except Exception as e:  # the checker is optional for the measurement itself
            out.setdefault("cpu_baseline", {"value": None, "unit": UNIT, "cores": 1, "kind": "port", "sample": f"failed: {e!r}"})
            out.setdefault("parity", {"ok": None, "error": repr(e)})
    eng.close()
    return out


def _bracket(spectra, abun2):
    t = np.log10(abun2) if abun2 > 1e-20 else -20.0
    met = spectra["metallicity"]
    m = 1
    while t > met[m]:
        m += 1
        if m + 1 == 5:
            break
    return m, float(np.clip((t - met[m - 1]) / (met[m] - met[m - 1]), 0, 1))


def point_parity(eng, sp, g, src, wt, ref):
    """GPU rates + diagnostics for the sources the oracle sampled.  Rates: 1e-9 relative plus the conditioning floor
    2e-13 * sum_s weight_s R_r(0) of R(d) - R(d + tau) (tests/test_point_gpu.py); diagnostics 1e-11."""
    idx = ref["idx"]
    r = eng.point(sp, src[idx], wt[idx])
    scale = np.zeros((6, 1))
    for leaf, w in zip(src[idx], wt[idx]):
        T = eng.point_tables(sp, *_bracket(sp, g["abun2"][leaf]))
        scale += w * T[[0, 2, 1, 3, 5, 4], 0][:, None]
    d = np.abs(r["rates"] - ref["rates"])
    strict = d / np.maximum(np.abs(ref["rates"]), 1e-300)
    m = ref["rates"] != 0
    within = bool(np.all(d <= 1e-9 * np.abs(ref["rates"]) + 2e-13 * scale))
    par = {"vs": "cpu oracle (libm), same grid, the sampled sources", "sources": int(idx.size),
           "nseg_equal": bool(r["nseg"] == ref["nseg"]), "math": "fast",
           "rates_within_1e-9_plus_floor": within,
           "worst_strict_rel": float(strict[m].max()) if m.any() else 0.0,
           "cells_above_1e-9_strict": int(np.sum(strict[m] > 1e-9)), "cells": int(m.sum())}
    for k in ("ndot_remaining", "ndot_boundary", "ndot_dust", "ndot_spectrum"):
        par["rel_linf_" + k] = rel_linf(r[k], ref["diag"][k], floor=1e-300)
    par["highest_pixel_level_equal"] = bool(np.array_equal(r["highest_pixel_level"], ref["diag"]["highest_pixel_level"]))
    par["ok"] = bool(within and par["nseg_equal"] and par["highest_pixel_level_equal"] and
                     all(par["rel_linf_" + k] < 1e-11 for k in ("ndot_remaining", "ndot_boundary", "ndot_dust", "ndot_spectrum")))
    return par


def combined_cpu_and_parity(eng, n, g, bg, sp, src, wt, ksi_all, cpu_seconds, ndirs=16, nsources=4):
    """one outer iteration on a SUBSET (ndirs directions, nsources sources) by the oracle (timed: the cpu baseline) and
    by the GPU (rays= / source subset): rates, J and the new species compared"""
    from oracle import ftte_oracle as fo
    from radiativetransfer_b200 import workloads as Wk
    torch_N = int(g["level"].size)
    ktab = Wk.rate_tables(5000)
    tgas = workload_temperature(torch_N)
    rays = ((np.arange(ndirs) * 37 + 5) % 192).astype(np.int32)
    s_idx = np.arange(min(nsources, src.size))
    t0 = time.perf_counter()
    og = fo.OracleGrid(n, g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
    t1 = time.perf_counter()
    op = og.point(sp, src[s_idx], wt[s_idx])
    od = og.diffuse_mt(bg["uvb"], bg["beta"], rays, nthreads=1)
    oc = fo.chemistry(n, g["box_size"], g["level"], g["rho"], tgas, g["HI"], g["HeI"], g["HeII"], ktab, rates=op["rates"],
                      J=od["J"], ksi=ksi_all)
    dt = time.perf_counter() - t1
    nseg = op["nseg"] + od["nseg"]
    cpu = {"value": nseg / dt, "unit": UNIT, "cores": 1, "kind": "port",
           "sample": f"{s_idx.size} of {src.size} sources + {ndirs} of 192 directions + solveRateEquations on the same grid, {dt:.1f} s, 1 thread"}
    # GPU, same subset, through the host-buffer calls
    eng.update_species(g["HI"], g["HeI"], g["HeII"])
    rp = eng.point(sp, src[s_idx], wt[s_idx])
    Jg, nsd = eng.diffuse(bg["uvb"], bg["beta"], rays=rays)
    par = {"vs": "cpu oracle (libm), same grid, subset of sources and directions", "sources": int(s_idx.size), "dirs": int(ndirs),
           "nseg_equal": bool(rp["nseg"] == op["nseg"] and nsd == od["nseg"]), "rel_linf_J": rel_linf(Jg, od["J"]),
           "math": "fast"}
    scale = np.zeros((6, 1))
    for leaf, w in zip(src[s_idx], wt[s_idx]):
        T = eng.point_tables(sp, *_bracket(sp, g["abun2"][leaf]))
        scale += w * T[[0, 2, 1, 3, 5, 4], 0][:, None]
    par["rates_within_1e-9_plus_floor"] = bool(np.all(np.abs(rp["rates"] - op["rates"]) <= 1e-9 * np.abs(op["rates"]) + 2e-13 * scale))
    # solveRateEquations on the device: (a) from the ORACLE's rates and J -> must reproduce the oracle's species bit for
    # bit (the kernel is IEEE operations in the reference's order); (b) from the GPU's own rates and J: end to end, where
    # the equilibrium amplifies the reference's rounding noise in cells whose point-source rates are a cancelled
    # difference (see point parity: strict errors up to 1e-2 in cells with vanishing rates)
    if not eng.multi:
        import torch
        s = torch.cuda.current_stream().cuda_stream
        R = torch.from_numpy(op["rates"]).cuda(); Jd = torch.from_numpy(od["J"]).cuda()
        eng.chemistry_device(R.data_ptr(), Jd.data_ptr(), ksi=ksi_all, stream=s)
        torch.cuda.synchronize()
        sg = eng.get_species()
        par["species_bit_identical_given_oracle_rates_and_J"] = bool(all(np.array_equal(a, b) for a, b in
                                                                      zip(sg, (oc["HI"], oc["HeI"], oc["HeII"]))))
        eng.update_species(g["HI"], g["HeI"], g["HeII"])
        R = torch.from_numpy(rp["rates"]).cuda(); Jd = torch.from_numpy(Jg).cuda()
        eng.chemistry_device(R.data_ptr(), Jd.data_ptr(), ksi=ksi_all, stream=s)
        torch.cuda.synchronize()
        sg = eng.get_species()
        par["rel_linf_species_end_to_end"] = max(rel_linf(a, b, floor=1e-300) for a, b in zip(sg, (oc["HI"], oc["HeI"], oc["HeII"])))
        par["chemistry_status"] = int(oc["status"])
    par["ok"] = bool(par["nseg_equal"] and par["rel_linf_J"] < 1e-9 and par["rates_within_1e-9_plus_floor"] and
                     par.get("species_bit_identical_given_oracle_rates_and_J", True) and
                     par.get("rel_linf_species_end_to_end", 0.0) < 1e-5)
    return cpu, par


def roofline_dict(res, world):
    peak, peak_src = measured_peak()
    kind = res["kind"]
    achieved = res["alg_bytes_rank"] / (res["sweep_ms"] * 1e-3) / 1e9 if res["sweep_ms"] > 0 else None
    # the library picks the kernel by shard / wave size: many zone tasks per launch -> two cells per thread; small
    # waves on a 2:1-balanced nested grid -> the one-launch streamed sweep (a handful of launches per step)
    per_pass = res["sweep_launches"]          # of the last sweep call
    uni = "rtb::sweep_cell2_kernel" if world <= 4 else "rtb::sweep_cell_kernel"
    amr = "rtb::amr_stream_kernel" if per_pass < 20 else "rtb::amr_wave_kernel"
    kernel = {"diffuse": uni if res["uniform"] else amr, "iterate": uni if res["uniform"] else amr,
              "point": "rtb::point_march_kernel", "combined": amr}[kind]
    rk = res["rank_kernel_ms"]
    d = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
         "traffic": ncu_traffic(res["workload"]) if world == 1 else None,
         "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/ncu_traffic.json)",
         "peak_source": peak_src, "kernel": kernel, "launches_per_step": res["sweep_launches"],
         "algorithmic_bytes_per_step_this_rank": res["alg_bytes_rank"], "kernel_ms_per_step": res["sweep_ms"],
         "kernel_ms_min_over_ranks": min(rk), "kernel_ms_max_over_ranks": max(rk),
         "note": ("72 B per leaf per direction (SURVEY.md 8d); zones are swept with their directions fused, so DRAM traffic "
                  "differs from the algorithmic bytes (profiles/)") if kind != "point" else
                 "136 B per segment (5 reads + 6 read-modify-writes, SURVEY.md 8d); bound by fp64 issue and gather latency"}
    if kernel == "rtb::amr_stream_kernel":
        d["algorithmic_bytes_per_launch"] = res["alg_bytes_rank"]      # the whole sweep is one launch of this kernel
    elif kind in ("diffuse", "iterate") and res["sweep_launches"] > 1:
        d["algorithmic_bytes_per_launch"] = res["alg_bytes_rank"] / max(1, res["sweep_launches"] - 1)
    return d


def emit(line):
    """the ONE JSON line, on the real stdout"""
    os.write(REAL_STDOUT, (json.dumps(line) + "\n").encode())


def main():
    global REAL_STDOUT
    # anything a library prints to file descriptor 1 (NCCL's version banner, ...) must not get between the driver and
    # the JSON line: fd 1 is pointed at stderr for the whole run, the line itself goes to a duplicate of the original
    sys.stdout.flush()
    REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rtb200", choices=["rtb200", "reference"])
    ap.add_argument("--workload", default="diffuse-256^3-uniform-192dir", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--secondary", default="diffuse-64^3-amr3-192dir,point-128^3-amr-100src,combined-64^3-amr3-192dir-64src")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64, at most "
                         f"{DUMP_BYTES // 10 ** 6} MB: a fixed seeded sample of leaves, DIR/leaf_index.npy, when larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.dump_outputs is not None and (args.impl != "rtb200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the outputs of the rtb200 arm on one GPU (one process)")
    if args.impl == "reference":
        run_reference(args)
        return

    env = Env()
    world = env.world
    cpu_s = 0.0 if args.no_cpu_baseline else args.cpu_seconds
    res = run_workload(env, args.workload, args.steps, args.warmup, cpu_s, faithful_too=True, dump_dir=args.dump_outputs)
    kind = res["kind"]
    line = None
    if env.rank == 0:
        metric = {"diffuse": METRIC, "iterate": METRIC, "point": METRIC_POINT, "combined": METRIC_COMBINED}[kind]
        cfg = make_config(args.workload, world)
        line = {
            "metric": metric, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": res["warmup"],
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg,
            "leaves": res["N"], "segment_updates_per_step": res["nseg_total"], "device_status": res["device_status"],
            "multi_gpu": {"mode": res["mode"], "reduce": {1: "peer-memory reduce-scatter kernel (fused epilogue)", 0: "NCCL reduce-scatter",
                                                         -1: "none (one GPU)"}[res["info"]["reduce_mode"]],
                          "slab_leaves": res["info"]["slab"]},
            "clocks": res["clocks"],
            "e2e": {"value": res["e2e_value"], "unit": UNIT, "ms_per_step": res["e2e_ms"], "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": res["d2h"],
                    "note": "host-buffer C-ABI calls on pinned arrays; on N > 1 GPUs every rank moves its slab only"},
            "gpu_launches": (res["launches"] + 1) * max(WORKLOADS[args.workload].get("iterations", 1), 1) * args.steps,
            "roofline": roofline_dict(res, world),
        }
        if "faithful_ms_per_step" in res:
            line["faithful_ms_per_step"] = res["faithful_ms_per_step"]
        for k in ("cpu_baseline", "parity"):
            if k in res:
                line[k] = res[k]
    # ---- secondary workloads (1 GPU only: keeps the default run within minutes) ----
    if world == 1 and not args.no_secondary and args.workload == "diffuse-256^3-uniform-192dir":
        sec = {}
        for w in [x for x in args.secondary.split(",") if x]:
            try:
                r = run_workload(env, w, steps=3, warmup=3, cpu_seconds=min(cpu_s, 6.0), with_clocks=False, e2e_steps=2)
                rf = roofline_dict(r, 1)
                sec[w] = {"ms_per_step": r["ms_per_step"], "value": r["value"], "unit": UNIT, "leaves": r["N"],
                          "segment_updates_per_step": r["nseg_total"], "e2e_ms_per_step": r["e2e_ms"],
                          "device_status": r["device_status"],
                          "roofline_frac": rf["frac"], "roofline_kernel": rf["kernel"], "traffic": rf["traffic"],
                          "parity": r.get("parity"), "cpu_baseline": r.get("cpu_baseline")}
            except Exception as e:
                sec[w] = {"error": repr(e)}
        if line is not None:
            line["secondary"] = sec
    if env.rank == 0:
        emit(line)
    env.close()


if __name__ == "__main__":
    main()
