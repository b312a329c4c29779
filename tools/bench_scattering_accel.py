"""Cost and gain of the accelerated source iteration (DESIGN.md 4.9), FAST arithmetic, 192 directions, one process, every
shape warmed up first.  Prints one JSON line per case with the card's name and power limit (read through NVML):
  * sweeps and ms per call (median of --reps calls) to tolerance 1e-8 with plain iteration and with Ng, at albedo 0.5
    and 0.9 (sigma = albedo / (1 - albedo) * kappa_abs, with the emission of tools/bench_scattering.py);
  * the time of one extrapolation: a 5-sweep call with Ng (one extrapolation) minus the same call without it;
  * config 4: 10 device-resident outer steps of solve + chemistry with scattering dust (mode 2, albedo 0.5,
    tolerance 1e-8), plain and with NG | WARM_START: total time and sweeps per step.

    python tools/bench_scattering_accel.py [--reps 3] [--cases uniform256,nested64] [--outer uniform256]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_scattering import CASES, card  # noqa: E402


def _grid(W, spec):
    n = spec["n"]
    g = W.uniform_grid(n, seed=1) if spec["levels"] == 0 else W.nested_grid(n, spec["levels"], W.disc_refine(spec["levels"]), seed=5)
    g = dict(g)
    g["abun2"] = np.random.default_rng(n).uniform(0.005, 0.04, g["level"].size)   # metallicity for the dust
    return g


def _kappa(g, beta):
    b = np.asarray(beta).reshape(9)
    return np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4], g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cases", default="uniform256,nested64")
    ap.add_argument("--outer", default="uniform256", help="grid of the config-4 outer loop ('' skips it)")
    a = ap.parse_args()
    import torch

    import radiativetransfer_b200 as rt
    from radiativetransfer_b200 import workloads as W
    name, limit = card()
    bg = W.uvb_background(3.0)
    beta = bg["beta"]
    s = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def open_grid(g):
        t = rt.Transport(device=0, math=rt.MATH_FAST)
        t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
        return t

    for case in [c for c in a.cases.split(",") if c]:
        spec = CASES[case]
        g = _grid(W, spec)
        N = g["level"].size
        uvb = bg["uvb"] * (1.0 if spec["levels"] == 0 else 1e-3)   # nested grids: inside the refined-leaf intensity guard
        kap = _kappa(g, beta)
        t = open_grid(g)
        t.set_emission(10.0 ** np.random.default_rng(42).uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap)
        J = torch.empty((3, N), dtype=torch.float64, device="cuda:0")

        def timed(sigma, max_iter, tol, ng):
            t.set_scattering(sigma, max_iterations=max_iter, tolerance=tol)
            t.set_scattering_acceleration(ng=ng)
            ms = []
            for _ in range(a.reps):
                e0.record(s)
                t.diffuse_device(uvb, beta, J.data_ptr(), stream=s.cuda_stream)
                e1.record(s)
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
            return float(np.median(ms)), [min(ms), max(ms)], t.last_scattering()["iterations"], \
                t.last_scattering_acceleration()["extrapolations"]

        for ng in (False, True):   # warm-up: every kernel of both paths at this shape
            t.set_scattering(kap, max_iterations=5, tolerance=0.0)
            t.set_scattering_acceleration(ng=ng)
            t.diffuse_device(uvb, beta, J.data_ptr(), stream=s.cuda_stream)
        torch.cuda.synchronize()
        plain5 = timed(kap, 5, 0.0, False)[0]
        ng5 = timed(kap, 5, 0.0, True)[0]
        out = {}
        for albedo in (0.5, 0.9):
            sigma = kap * albedo / (1.0 - albedo)
            p, ps, pi, _ = timed(sigma, 2000, 1e-8, False)
            q, qs, qi, qe = timed(sigma, 2000, 1e-8, True)
            out[str(albedo)] = dict(plain_sweeps=pi, plain_ms=p, plain_spread=ps, ng_sweeps=qi, ng_extrapolations=qe,
                                    ng_ms=q, ng_spread=qs, sweep_ratio=qi / pi, time_ratio=q / p)
        t.close()
        print(json.dumps(dict(case=case, n=spec["n"], levels=spec["levels"], nleaf=N, directions=192, math="fast",
                              tolerance=1e-8, by_albedo=out, call_5_sweeps_plain_ms=plain5, call_5_sweeps_ng_ms=ng5,
                              extrapolation_ms=ng5 - plain5, device=name, power_limit=limit, reps=a.reps)), flush=True)

    if a.outer:
        spec = CASES[a.outer]
        g = _grid(W, spec)
        N = g["level"].size
        uvb = bg["uvb"] * (1.0 if spec["levels"] == 0 else 1e-3)
        bd = W.uvb_dust_beta(bg["alpha"], W.synthetic_spectra()["a_dust"])
        kd1 = ((0.76 * g["rho"]) / 1.6726231e-24 * bd[0]) * g["abun2"] / 0.2
        bd = bd * (np.max(_kappa(g, beta)[0]) / np.max(kd1))   # the largest dust opacity equals the gas's largest
        ktab = W.rate_tables(500)
        tgas = 10.0 ** np.random.default_rng(2).uniform(4.0, 4.1, N)
        ksi = np.concatenate([bg["ksi24"], bg["ksi25"], bg["ksi26"]])
        J = torch.empty((3, N), dtype=torch.float64, device="cuda:0")
        res = {}
        for label, acc in (("plain", False), ("ng_warm", True)):
            t = open_grid(g)
            t.set_rate_tables(ktab)
            t.set_temperature(tgas)
            t.set_dust(2, bd, albedo=(0.5, 0.5, 0.5), max_iterations=2000, tolerance=1e-8)
            t.set_scattering_acceleration(ng=acc, warm_start=acc)
            t.diffuse_device(uvb, beta, J.data_ptr(), stream=s.cuda_stream)   # warm-up, then the species start over
            torch.cuda.synchronize()
            t.update_species(HI=g["HI"], HeI=g["HeI"], HeII=g["HeII"])
            t.set_scattering_acceleration(ng=acc, warm_start=acc)
            t.set_dust(0)
            t.set_dust(2, bd, albedo=(0.5, 0.5, 0.5), max_iterations=2000, tolerance=1e-8)   # drops the warm-up's J
            sweeps, warm = [], []
            e0.record(s)
            for _ in range(10):
                t.diffuse_device(uvb, beta, J.data_ptr(), stream=s.cuda_stream)
                sweeps.append(t.last_scattering()["iterations"])
                warm.append(t.last_scattering_acceleration()["warm_start"])
                t.chemistry_device(0, J.data_ptr(), ksi=ksi, stream=s.cuda_stream, want_change=False)
            e1.record(s)
            e1.synchronize()
            res[label] = dict(total_ms=e0.elapsed_time(e1), sweeps_per_step=sweeps, total_sweeps=int(sum(sweeps)),
                              warm_started=warm)
            t.close()
        print(json.dumps(dict(case="config4-outer10-" + a.outer, nleaf=N, directions=192, math="fast", dust_mode=2,
                              albedo=0.5, tolerance=1e-8, steps=10, **res,
                              speedup=res["plain"]["total_ms"] / res["ng_warm"]["total_ms"],
                              device=name, power_limit=limit)), flush=True)


if __name__ == "__main__":
    main()
