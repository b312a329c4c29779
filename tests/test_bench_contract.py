"""bench.py contract on a CPU-only box: the reference arm prints one JSON line with the agreed keys (tiny workload),
and the product arm refuses to run without a CUDA device instead of falling back.  --dump-outputs: the sample it
writes (CPU) and what it writes on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT, _have_gpu

import pytest


def _run(args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


@pytest.mark.parametrize("workload", ["diffuse-64^3-uniform-192dir", "point-32^3-uniform-1src"])
def test_reference_arm_prints_one_json_line(workload):
    r = _run(["--impl", "reference", "--workload", workload, "--steps", "1", "--warmup", "0", "--cpu-threads", "2"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "higher_is_better", "scaling", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["config"]["workload"] == workload
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 2
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


@pytest.mark.skipif(_have_gpu(), reason="only meaningful without a CUDA device")
def test_product_arm_has_no_cpu_fallback():
    r = _run(["--workload", "diffuse-64^3-uniform-192dir", "--steps", "1", "--warmup", "3", "--no-cpu-baseline"])
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)


def test_dump_outputs_writes_all_leaves_or_a_fixed_sample_within_the_cap(tmp_path, monkeypatch):
    import torch
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)     # importing bench sets it
    import bench
    rng = np.random.default_rng(1)
    N = 5000
    arrays = {"jmean": rng.random((3, N)), "rates": torch.from_numpy(rng.random((6, N)))}
    bench.dump_outputs(str(tmp_path / "all"), arrays, 123, N)
    assert np.array_equal(np.load(tmp_path / "all" / "leaf_index.npy"), np.arange(N))
    assert np.array_equal(np.load(tmp_path / "all" / "jmean.npy"), arrays["jmean"])
    assert np.array_equal(np.load(tmp_path / "all" / "rates.npy"), arrays["rates"].numpy())
    assert np.array_equal(np.load(tmp_path / "all" / "segment_updates.npy"), [123.0])
    cap = 200_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, 123, N, max_bytes=cap)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["jmean.npy", "leaf_index.npy", "rates.npy", "segment_updates.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= cap
    idx = np.load(tmp_path / "a" / "leaf_index.npy")
    assert 1000 < idx.size < N and np.all(np.diff(idx) > 0)
    for name in ("jmean", "rates"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, b)
        assert np.array_equal(a, np.asarray(arrays[name])[:, idx.astype(np.int64)])


@pytest.mark.gpu
def test_dump_outputs_are_what_the_library_computes(build_product, tmp_path):
    """the dumped outputs of the timed path equal the host-buffer calls on the same seeded inputs"""
    import radiativetransfer_b200 as rt
    from radiativetransfer_b200 import workloads as W
    r = _run(["--workload", "diffuse-32^3-uniform-192dir", "--steps", "2", "--warmup", "0", "--no-cpu-baseline",
              "--no-secondary", "--dump-outputs", str(tmp_path / "d")])
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])["steps"] == 2
    r = _run(["--workload", "point-16^3-amr-4src", "--steps", "1", "--warmup", "0", "--no-cpu-baseline",
              "--dump-outputs", str(tmp_path / "p")])
    assert r.returncode == 0, r.stderr[-2000:]
    t = rt.Transport(device=0)
    g, bg = W.uniform_grid(32, seed=1), W.uvb_background(3.0)
    t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
    J, nseg = t.diffuse(bg["uvb"], bg["beta"])
    assert np.array_equal(np.load(tmp_path / "d" / "leaf_index.npy"), np.arange(32 ** 3))
    assert np.array_equal(np.load(tmp_path / "d" / "jmean.npy"), J)
    assert np.array_equal(np.load(tmp_path / "d" / "segment_updates.npy"), [float(nseg)])
    fourpi = 4.0 * W.PI
    k24 = fourpi * J[0] * bg["ksi24"][0] + fourpi * J[1] * bg["ksi24"][1] + fourpi * J[2] * bg["ksi24"][2]
    k25 = fourpi * J[2] * bg["ksi25"][0]
    k26 = fourpi * J[1] * bg["ksi26"][0] + fourpi * J[2] * bg["ksi26"][1]
    assert np.allclose(np.load(tmp_path / "d" / "photo_rates.npy"), np.stack([k24, k25, k26]), rtol=1e-14, atol=0)
    g, src = W.point_workload(16, 4)
    t.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
    p = t.point(W.synthetic_spectra(), src, np.ones(src.size, dtype=np.int32))
    t.close()
    rates = np.load(tmp_path / "p" / "rates.npy")
    assert rates.shape == p["rates"].shape and np.abs(p["rates"]).max() > 0
    assert np.allclose(rates, p["rates"], rtol=1e-9, atol=1e-12 * np.abs(p["rates"]).max())   # summation order only
    assert np.array_equal(np.load(tmp_path / "p" / "segment_updates.npy"), [float(p["nseg"])])
