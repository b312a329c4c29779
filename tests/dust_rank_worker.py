"""Worker of tests/test_dust_gpu.py::test_one_process_per_gpu (launched by torch.distributed.run, one rank per GPU).
Every rank joins the device group with rtb200_create_rank, sets the dust (scalars, the same on every rank), runs the
diffuse calls collectively (absorbing dust, and scattering dust with a fixed count and a tolerance; host-buffer and
resident calls) and compares ITS slab of J and the iteration count with the single-device solve it computes itself."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist

    import radiativetransfer_b200 as rt
    from conftest import rel_err
    from radiativetransfer_b200 import workloads as W

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")          # plumbing only: broadcasts the NCCL unique ids of the library's own groups

    def new_uid():
        uid = [rt.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        return uid[0]

    bg = W.uvb_background(3.0)
    uvb, beta = bg["uvb"], bg["beta"]
    bd0 = W.uvb_dust_beta(bg["alpha"], W.synthetic_spectra()["a_dust"])
    for g, scale in ((W.uniform_grid(24, seed=3), 1.0), (W.nested_grid(6, 2, W.central_box_refine(0.2, 0.7, levels=2), seed=5), 1e-3)):
        N = g["level"].size
        g["abun2"] = np.random.default_rng(11).uniform(0.005, 0.04, N)
        for mode, albedo, max_iter, tol in ((1, (0.0, 0.0, 0.0), 1, 0.0), (2, (0.3, 0.5, 0.7), 4, 0.0),
                                            (2, (0.3, 0.5, 0.7), 100, 1e-9)):
            col = g["HI"] if mode == 1 else g["rho"] / W.MP
            bd = bd0 * (np.max(g["HI"] * beta[0][0]) / np.max(col * bd0[0] * g["abun2"] / 0.2))   # dust within the gas's range
            one = rt.Transport(device=local, math=rt.MATH_FAITHFUL)
            one.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
            one.set_dust(mode, bd, albedo=albedo, max_iterations=max_iter, tolerance=tol)
            J1, nseg1 = one.diffuse(uvb * scale, beta)
            s1 = one.last_scattering()
            one.close()
            grp = rt.Transport(device=local, comm=(world, rank, new_uid()), math=rt.MATH_FAITHFUL)
            grp.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
            off, cnt, _, _, _ = grp.slab(0)
            grp.set_dust(mode, bd, albedo=albedo, max_iterations=max_iter, tolerance=tol)
            J = np.full((3, N), -1.0)
            _, nseg = grp.diffuse(uvb * scale, beta, out=J)
            s = grp.last_scattering()
            t = torch.tensor([nseg], dtype=torch.int64); dist.all_reduce(t)
            assert int(t[0]) == nseg1, (int(t[0]), nseg1)
            assert s["iterations"] == s1["iterations"], (s, s1)
            err = rel_err(J[:, off:off + cnt], J1[:, off:off + cnt])
            assert err < 1e-12, err
            grp.diffuse_resident(uvb * scale, beta)
            grp.sync()
            assert grp.last_scattering()["iterations"] == s["iterations"]
            _, _, Js, _, _ = grp.slab_get(0)
            assert np.array_equal(Js, J[:, off:off + cnt])
            print(f"rank {rank}: N={N} dust mode {mode} albedo {albedo} K<={max_iter} tol={tol}: {s['iterations']} "
                  f"iterations, err {err:.3e}", flush=True)
            grp.close()
    dist.barrier()
    print("RANK-OK", rank, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
