"""Worker of tests/test_scattering_gpu.py::test_one_process_per_gpu (launched by torch.distributed.run, one rank per
GPU).  Every rank joins the device group with rtb200_create_rank, sets emission and scattering slab-wise, runs the source
iteration collectively (host-buffer and resident calls, fixed count and tolerance) and compares ITS slab of J and the
iteration count with the single-device solve it computes on its own GPU."""
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
    for g in (W.uniform_grid(24, seed=3), W.nested_grid(6, 2, W.central_box_refine(0.2, 0.7, levels=2), seed=5)):
        N = g["level"].size
        b = np.asarray(beta).reshape(9)
        kap = np.maximum(np.array([g["HI"] * b[0], g["HI"] * b[3] + g["HeI"] * b[4],
                                   g["HI"] * b[6] + g["HeI"] * b[7] + g["HeII"] * b[8]]), 1e-30)
        rng = np.random.default_rng(17)
        a = rng.uniform(0.1, 0.9, size=kap.shape)
        sigma = kap * a / (1.0 - a)
        eta = 10.0 ** rng.uniform(-3.0, 0.0, size=kap.shape) * uvb[:, None] * kap
        for max_iter, tol in ((4, 0.0), (100, 1e-9)):
            one = rt.Transport(device=local, math=rt.MATH_FAITHFUL)
            one.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
            one.set_emission(eta)
            one.set_scattering(sigma, max_iterations=max_iter, tolerance=tol)
            J1, nseg1 = one.diffuse(uvb, beta)
            s1 = one.last_scattering()
            one.close()
            grp = rt.Transport(device=local, comm=(world, rank, new_uid()), math=rt.MATH_FAITHFUL)
            grp.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
            off, cnt, _, _, _ = grp.slab(0)
            mine = np.zeros((3, N)); mine[:, off:off + cnt] = sigma[:, off:off + cnt]    # a rank only owns its slab
            mine_eta = np.zeros((3, N)); mine_eta[:, off:off + cnt] = eta[:, off:off + cnt]
            grp.set_emission(mine_eta)
            grp.set_scattering(mine, max_iterations=max_iter, tolerance=tol)
            J = np.full((3, N), -1.0)
            _, nseg = grp.diffuse(uvb, beta, out=J)
            s = grp.last_scattering()
            t = torch.tensor([nseg], dtype=torch.int64); dist.all_reduce(t)
            assert int(t[0]) == nseg1, (int(t[0]), nseg1)
            assert s["iterations"] == s1["iterations"], (s, s1)
            err = rel_err(J[:, off:off + cnt], J1[:, off:off + cnt])
            assert err < 1e-12, err
            grp.diffuse_resident(uvb, beta)
            grp.sync()
            assert grp.last_scattering()["iterations"] == s["iterations"]
            _, _, Js, _, _ = grp.slab_get(0)
            assert np.array_equal(Js, J[:, off:off + cnt])
            print(f"rank {rank}: N={N} K<={max_iter} tol={tol}: {s['iterations']} iterations, err {err:.3e}", flush=True)
            grp.close()
    dist.barrier()
    print("RANK-OK", rank, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
