"""Worker of tests/test_heating_gpu.py::test_one_process_per_gpu (launched by torch.distributed.run, one rank per GPU).
Every rank joins the device group with rtb200_create_rank, sets dust and heating (the same scalars on every rank), runs
the host-buffer and the resident diffuse call collectively, and checks ITS slab of the heating fields: equal to the
numpy pass (tests/heating_oracle.py) of the group's own J bit for bit, and to the single-device fields it computes
itself within 1e-13."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist

    import heating_oracle as HO
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
    gamma, width = W.uvb_heating(bg["table"], bg["alpha"])
    bd0 = W.uvb_dust_beta(bg["alpha"], W.synthetic_spectra()["a_dust"])
    for g, scale in ((W.uniform_grid(24, seed=3), 1.0), (W.nested_grid(6, 2, W.central_box_refine(0.2, 0.7, levels=2), seed=5), 1e-3)):
        N = g["level"].size
        g["abun2"] = np.random.default_rng(11).uniform(0.005, 0.04, N)
        bd = bd0 * (np.max(g["HI"] * beta[0][0]) / np.max(g["rho"] / W.MP * bd0[0] * g["abun2"] / 0.2))
        for albedo, max_iter in (((0.0, 0.0, 0.0), 1), ((0.3, 0.5, 0.7), 3)):
            one = rt.Transport(device=local)
            one.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
            one.set_dust(2, bd, albedo=albedo, max_iterations=max_iter, tolerance=0.0)
            one.set_heating(gamma, width)
            one.diffuse(uvb * scale, beta)
            H1 = HO.fields(one.last_heating())
            one.close()
            grp = rt.Transport(device=local, comm=(world, rank, new_uid()))
            grp.set_grid(g["nx"], g["level"], g["HI"], g["HeI"], g["HeII"], g["rho"], g["abun2"], g["box_size"])
            off, cnt, _, _, _ = grp.slab(0)
            grp.set_dust(2, bd, albedo=albedo, max_iterations=max_iter, tolerance=0.0)
            grp.set_heating(gamma, width)
            J = np.full((3, N), -1.0)
            grp.diffuse(uvb * scale, beta, out=J)
            H = HO.fields(grp.last_heating())
            sl = slice(off, off + cnt)
            want = HO.heating(J[:, sl], {k: g[k][sl] for k in ("HI", "HeI", "HeII", "rho", "abun2")}, gamma, width, 2, bd,
                              albedo)
            assert np.array_equal(H[:, sl], want)
            err = rel_err(H[:, sl], H1[:, sl], floor=1e-300)
            assert err < 1e-13, err
            grp.diffuse_resident(uvb * scale, beta)
            grp.sync()
            assert np.array_equal(HO.fields(grp.last_heating())[:, sl], H[:, sl])
            print(f"rank {rank}: N={N} albedo {albedo}: heating fields err vs single {err:.3e}", flush=True)
            grp.close()
    dist.barrier()
    print("RANK-OK", rank, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
