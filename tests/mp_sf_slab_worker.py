"""Worker of tests/test_gpu_sf_slabs.py: one rank per GPU (torchrun), structure factors of the slab-decomposed box with the
all-to-all over NCCL.  Rank 0 also steps the WHOLE box on its own GPU with the one-GPU accumulator and compares."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bflbm_b200 as b  # noqa: E402
from bflbm_b200.distributed import SlabLattice  # noqa: E402


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    nx, ny, nz, lz = 40, 24, 24 * world, 4
    prm = b.Params(kBT=1e-5, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0, tau_f=0.7, tau_g=0.55, seed=4711)
    pairs = b.REFERENCE_PAIRS
    scaling = np.linspace(0.5, 2.0, len(pairs))
    S = SlabLattice(nx, ny, nz, params=prm, device=local)
    S.lat.set_tiling(lz)
    S.init_droplet(0.3)
    with b.SlabStructureFactor(S, pairs, scaling) as sf:
        for _ in range(4):
            S.step(3)
            sf.fort_structure()
        got = sf.result(zero_avg=True, imag=True)
        ok = sf.samples == 4
    err = 0.0
    if rank == 0:
        with b.Lattice(nx, ny, nz, params=prm, device=local) as W:
            W.set_tiling(lz)
            W.init_droplet(0.3)
            with b.StructureFactor(W, pairs, scaling) as sw:
                for _ in range(4):
                    W.step(3)
                    sw.fort_structure()
                wr, wi = sw.result(zero_avg=True, imag=True)
        scale = np.abs(wr + 1j * wi).max(axis=(1, 2, 3), keepdims=True)
        err = max((np.abs(got[0] - wr) / scale).max(), (np.abs(got[1] - wi) / scale).max())
        ok &= bool(err <= 1e-12)
    else:
        ok &= got is None
    t = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    S.lat.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MP_SF_SLAB_OK" if int(t.item()) == 1 else "MP_SF_SLAB_MISMATCH", world, f"max rel err {err:.3e}", flush=True)
    sys.exit(0 if int(t.item()) == 1 else 1)


if __name__ == "__main__":
    main()
