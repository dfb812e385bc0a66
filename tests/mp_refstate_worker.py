"""Worker of tests/test_gpu_reference_state.py: one rank per GPU (torchrun), reference-state noise on NCCL slabs.  The centre of
mass travels through a sum all-reduce after every step; in peer mode the halo still goes by peer stores.  Every rank also steps
the whole box on the brick kernel with the same brick height and compares its slab and the shift bit for bit."""
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
    nx, ny, nz, lz = 32, 16, 16 * world, 4
    prm = b.Params(kBT=1e-5, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0, tau_f=0.7, tau_g=0.55, seed=4711)
    peer = os.environ.get("MP_PEER", "0") == "1"
    # equilibrium profiles: the droplet's densities, displaced by (3, -1, 2) cells along (z, y, x) and modulated
    with b.Lattice(nx, ny, nz, params=b.Params(kBT=0.0, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0), device=local) as eq_lat:
        eq_lat.init_droplet(0.3)
        hb = eq_lat.hydrovars_bar()
    rho_eq, phi_eq = (np.roll(hb[k], (3, -1, 2), axis=(0, 1, 2)).copy() for k in (0, 1))
    zz, yy, xx = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    rho_eq *= 1.0 + 0.3 * np.cos(2 * np.pi * (xx + 0.3) / nx) * np.cos(2 * np.pi * (yy - 1.1) / ny) * np.sin(2 * np.pi * (zz + 0.7) / nz)
    eq = (rho_eq, phi_eq, rho_eq + phi_eq)
    S = SlabLattice(nx, ny, nz, params=prm, device=local, peer=peer)
    S.lat.set_tiling(lz)
    S.set_reference_state(*eq)
    S.init_droplet(0.3)
    sl = slice(S.z0, S.z0 + S.nzl)
    with b.Lattice(nx, ny, nz, params=prm, device=local) as whole:
        whole.set_reference_state(*eq)
        whole.set_algorithm("fused")
        whole.set_tiling(lz)
        whole.init_droplet(0.3)
        ok = True
        for _ in range(5):
            S.step(4)
            whole.step(4)
            ok &= bool(np.array_equal(S.lat.reference_shift(), whole.reference_shift()))
        fw, gw = whole.populations()
        fs, gs = S.lat.populations()
        ok &= np.array_equal(fw[:, sl], fs) and np.array_equal(gw[:, sl], gs)
        ok &= np.array_equal(whole.noise()[0][:, sl], S.lat.noise()[0])
        if peer:
            ok &= S.lat.halo_error() == 0
    t = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    S.lat.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print(f"MP_REFSTATE_{'OK' if int(t.item()) else 'FAIL'} {world} {'peer' if peer else 'nccl'}", flush=True)
    return 0 if int(t.item()) else 1


if __name__ == "__main__":
    sys.exit(main())
