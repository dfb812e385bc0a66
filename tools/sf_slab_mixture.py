"""BASELINE config 4 evidence: S(k) of the 512^3 fluctuating mixture (examples/Parameters.mixture_noise: alpha0 = 0, kBT = 1e-5)
on a box split over the ranks, accumulated with the slab-decomposed structure factor (include/bflbm_sf_slab.h).  Mixture.ipynb
expects S flat in k; this records the shell means of S_rho_rho / (kBT / cs2) and S_phi_phi / (kBT / cs2) with the estimator of
tests/stats.py.  Run under torch.distributed.run, one rank per GPU:

    python -m torch.distributed.run --nproc-per-node=8 tools/sf_slab_mixture.py [--n 512] [--warmup 500] [--samples 5] [--every 100]

Rank 0 prints one JSON line with the card's name and power limit."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bflbm_b200 as b  # noqa: E402
import stats  # noqa: E402
from bflbm_b200.distributed import SlabLattice  # noqa: E402
from sf_slab_timing import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=500)
    ap.add_argument("--samples", type=int, default=5)
    ap.add_argument("--every", type=int, default=100)
    ap.add_argument("--bins", type=int, default=6)
    a = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    name, limit = card()
    n, kBT = a.n, 1e-5
    S = SlabLattice(n, n, n, params=b.Params(kBT=kBT, alpha0=0.0, seed=2024), device=local)
    S.init_mixture()
    t0 = time.time()
    S.step(a.warmup)
    pairs = [(0, 0), (1, 1)]
    with b.SlabStructureFactor(S, pairs) as sf:
        for _ in range(a.samples):
            S.step(a.every)
            sf.fort_structure()
        s = sf.result(zero_avg=True)
    mass = torch.tensor(S.lat.total_mass(), dtype=torch.float64, device="cuda")
    dist.all_reduce(mass)
    torch.cuda.synchronize()
    wall = time.time() - t0
    S.lat.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        est = stats.StructureFactor(pairs)
        est.acc, est.n = np.fft.ifftshift(s, axes=(1, 2, 3)), 1  # the estimator shifts and zeroes k = 0 itself
        k, shells = est.shell_means(a.bins)
        norm = kBT / stats.CS2
        print(json.dumps(dict(gpu=name, power_limit=limit, world=world, box=[n, n, n], kBT=kBT, alpha0=0.0,
                              steps=a.warmup + a.samples * a.every, warmup=a.warmup, samples=a.samples, every=a.every,
                              mean_rho=float(mass[0]) / n ** 3, mean_phi=float(mass[1]) / n ** 3,
                              k_shell=[round(float(x), 4) for x in k],
                              S_rho_rho_over_kBT_cs2=[round(float(x), 4) for x in shells[0] / norm],
                              S_phi_phi_over_kBT_cs2=[round(float(x), 4) for x in shells[1] / norm],
                              wall_s=round(wall, 1))), flush=True)


if __name__ == "__main__":
    main()
