#!/usr/bin/env python
"""Step time of the reference-state noise (USE_REF_STATE) on one B200, and on NCCL slabs.

One GPU, for each box (droplet, radius 0.3, kBT = 1e-5):
  twopass_ref   the thread-per-cell two-pass kernels with the reference state (what a whole box selects by default)
  brick_ref     the one-pass brick kernel with the reference state (bflbm_set_algorithm(h, 0))
  brick_plain   the brick kernel without a reference state
  brick_ref_profile  per-step device time of {step kernel, brick-face fold, centre of mass, -} from the event profiler (a separate
                run: events cost launch overhead); the third interval is k_fold<2> + k_com_chunks + k_com_fold_chunks +
                k_com_shift_planes.
With --nproc-per-node N (N >= 2) the script restarts itself under torchrun: N NCCL ranks, one slab each, reference state on; it
reports ms/step and the time of the centre-of-mass all-reduce alone (4 * nz doubles), measured over the same number of calls.

The equilibrium profiles are the analytic droplet (LBM_binary.H:709-737) displaced by (3, -1, 2) cells: a stand-in for the
equilibrium_* files of a kBT = 0 run, with the same memory traffic.  Timings are host clocks around device-synchronised
work.  The JSON records the GPU name, power limit and maximum SM clock read in the same run; clocks are not locked, and the
card's own power management applies.
usage: tools/refstate_timing.py [--sizes 512 256] [--steps 200] [--warmup 20] [--nproc-per-node N] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bflbm_b200 as b  # noqa: E402

PRM = dict(kBT=1e-5, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0, seed=2024)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()
    except Exception as e:  # the numbers stay, but say that the card could not be named
        return [f"nvidia-smi failed: {e}"]


def equilibrium(n):
    """droplet densities of LBM_init_droplet on an n^3 box, displaced by (3, -1, 2) cells along (z, y, x)"""
    c = np.arange(n, dtype=np.float64)
    rx, ry = (c - n / 2.0)[None, None, :], (c - n / 2.0)[None, :, None]
    rz = (np.arange(n) - n // 2).astype(np.float64)[:, None, None]
    r = np.sqrt(rx * rx + ry * ry + rz * rz)
    rho = (PRM["rho_hi"] - PRM["rho_lo"]) * (1.0 + np.tanh((0.3 * n - r) / np.sqrt(PRM["kappa"]))) / 2.0 + PRM["rho_lo"]
    rho = np.roll(rho, (3, -1, 2), axis=(0, 1, 2))
    phi = (PRM["rho_hi"] + PRM["rho_lo"]) - rho
    return rho, phi, rho + phi


def time_steps(lat, steps, warmup):
    lat.step(warmup)
    lat.sync()
    t = time.perf_counter()
    lat.step(steps)
    lat.sync()
    return (time.perf_counter() - t) * 1e3 / steps


def one_gpu(n, steps, warmup):
    eq = equilibrium(n)
    out = {"box": [n, n, n], "steps": steps, "warmup": warmup}
    for name in ("twopass_ref", "brick_ref", "brick_plain", "brick_ref_profile"):
        with b.Lattice(n, params=b.Params(**PRM)) as lat:
            if name != "brick_plain":
                lat.set_reference_state(*eq)
            if name != "twopass_ref":
                lat.set_algorithm("fused")
            lat.init_droplet(0.3)
            if name == "brick_ref_profile":
                lat.step(warmup)
                lat.set_profiling(2)
                lat.step(steps)
                ms, k = lat.profile()
                out[name] = {"ms_per_step": ms, "steps": k, "intervals": ["step kernel", "brick-face fold", "centre of mass", "-"]}
            else:
                out[name] = {"ms_per_step": time_steps(lat, steps, warmup), "algorithm": lat.last_step()["algorithm"],
                             "device_bytes": lat.device_bytes}
            print(n, name, out[name], flush=True)
    p = out["brick_ref_profile"]["ms_per_step"]
    out["com_share_of_brick_ref_step"] = p[2] / sum(p)
    out["speedup_brick_ref_over_twopass_ref"] = out["twopass_ref"]["ms_per_step"] / out["brick_ref"]["ms_per_step"]
    out["cells_per_s_brick_ref"] = n ** 3 / (out["brick_ref"]["ms_per_step"] * 1e-3)
    return out


def worker(n, steps, warmup, out_path):
    import torch
    import torch.distributed as dist
    from bflbm_b200.distributed import SlabLattice
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    S = SlabLattice(n, n, n, params=b.Params(**PRM), device=local)
    S.set_reference_state(*equilibrium(n))
    S.init_droplet(0.3)
    S.step(warmup)
    S.lat.sync()
    dist.barrier()
    t = time.perf_counter()
    S.step(steps)
    S.lat.sync()
    ms_step = (time.perf_counter() - t) * 1e3 / steps
    dist.barrier()
    t = time.perf_counter()
    with torch.cuda.stream(S.stream):
        for _ in range(steps):
            dist.all_reduce(S.com, op=dist.ReduceOp.SUM)
    S.stream.synchronize()
    ms_ar = (time.perf_counter() - t) * 1e3 / steps
    res = torch.tensor([ms_step, ms_ar], dtype=torch.float64, device="cuda")
    dist.all_reduce(res, op=dist.ReduceOp.MAX)
    if dist.get_rank() == 0:
        with open(out_path, "w") as fh:
            json.dump({"ranks": dist.get_world_size(), "box": [n, n, n], "ms_per_step": res[0].item(),
                       "com_allreduce_ms": res[1].item(), "com_allreduce_share": res[1].item() / res[0].item(),
                       "com_allreduce_bytes": 8 * 4 * n}, fh)
    S.lat.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[512, 256])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--nproc-per-node", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "refstate_timing.json"))
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a.sizes[0], a.steps, a.warmup, a.worker)
    res = {"gpu": gpu_info(), "kBT": PRM["kBT"], "one_gpu": [one_gpu(n, a.steps, a.warmup) for n in a.sizes]}
    if a.nproc_per_node > 1:
        res["slabs"] = []
        for n in a.sizes:
            tmp = a.out + f".slabs{n}.tmp"
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.nproc_per_node}",
                   "--master-addr", "127.0.0.1", "--master-port", "29710", os.path.abspath(__file__), "--sizes", str(n),
                   "--steps", str(a.steps), "--warmup", str(a.warmup), "--worker", tmp]
            subprocess.run(cmd, check=True)
            with open(tmp) as fh:
                res["slabs"].append(json.load(fh))
            os.remove(tmp)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    sys.exit(main())
