"""Time one structure-factor accumulate of the slab-decomposed box (include/bflbm_sf_slab.h) against 100 steps of the same slabs
(the reference's out_SF_step).  Run under torch.distributed.run, one rank per GPU:

    python -m torch.distributed.run --nproc-per-node=N tools/sf_slab_timing.py [--n 512] [--repeats 3]

The accumulate is timed round by round with CUDA events on the slab's stream and split into the observer, 2-D FFT + pack,
exchange (NCCL all-to-all) and z-FFT + accumulate; the observer is timed on its own afterwards (same kernel, same slab) and
taken out of round 0's begin.  With one rank the existing whole-box accumulator (bflbm_sf_accumulate) is timed on the same box
too.  Rank 0 prints one JSON line with the card's name and power limit, read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bflbm_b200 as b  # noqa: E402
from bflbm_b200.distributed import SlabLattice  # noqa: E402
from bflbm_b200.structure_factor import _slab_check  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def max_over_ranks(x: float) -> float:
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed_accumulate(sf, S):
    """One fort_structure with events between its phases; returns per-phase milliseconds (begin, exchange, end summed over
    rounds) and the total."""
    lib = sf.lib
    h = sf.h[0]
    ev = []
    stream = S.stream
    with torch.cuda.stream(stream):
        for v in range(sf.rounds):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record(stream)
            _slab_check(lib.bflbm_sf_slab_begin(h, v), "bflbm_sf_slab_begin")
            e[1].record(stream)
            sf._exchange()
            e[2].record(stream)
            _slab_check(lib.bflbm_sf_slab_end(h, v), "bflbm_sf_slab_end")
            e[3].record(stream)
            ev.append(e)
    stream.synchronize()
    begin = sum(e[0].elapsed_time(e[1]) for e in ev)
    exch = sum(e[1].elapsed_time(e[2]) for e in ev)
    end = sum(e[2].elapsed_time(e[3]) for e in ev)
    return begin, exch, end, ev[0][0].elapsed_time(ev[-1][3])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=100)
    a = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    n = a.n
    name, limit = card()
    prm = b.Params(kBT=1e-5, alpha0=0.0, seed=7)  # examples/Parameters.mixture_noise
    S = SlabLattice(n, n, n, params=prm, device=local)
    S.init_mixture()
    S.step(5)
    res = dict(gpu=name, power_limit=limit, world=world, box=[n, n, n], pairs=len(b.REFERENCE_PAIRS))
    sf = b.SlabStructureFactor(S, b.REFERENCE_PAIRS)
    res["rounds"] = sf.rounds
    sf.fort_structure()  # warm-up: plans, NCCL communicators, first launches
    runs = []
    for _ in range(a.repeats):
        dist.barrier()
        runs.append(timed_accumulate(sf, S))
    runs = [[max_over_ranks(x) for x in r] for r in runs]
    begin, exch, end, total = (float(np.median([r[i] for r in runs])) for i in range(4))
    sf.close()
    # the observer on its own: the same kernel into a buffer of the same size
    buf = torch.empty(22 * S.lat.nz * n * n, dtype=torch.float64, device="cuda")
    obs = []
    for _ in range(a.repeats + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(S.stream)
        b.lattice._check(S.lat.lib.bflbm_get_hydrovars_device(S.lat.h, ctypes.c_void_p(buf.data_ptr())))
        e1.record(S.stream)
        S.stream.synchronize()
        obs.append(e0.elapsed_time(e1))
    observer = max_over_ranks(float(np.median(obs[1:])))
    del buf
    torch.cuda.empty_cache()
    # 100 steps of the same slabs (halo messages over NCCL, as in the accumulate)
    S.step(5)
    steps = []
    for _ in range(2):
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(S.stream)
        S.step(a.steps)
        e1.record(S.stream)
        S.stream.synchronize()
        steps.append(max_over_ranks(e0.elapsed_time(e1)))
    res.update(fort_structure_ms=round(total, 2), observer_ms=round(observer, 2), fft2d_pack_ms=round(begin - observer, 2),
               exchange_ms=round(exch, 2), zfft_accumulate_ms=round(end, 2), steps=a.steps, steps_ms=round(min(steps), 2),
               accumulate_over_steps=round(total / min(steps), 3),
               bytes_sent_per_rank=16 * sum(slab_counts(n, world, rank)) * res["rounds"])
    if world == 1:  # the existing whole-box accumulator on the same box
        with b.StructureFactor(S.lat, b.REFERENCE_PAIRS) as sw:
            sw.fort_structure()
            t = []
            for _ in range(a.repeats):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                sw.fort_structure()
                e1.record()
                torch.cuda.synchronize()
                t.append(e0.elapsed_time(e1))
            res["whole_box_sf_accumulate_ms"] = round(float(np.median(t)), 2)
    S.lat.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(res), flush=True)


def slab_counts(n, world, rank):
    """Complex values this rank sends to the OTHER ranks per variable (its own block stays local)."""
    from bflbm_b200.distributed import slab_bounds
    _, nzl = slab_bounds(n, world, rank)
    nxh = n // 2 + 1
    base, rem = divmod(nxh, world)
    return [nzl * n * (base + (1 if d < rem else 0)) for d in range(world) if d != rank]


if __name__ == "__main__":
    main()
