#!/usr/bin/env python
"""bench.py -- MLUPS of the fluctuating binary D3Q19 step on N B200s (weak scaling), with roofline and CPU baseline.

Contract (one JSON line on stdout from rank 0):
  metric   "MLUPS (fp64 binary fluct D3Q19)"  -- BASELINE.json's metric
  value    whole-job million lattice-cell updates per second, state resident in HBM, CUDA-event timed,
           max over ranks
  e2e      same metric through the C ABI with HOST buffers: output intervals of the reference driver
           (plot_int = 200 steps, main_run_job.cpp:90): restart upload of fold/gold (LBM_init) from pinned
           host memory -> steps -> download of the 9 hydrovsbar fields (what WriteOutput writes); three
           consecutive intervals with the asynchronous transfer calls (next checkpoint and last frame travel
           next to the steps), and one interval with the blocking calls beside it (e2e.serial_interval)
  roofline dominant kernel (fused collide+stream+density-scatter) against the MEASURED HBM copy bandwidth
           (MEASURED_PEAKS.json), algorithmic bytes = 608 B per cell update (SURVEY.md 8(d))
  cpu_baseline  the reference's own LBM_timestep (oracle/_ref, OpenMP over the shim loops) or the C port,
           timed on this host on a bounded sample

`--impl reference` times the reference's CPU implementation alone (rank 0 only).
`--dump-outputs DIR` (one GPU) writes what the timed steps left on the device, a fixed sample of cells, as DIR/*.npy: two
builds run with the same arguments can be compared output for output (dump_outputs below).
A "step" is one LBM_timestep of the whole lattice.  Workload at every N: 512^3 cells per GPU (config 5 of
BASELINE.json, weak scaling; slabs stacked along z), mixture rho = phi = 1 with kBT = 1e-5, alpha0 = 1.5.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MLUPS (fp64 binary fluct D3Q19)"
UNIT = "MLUPS"
BYTES_PER_CELL = 608  # 2 species x 19 populations x (1 read + 1 write) x 8 B
PARAMS = dict(kBT=1e-5, tau_f=0.5, tau_g=0.5, alpha0=1.5, alpha1=0.0, kappa=4.0, rho_lo=0.0, rho_hi=1.0, seed=12345)
E2E_STEPS = 200  # reference plot_int, main_run_job.cpp:90


def cells_local_hint(a, nzl):
    return a.nx * a.ny * nzl


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nx", type=int, default=512)
    ap.add_argument("--ny", type=int, default=512)
    ap.add_argument("--nz", type=int, default=512, help="planes PER GPU (weak scaling) / of the whole box (strong scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, BASELINE configs[4]): nz planes per GPU; strong (configs[3]): nz planes in total, split over the GPUs")
    ap.add_argument("--algo", default="fused", choices=["fused", "twopass", "auto"],
                    help="auto = the library's own choice (two-pass kernels for whole boxes <= 150k cells)")
    ap.add_argument("--kbt", type=float, default=PARAMS["kBT"])
    ap.add_argument("--brick-lz", type=int, default=0)
    ap.add_argument("--halo", default="peer", choices=["peer", "nccl"],
                    help="N > 1: ghost exchange by peer-to-peer stores into CUDA-IPC-mapped mailboxes (default) or NCCL send/recv")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=E2E_STEPS)
    ap.add_argument("--e2e-intervals", type=int, default=3, help="restart -> steps -> frame intervals of the pipelined e2e leg")
    ap.add_argument("--cpu-size", type=int, default=128, help="edge of the CPU arm's sample box (128^3: 2.6 GB, out of L3)")
    ap.add_argument("--cpu-steps", type=int, default=0, help="0 = sized for ~10-20 s")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU: after the timed steps write f, g (populations) and the 22 hydrovs fields at a fixed seeded sample of "
                         "cells as DIR/{f,g,hydrovars}.npy (float64)")
    return ap.parse_args()


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); power.append(float(p[2]))
            except ValueError:
                continue
            for nme, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(index):
    """Pins this rank to the CPUs of the NUMA node its GPU hangs off, BEFORE the pinned host buffers are allocated (first touch puts
    their pages on that node).  Round 1: eight ranks uploading 40.8 GB each from one node's memory fell from 48 to 18 GB/s per GPU.
    Best effort; returns a description for the JSON line."""
    try:
        bus = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=10).stdout.strip().lower()
        bus = bus[4:] if len(bus) > 12 else bus  # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "single NUMA node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"rank bound to NUMA node {node} ({len(cpus)} cpus) of GPU {index}"
        return "no usable cpus on the GPU's node"
    except Exception as e:  # noqa
        return f"not bound ({type(e).__name__})"


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------- CPU baseline
def host_cores():
    """Cores this process may use.  Deliberately NOT OMP_NUM_THREADS: torch.distributed.run exports OMP_NUM_THREADS=1 to
    its workers, which in round 1 made the N >= 2 reference arm a 1-core run and the N = 1 arm an all-core run."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _cpu_oracle(size, kbt):
    # the checkers are built by __graft_entry__.build(); the bench only loads them, so it can run from a read-only tree
    from oracle import oracle as om
    prm = dict(kBT=kbt, tau_f=PARAMS["tau_f"], tau_g=PARAMS["tau_g"], alpha0=PARAMS["alpha0"], alpha1=0.0, kappa=PARAMS["kappa"])
    if om.RefOracle.available(fast=True):
        O = om.RefOracle(size, size, size, fast=True)
        O.set_params(**prm)
        O.set_rng(2, 12345)  # per-thread mt19937 + std::normal_distribution behind amrex::RandomNormal
        return O, "reference", "reference headers (LBM_binary.H, LBM_d3q19.H) over oracle/shim, -O3 -march=x86-64-v3, OpenMP over the shim loops"
    O = om.PortOracle(size, size, size, fast=True)
    O.set_params(**prm, rho_lo=0.0, rho_hi=1.0)
    return O, "port", "C port oracle/bflbm_oracle.c, -O3 -march=x86-64-v3, OpenMP"


def cpu_reference_run(size, kbt, steps=0, warmup=1, budget_s=10.0):
    """Times the reference's LBM_timestep on the host cores, twice: on ALL cores this process may use, and on ONE core
    (the reference's shipped build is serial, GNUmakefile:16-19: that is the faithful figure).  Thread counts are set
    explicitly through omp_set_num_threads.  steps = 0: sized for ~budget_s seconds.
    Returns (cpu_baseline dict, seconds per all-core step)."""
    O, kind, how = _cpu_oracle(size, kbt)
    cells = size ** 3

    def timed(nthreads, steps, warmup, budget):
        O.set_num_threads(nthreads)
        O.init_mixture()
        t0 = time.perf_counter()
        O.step(max(1, warmup))  # first step also takes the page faults
        per = (time.perf_counter() - t0) / max(1, warmup)
        if steps <= 0:
            steps = int(max(1, min(400, budget / max(per, 1e-4))))
        t0 = time.perf_counter()
        O.step(steps)
        dt = time.perf_counter() - t0
        return cells * steps / dt / 1e6, steps, dt

    cores = host_cores()
    v_all, n_all, dt_all = timed(cores, steps, warmup, budget_s)
    v_one, n_one, dt_one = timed(1, 0, 1, budget_s / 2)
    res = {"value": v_all, "unit": UNIT, "cores": cores, "kind": kind,
           "one_core": {"value": v_one, "unit": UNIT, "cores": 1, "steps": n_one, "seconds": dt_one},
           "sample": f"mixture {size}^3 ({cells * 154 * 8 / 1e9:.1f} GB of reference MultiFabs: out of cache like the real job), "
                     f"kBT={kbt:g}; all {cores} cores: {n_all} steps of LBM_timestep in {dt_all:.1f} s; 1 core: {n_one} steps in {dt_one:.1f} s ({how})"}
    O.close()
    return res, dt_all / n_all


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # K timed "steps" after W warm-up steps, each one LBM_timestep of the cpu_size^3 sample box, on all host cores;
    # the same measurement at every --gpus N (the CPU arm does not depend on N)
    res, sec_per_step = cpu_reference_run(a.cpu_size, a.kbt, steps=a.steps if a.cpu_steps <= 0 else a.cpu_steps, warmup=max(1, a.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"mixture rho=phi=1, kBT={a.kbt:g}, alpha0={PARAMS['alpha0']}, tau=1/2; bounded sample {a.cpu_size}^3 of the "
                               f"{a.nx}x{a.ny}x{a.nz * a.gpus} job", "sample_cells": a.cpu_size ** 3},
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- GPU arm
def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    import bflbm_b200 as b

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the b200 arm)")
    if a.dump_outputs and world > 1:
        raise SystemExit("bench.py --dump-outputs: one GPU only")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if a.scaling == "strong":
        if a.nz % world:
            raise SystemExit("bench.py --scaling strong: --nz must be divisible by the number of GPUs")
        nzl, nz_global = a.nz // world, a.nz
    else:
        nzl = a.nz
        nz_global = nzl * world
    prm = b.Params(**{**PARAMS, "kBT": a.kbt})
    stream = torch.cuda.Stream()  # a real (non-default) stream: the library launches on it and the events are recorded on it
    torch.cuda.set_stream(stream)

    halo = None
    slab_parity = None
    if world == 1:
        lat = b.Lattice(a.nx, a.ny, nzl, params=prm, device=local)
        stepper = lat
    else:
        from bflbm_b200.distributed import SlabLattice
        # correctness evidence in the line itself: the very path that is about to be timed, on a small box, against the
        # whole box stepped on this rank's GPU -- bitwise, noise on (untimed)
        slab_parity, halo = slab_parity_check(b, np, torch, dist, local, a.halo)
        stepper = SlabLattice(a.nx, a.ny, nz_global, params=prm, device=local, peer=(halo == "peer"))
        lat = stepper.lat
        stepper.stream = stream  # the NCCL exchange must be queued on the stream the library launches on
    lat.set_stream(stream.cuda_stream)
    if a.algo != "auto":
        lat.set_algorithm(a.algo)
    if a.brick_lz:
        lat.set_tiling(a.brick_lz)
    stepper.init_mixture()
    cells_local = a.nx * a.ny * nzl
    cells = cells_local * world

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- timed region: W warm-up steps, then exactly K steps, CUDA events on the launching stream -------
    stepper.step(a.warmup)
    barrier()
    # Duration of the dominant kernel: CUDA events around every launch, read back after the timed region (library mode 2:
    # no host synchronisation per step).  Event records make the steps plain launches instead of graph replays and put a
    # slab step on one stream, so they go INTO the timed region only where that costs nothing: one GPU, steps of
    # milliseconds.  Small boxes and slabs are timed undisturbed and profiled in a second pass of the same K steps.
    profile_in_timed = world == 1 and cells_local_hint(a, nzl) >= (1 << 24) and os.environ.get("BFLBM_BENCH_PROFILE_IN_TIMED", "1") != "0"
    if profile_in_timed:
        lat.set_profiling(2)
        barrier()
    launches0 = lat.kernel_launches
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    stepper.step(a.steps)
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if profile_in_timed:
        prof_timed = lat.profile()
        lat.set_profiling(0)
    launches = lat.kernel_launches - launches0
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    value = cells * a.steps / (ms * 1e-3) / 1e6
    nan_count = 0
    try:
        nan_count = lat.check_nan()
    except b.BflbmError:
        nan_count = -1
    mass = list(lat.total_mass())  # global species masses after the timed steps (conserved exactly: = cells for the mixture)
    if world > 1:
        mt = torch.tensor(mass, device="cuda", dtype=torch.float64)
        dist.all_reduce(mt, op=dist.ReduceOp.SUM)
        mass = [float(v) for v in mt.tolist()]
    if a.dump_outputs:  # before anything steps the lattice again
        dump_outputs(b, np, torch, lat, a.dump_outputs)

    # ---- dominant kernel alone: per-kernel events inside the library, same step count -------------------
    roofline = None
    peak, peak_src = measured_peak()
    if profile_in_timed:
        per_kernel, nprof = prof_timed
        kernel_src = "CUDA events around every launch of the timed region (read back after it)"
    else:
        lat.set_profiling(True)
        stepper.step(a.steps)
        lat.sync()
        per_kernel, nprof = lat.profile()
        lat.set_profiling(False)
        kernel_src = "second pass of the same K steps right after the timed region (plain launches, events around every launch)"
    if nprof > 0 and per_kernel[0] > 0:
        achieved = BYTES_PER_CELL * cells_local / (per_kernel[0] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                    "peak_source": peak_src, "kernel": {"fused": "k_step_fused", "twopass": "k_step_twopass", "auto": "library's choice"}[a.algo],
                    "kernel_ms": per_kernel[0], "kernel_ms_source": kernel_src, "other_kernels_ms": {"fold_or_wrap": per_kernel[1], "pack_or_density": per_kernel[2],
                                                                     "unpack_or_wrap": per_kernel[3]},
                    "algorithmic_bytes_per_cell": BYTES_PER_CELL,
                    "step_frac_of_roofline": (BYTES_PER_CELL * cells_local / (ms / a.steps * 1e-3) / 1e9) / peak}
        # DRAM bytes of one launch: an ncu capture of ONE configuration (profiles/traffic.json), not a measurement of this run.
        # Reported only when this run is that configuration (same cells per GPU, kernel variant); otherwise null.
        tr = os.path.join(ROOT, "profiles", "traffic.json")
        roofline["traffic_source"] = None
        if os.path.exists(tr):
            try:
                t = json.load(open(tr))
                same = (t.get("nx"), t.get("ny"), t.get("nz_local")) == (a.nx, a.ny, nzl) and bool(t.get("noise")) == (a.kbt > 0) and \
                    t.get("algorithm", "fused") == a.algo and bool(t.get("rate1", True)) == (os.environ.get("BFLBM_RATE1", "1") != "0")
                if same:
                    roofline["traffic"] = t.get("bytes_per_launch")
                    roofline["traffic_source"] = "ncu capture of this configuration, not of this run: " + str(t.get("source"))
                else:
                    roofline["traffic_source"] = "no ncu capture for this configuration"
            except Exception:
                pass

    # ---- end to end through the C ABI with host buffers ---------------------------------------------------
    e2e = None
    if not a.no_e2e:
        e2e = run_e2e(a, b, np, torch, lat, stepper, world, cells, cells_local)

    cpu = None
    if rank == 0 and not a.no_cpu and world == 1:
        cpu, _ = cpu_reference_run(a.cpu_size, a.kbt, steps=a.cpu_steps)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"{a.scaling}-scaling {a.nx}x{a.ny}x{nzl} cells per GPU ({a.nx}x{a.ny}x{nz_global} total), fluctuating binary "
                                   f"D3Q19 mixture rho=phi=1, kBT={a.kbt:g}, alpha0={PARAMS['alpha0']}, tau_f=tau_g=1/2 "
                                   f"(BASELINE.json configs[{4 if a.scaling == 'weak' else 3}])",
                       "cells_per_gpu": cells_local, "algorithm": a.algo, "parallelism": f"z-slabs x{world}",
                       "l2": "working set (two lattices, %.1f GB per GPU) far exceeds the 126 MB L2; no flush needed" % (lat.device_bytes / 1e9),
                       "timed_window_s": ms * 1e-3,  # a sustained run (>= 1 s) reaches the board power limit and runs ~3 % slower (DESIGN.md section 6)
                       "nonfinite_after_run": nan_count, "mass_rho": mass[0], "mass_phi": mass[1], "cells": cells,
                       "halo": None if world == 1 else ("peer-to-peer stores into CUDA-IPC-mapped mailboxes, device-side flags (no collective per step)"
                                                        if halo == "peer" else "NCCL send/recv (torch.distributed)"),
                       "slab_parity": slab_parity, "numa": numa},
            "clocks": clocks, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_CELLS = 1 << 16  # cells written by --dump-outputs: 60 float64 per cell, 31.5 MB in all


def dump_outputs(b, np, torch, lat, out_dir):
    """What a caller of the timed steps receives -- the populations f, g (fold, gold) and the 22 hydrovs fields -- at DUMP_CELLS
    cells drawn with a fixed seed (every cell of a smaller box), written as float64 arrays (components, cells) to
    out_dir/{f,g,hydrovars}.npy.  The fields are copied device to device and sampled there: at 512^3 the full populations
    are 40.8 GB."""
    from bflbm_b200.lattice import _check
    n = lat.nx * lat.ny * lat.nz
    cells = np.arange(n) if n <= DUMP_CELLS else np.sort(np.random.default_rng(0).choice(n, DUMP_CELLS, replace=False))
    dev = torch.device("cuda", lat.device)
    cells = torch.from_numpy(cells).to(dev)
    f = torch.empty((b.NVEL, n), dtype=torch.float64, device=dev)
    g = torch.empty_like(f)
    _check(lat.lib.bflbm_get_populations_device(lat.h, f.data_ptr(), g.data_ptr()))
    out = {"f": f[:, cells].cpu().numpy(), "g": g[:, cells].cpu().numpy()}
    # beside the lattice (91.4 GB at 512^3) there are f and g together (40.8 GB), then hydrovs alone (23.6 GB); the cache is
    # emptied in between and at the end, so the library's later allocations (the e2e leg's staging area) find the memory free
    del f, g
    torch.cuda.empty_cache()
    h = torch.empty((b.NHYDRO, n), dtype=torch.float64, device=dev)
    _check(lat.lib.bflbm_get_hydrovars_device(lat.h, h.data_ptr()))
    out["hydrovars"] = h[:, cells].cpu().numpy()
    del h
    torch.cuda.empty_cache()
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def slab_parity_check(b, np, torch, dist, local, want):
    """Slabs over the ranks of this job vs the whole box on one GPU: every rank compares its slab bit for bit after 12
    fluctuating steps and a restart.  Also decides the halo transport: peer-to-peer stores through CUDA-IPC-mapped mailboxes
    (default), NCCL send/recv if the mapping is refused (or --halo nccl)."""
    from bflbm_b200.distributed import SlabLattice
    world = dist.get_world_size()
    nx, ny, nz, lz = 64, 48, 16 * world, 4
    prm = b.Params(kBT=1e-5, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0, tau_f=0.5, tau_g=0.5, seed=4711)
    halo = want
    S = None
    if halo == "peer":
        ok_here = 1
        try:
            S = SlabLattice(nx, ny, nz, params=prm, device=local, peer=True)
        except b.BflbmError:
            ok_here = 0
        t = torch.tensor([ok_here], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 0:
            halo = "nccl"
            if S is not None:
                S.lat.close()
            S = None
    if S is None:
        S = SlabLattice(nx, ny, nz, params=prm, device=local, peer=False)
    S.lat.set_tiling(lz)
    S.init_droplet(0.3)
    ok = True
    with b.Lattice(nx, ny, nz, params=prm, device=local) as whole:
        whole.set_tiling(lz)
        whole.init_droplet(0.3)
        sl = slice(S.z0, S.z0 + S.nzl)
        for _ in range(3):
            S.step(4)
            whole.step(4)
            ok &= bool(np.array_equal(whole.hydrovars()[:, sl], S.lat.hydrovars()))
        fw, gw = whole.populations()
        fs, gs = S.lat.populations()
        ok &= bool(np.array_equal(fw[:, sl], fs) and np.array_equal(gw[:, sl], gs))
    if halo == "peer":
        ok &= S.lat.halo_error() == 0
    S.lat.close()
    t = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return ("bitwise" if int(t.item()) == 1 else "MISMATCH"), halo


def run_e2e(a, b, np, torch, lat, stepper, world, cells, cells_local):
    """The reference driver's restart -> steps -> frame cycle through the public API with HOST buffers, wall clock.

    One interval = upload of a host checkpoint (LoadSingleMultiFab + LBM_init, main_run_job.cpp:244-268), `--e2e-steps`
    steps, download of hydrovsbar to the host (the frame the driver writes, :372-385).  Measured twice:
      serial     one interval with the blocking calls (bflbm_init_from_populations[_slab], bflbm_step, bflbm_get_hydrovars_bar);
      pipelined  `--e2e-intervals` consecutive intervals (an ensemble of restarts) with the asynchronous calls: the checkpoint
                 of interval i+1 is staged and the frame of interval i-1 is downloaded next to the steps of interval i.  Every
                 byte still crosses PCIe inside the timed region; the first upload and the last download are exposed.
    The line's e2e.value is the pipelined figure; the serial one is reported beside it."""
    import torch.distributed as dist
    nsteps, M = a.e2e_steps, max(1, a.e2e_intervals)
    ghosted = world > 1
    try:
        out = torch.empty((9, lat.nz, lat.ny, lat.nx), dtype=torch.float64, pin_memory=True).numpy()
        pinned = True
    except Exception:
        out = np.empty((9, lat.nz, lat.ny, lat.nx))
        pinned = False
    # the host checkpoint (untimed)
    if ghosted:
        fg = stepper.host_checkpoint()
        f, g = fg[0], fg[1]
    else:
        shape = (19, lat.nz, lat.ny, lat.nx)
        try:
            f = torch.empty(shape, dtype=torch.float64, pin_memory=True).numpy()
            g = torch.empty(shape, dtype=torch.float64, pin_memory=True).numpy()
        except Exception:
            pinned = False
            f, g = np.empty(shape), np.empty(shape)
        from bflbm_b200.lattice import _check
        _check(lat.lib.bflbm_get_populations(lat.h, f.ctypes.data, g.ctypes.data))
    h2d = f.nbytes + g.nbytes
    d2h = out.nbytes

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(vals, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    # ---- serial: one interval, blocking calls --------------------------------------------------------------
    barrier()
    t0 = time.perf_counter()
    if ghosted:
        stepper.init_from_populations_slab(f, g)
    else:
        lat.init_from_populations(f, g)      # returns when the host buffers are free again
    t1 = time.perf_counter()
    stepper.step(nsteps)
    lat.sync()
    t2 = time.perf_counter()
    from bflbm_b200.lattice import _check
    _check(lat.lib.bflbm_get_hydrovars_bar(lat.h, out.ctypes.data))
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    dt, up, st, down = max_over_ranks([t3 - t0, t1 - t0, t2 - t1, t3 - t2])
    mass_serial = float(out[0].sum())
    serial = {"value": cells * nsteps / dt / 1e6, "unit": UNIT, "seconds": dt, "phases_s": {"upload": up, "steps": st, "download": down},
              "h2d_gb_per_s_per_gpu": h2d / up / 1e9, "result_mass_rho": mass_serial,
              "what": "bflbm_init_from_populations%s(host f,g) + %d steps + bflbm_get_hydrovars_bar(host), blocking calls" % ("_slab + halo refresh" if ghosted else "", nsteps)}

    # ---- pipelined: M intervals, asynchronous calls ------------------------------------------------------------
    # the staging area must fit beside the lattice on every rank; otherwise the serial interval is the e2e figure
    ok_here, why = 1, ""
    try:   # untimed probe of the whole route: allocates the staging area outside the timed region, like the lattice itself
        if os.environ.get("BFLBM_BENCH_NO_STAGING") == "1":   # test hook: take the fallback below
            raise b.BflbmError("staging switched off by BFLBM_BENCH_NO_STAGING")
        lat.stage_populations(f, g, ghosted=ghosted)
        stepper.init_from_staged()
        lat.hydrovars_bar_async(out)
        lat.download_wait()
    except b.BflbmError as err:
        ok_here, why = 0, str(err)
    all_ok = -max_over_ranks([-ok_here])[0] == 1
    if not all_ok:
        try:
            lat.release_staging()
        except b.BflbmError:
            pass
        return {"value": serial["value"], "unit": UNIT, "h2d_bytes_per_step": h2d / nsteps, "d2h_bytes_per_step": d2h / nsteps,
                "steps_per_interval": nsteps, "intervals": 1, "seconds": serial["seconds"], "pinned_host": pinned, "what": serial["what"],
                "phases_s": serial["phases_s"], "result_mass_rho": mass_serial,
                "pipelined": "unavailable: " + (why or "another rank could not allocate its staging area")}
    barrier()
    t0 = time.perf_counter()
    lat.stage_populations(f, g, ghosted=ghosted)   # interval 0: nothing to hide behind
    masses = []
    for i in range(M):
        stepper.init_from_staged()
        if i + 1 < M:
            lat.stage_populations(f, g, ghosted=ghosted)   # travels during this interval's steps
        stepper.step(nsteps)
        if i > 0:
            lat.download_wait()                    # frame i-1 has long arrived: read it before `out` is reused
            masses.append(float(out[0, ::max(1, lat.nz // 8)].sum()))
        lat.hydrovars_bar_async(out)               # frame i travels during the next interval's steps
    lat.download_wait()
    lat.sync()
    torch.cuda.synchronize()
    dtp = time.perf_counter() - t0
    dtp, = max_over_ranks([dtp])
    mass = float(out[0].sum())
    masses.append(float(out[0, ::max(1, lat.nz // 8)].sum()))
    lat.release_staging()
    return {"value": cells * nsteps * M / dtp / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d / nsteps, "d2h_bytes_per_step": d2h / nsteps,
            "steps_per_interval": nsteps, "intervals": M, "seconds": dtp, "pinned_host": pinned,
            "what": "%d x [bflbm_stage_populations(host f,g) -> bflbm_init_from_staged%s + %d steps + bflbm_get_hydrovars_bar_async(host)], "
                    "uploads and downloads on the lattice's copy stream next to the steps, first upload and last download exposed; "
                    "wall clock%s" % (M, " + halo refresh" if ghosted else "", nsteps, ", max over ranks" if world > 1 else ""),
            "result_mass_rho": mass, "frames_equal": bool(all(abs(m - masses[0]) <= 1e-9 * abs(masses[0]) for m in masses)),
            "serial_interval": serial}


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference" and args.dump_outputs:
        raise SystemExit("bench.py --dump-outputs: the b200 arm only")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200(args)
