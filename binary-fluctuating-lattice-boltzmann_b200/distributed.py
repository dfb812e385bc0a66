"""Slab decomposition of the periodic box over the GPUs of one node: one process per GPU, torch.distributed
for the plumbing (NCCL over NVLink for the ghost messages, gloo in the CPU tests).

The reference's only parallelism is AMReX's box decomposition + FillBoundary (main_run_job.cpp:140-145,
LBM_binary.H:130-131, 312, 353, 553-555: seven ghost fills of 19..22 components x 2 layers per step).
Here the box is cut into P slabs along z (the slowest array axis, so ghost planes are contiguous) and ONE message
of 14 doubles per face cell goes to each z-neighbour per step (include/bflbm.h, "slab halo exchange"):
5+5 populations that stream across the face and the two (rho, phi) partial-sum planes.  There is no other
collective on the data path; the noise is keyed by GLOBAL cell index, so results do not depend on P.
"""
from __future__ import annotations

import ctypes

import numpy as np

from .lattice import Lattice, Params, _check, NVEL


def slab_bounds(nz_global: int, world: int, rank: int) -> tuple[int, int]:
    """(z0, nz_local) of `rank`: contiguous, sizes differ by at most one plane (remainder to the low ranks)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    base, rem = divmod(nz_global, world)
    if base < 2:
        raise ValueError(f"nz={nz_global} is too small for {world} slabs (need >= 2 planes per slab)")
    nzl = base + (1 if rank < rem else 0)
    z0 = rank * base + min(rank, rem)
    return z0, nzl


def neighbours(world: int, rank: int) -> tuple[int, int]:
    """(rank below, rank above) on the periodic ring; side 0 = towards lower z."""
    return (rank - 1) % world, (rank + 1) % world


def exchange_ring(send_lo, send_hi, recv_lo, recv_hi, rank: int, world: int, group=None):
    """Moves send_lo -> lower neighbour's recv_hi and send_hi -> upper neighbour's recv_lo (periodic ring).
    Tensors may live on the GPU (nccl) or the CPU (gloo).  One batched group of two sends and two receives,
    which NCCL runs as a single fused kernel over NVLink."""
    import torch.distributed as dist
    if world == 1:
        recv_hi.copy_(send_lo)
        recv_lo.copy_(send_hi)
        return
    lo, hi = neighbours(world, rank)
    ops = [dist.P2POp(dist.isend, send_lo, lo, group=group), dist.P2POp(dist.isend, send_hi, hi, group=group),
           dist.P2POp(dist.irecv, recv_lo, lo, group=group), dist.P2POp(dist.irecv, recv_hi, hi, group=group)]
    if world == 2:
        # both neighbours are the same peer: order the two messages explicitly (send order = receive order)
        ops = [dist.P2POp(dist.isend, send_lo, lo, group=group), dist.P2POp(dist.irecv, recv_hi, hi, group=group),
               dist.P2POp(dist.isend, send_hi, hi, group=group), dist.P2POp(dist.irecv, recv_lo, lo, group=group)]
    for req in dist.batch_isend_irecv(ops):
        req.wait()


def gather_ring_handles(handle: bytes, rank: int, world: int, group=None) -> tuple[bytes, bytes]:
    """Peer mode plumbing: every rank publishes the 64-byte CUDA-IPC handle of its mailbox (bflbm_peer_ipc_handle); returns the
    handles of (lower neighbour, upper neighbour) on the periodic ring.  The only collective of the peer path, once per run."""
    import torch.distributed as dist
    handles = [None] * world
    if world == 1:
        handles[0] = handle
    else:
        dist.all_gather_object(handles, handle, group=group)
    lo, hi = neighbours(world, rank)
    return handles[lo], handles[hi]


def _device_tensor(ptr: int, n: int, device):
    """float64 torch view of `n` doubles of device memory owned by the C library."""
    import torch

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 3, "strides": None}
    return torch.as_tensor(h, device=device)


class EmulatedSlabs:
    """P slabs of one box held by ONE process on ONE GPU, stepped in lock-step with device-to-device copies in
    place of the NCCL messages.  Exercises exactly the library path a multi-GPU run takes (bflbm_create_slab,
    step_begin / step_end, halo buffers); used by the single-GPU tests of the slab logic.  structure_factor.SlabStructureFactor
    accepts it in place of a SlabLattice and moves its all-to-all blocks by device copies as well.

    zsplit: optional first planes of the slabs plus nz (nslabs + 1 entries) for an uneven cut; default slab_bounds."""

    def __init__(self, nx, ny, nz, nslabs, params: Params | None = None, device: int = 0, brick_lz: int = 0, peer: bool = False,
                 zsplit=None):
        import torch
        self.world, self.nz_global = nslabs, nz
        self.peer = peer
        self.device = torch.device("cuda", device)
        self.stream = torch.cuda.Stream(device=self.device)
        if zsplit is None:
            self.bounds = [slab_bounds(nz, nslabs, r) for r in range(nslabs)]
        else:
            if len(zsplit) != nslabs + 1 or zsplit[0] != 0 or zsplit[-1] != nz or any(b - a < 2 for a, b in zip(zsplit, zsplit[1:])):
                raise ValueError(f"zsplit {list(zsplit)}: need 0 = z_0 < z_1 < ... < z_{nslabs} = {nz}, >= 2 planes per slab")
            self.bounds = [(int(a), int(b - a)) for a, b in zip(zsplit, zsplit[1:])]
        self.lats = [Lattice(nx, ny, nz, params=params, device=device, slab=b) for b in self.bounds]
        for lat in self.lats:
            lat.set_stream(self.stream.cuda_stream)
            if brick_lz:
                lat.set_tiling(brick_lz)
        n = int(self.lats[0].lib.bflbm_halo_doubles(self.lats[0].h))
        lib = self.lats[0].lib
        self.send = [[_device_tensor(lib.bflbm_halo_send_buffer(l.h, s), n, self.device) for s in (0, 1)] for l in self.lats]
        self.recv = [[_device_tensor(lib.bflbm_halo_recv_buffer(l.h, s), n, self.device) for s in (0, 1)] for l in self.lats]
        if peer:  # peer mode on one device: the "neighbour's mailbox" is ordinary device memory of the same GPU
            for r, lat in enumerate(self.lats):
                lo, hi = neighbours(self.world, r)
                lat.peer_connect(0, self.lats[lo])
                lat.peer_connect(1, self.lats[hi])
        self.com = None          # reference-state noise: the slabs' centre-of-mass buffers
        self.initialized = False

    def set_reference_state(self, rho_eq=None, phi_eq=None, rhot_eq=None):
        """Lattice.set_reference_state on every slab (whole-box arrays); steps and inits then exchange the centre of mass."""
        self._all("set_reference_state", rho_eq, phi_eq, rhot_eq)
        if rho_eq is None:
            self.com = None
            return
        n = 4 * self.nz_global
        self.com = [_device_tensor(lat.com_buffer_pointer(), n, self.device) for lat in self.lats]
        if self.initialized:
            self._com_exchange()

    def _com_exchange(self):
        """the sum all-reduce of the centre-of-mass buffers: every entry has one owner and zeros elsewhere, so device copies of
        each slab's own planes into the others' buffers give the sum"""
        import torch
        if self.com is None:
            return
        with torch.cuda.stream(self.stream):
            for r in range(self.world):
                for s, (z0, nzl) in enumerate(self.bounds):
                    if s != r:
                        self.com[r][4 * z0:4 * (z0 + nzl)].copy_(self.com[s][4 * z0:4 * (z0 + nzl)])
        for lat in self.lats:
            lat.com_update()

    def close(self):
        for lat in self.lats:
            lat.close()

    def _exchange(self):
        import torch
        if self.peer:  # the pack kernels have already written into the neighbours' mailboxes
            return
        with torch.cuda.stream(self.stream):
            for r in range(self.world):
                lo, hi = neighbours(self.world, r)
                self.recv[lo][1].copy_(self.send[r][0])  # my message towards lower z arrives from above at the lower neighbour
                self.recv[hi][0].copy_(self.send[r][1])

    def _all(self, name, *a):
        for lat in self.lats:
            getattr(lat, name)(*a)

    def _init(self, name, *a):
        self._all(name, *a)
        self.initialized = True
        self._com_exchange()

    def init_mixture(self):
        self._init("init_mixture")

    def init_stripe(self, frac=0.5):
        self._init("init_stripe", frac)

    def init_droplet(self, radius=0.2):
        self._init("init_droplet", radius)

    def init_from_global_populations(self, f, g):
        for lat, (z0, nzl) in zip(self.lats, self.bounds):
            idx = [(z % self.nz_global) for z in range(z0 - 1, z0 + nzl + 1)]
            lat.init_from_populations_slab(np.ascontiguousarray(f[:, idx]), np.ascontiguousarray(g[:, idx]))
        for lat in self.lats:
            _check(lat.lib.bflbm_halo_refresh_begin(lat.h))
        self._exchange()
        for lat in self.lats:
            _check(lat.lib.bflbm_halo_refresh_end(lat.h))
        self.initialized = True
        self._com_exchange()

    def step(self, n=1):
        for _ in range(int(n)):
            for lat in self.lats:
                _check(lat.lib.bflbm_step_begin(lat.h))
            self._exchange()
            for lat in self.lats:
                _check(lat.lib.bflbm_step_end(lat.h))
            self._com_exchange()

    def gather(self, name):
        """Concatenates a getter's result over the slabs along z (tuple results element-wise)."""
        parts = [getattr(lat, name)() for lat in self.lats]
        if isinstance(parts[0], tuple):
            return tuple(np.concatenate([p[i] for p in parts], axis=1) for i in range(len(parts[0])))
        axis = 0 if name == "normals" else 1
        return np.concatenate(parts, axis=axis)


class SlabLattice:
    """One rank's slab of a periodic nx*ny*nz box.  Mirrors Lattice (init_*, step, getters on the local slab)."""

    def __init__(self, nx, ny, nz, params: Params | None = None, device: int = 0, group=None, peer: bool = False):
        import torch
        import torch.distributed as dist
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.group = group
        self.nz_global = nz
        self.z0, self.nzl = slab_bounds(nz, self.world, self.rank)
        self.lat = Lattice(nx, ny, nz, params=params, device=device, slab=(self.z0, self.nzl))
        self.device = torch.device("cuda", device)
        # one stream for the library's kernels AND torch's collectives, so that pack -> send/recv -> unpack are ordered
        self.stream = torch.cuda.Stream(device=self.device)
        self.lat.set_stream(self.stream.cuda_stream)
        n = int(self.lat.lib.bflbm_halo_doubles(self.lat.h))
        lib, h = self.lat.lib, self.lat.h
        self.send = [_device_tensor(lib.bflbm_halo_send_buffer(h, s), n, self.device) for s in (0, 1)]
        self.recv = [_device_tensor(lib.bflbm_halo_recv_buffer(h, s), n, self.device) for s in (0, 1)]
        self.halo_bytes_per_step = 2 * n * 8
        self.com = None          # reference-state noise: the centre-of-mass buffer, sum-all-reduced after every step and init
        self.initialized = False
        # peer mode: neighbours' mailboxes mapped through CUDA IPC; from then on a step needs no collective and no Python
        self.peer = False
        if peer:
            self.connect_peers()

    def connect_peers(self):
        if self.world == 1:
            self.lat.peer_connect(0, self.lat)
            self.lat.peer_connect(1, self.lat)
        else:
            lo, hi = gather_ring_handles(self.lat.peer_ipc_handle(), self.rank, self.world, self.group)
            self.lat.peer_connect_ipc(0, lo)
            self.lat.peer_connect_ipc(1, hi)
        self.peer = True

    # -- delegation --------------------------------------------------------------------------------
    def __getattr__(self, name):
        return getattr(self.lat, name)

    def _exchange(self):
        import torch
        if self.peer:
            return
        with torch.cuda.stream(self.stream):
            exchange_ring(self.send[0], self.send[1], self.recv[0], self.recv[1], self.rank, self.world, self.group)

    def set_reference_state(self, rho_eq=None, phi_eq=None, rhot_eq=None):
        """Lattice.set_reference_state (whole-box arrays on every rank); steps and inits then all-reduce the centre of mass.  In
        peer mode the halo still travels by peer stores; only the centre of mass uses the collective."""
        self.lat.set_reference_state(rho_eq, phi_eq, rhot_eq)
        if rho_eq is None:
            self.com = None
            return
        self.com = _device_tensor(self.lat.com_buffer_pointer(), 4 * self.nz_global, self.device)
        if self.initialized:
            self._com_exchange()

    def _com_exchange(self):
        """sum all-reduce of the per-plane centre-of-mass sums (one owner per entry: the same bits on every rank), then the shift"""
        import torch
        import torch.distributed as dist
        if self.com is None:
            return
        if self.world > 1:
            with torch.cuda.stream(self.stream):
                dist.all_reduce(self.com, op=dist.ReduceOp.SUM, group=self.group)
        self.lat.com_update()

    def _initialized(self):
        self.initialized = True
        self._com_exchange()

    def init_mixture(self):
        self.lat.init_mixture()
        self._initialized()

    def init_stripe(self, frac=0.5):
        self.lat.init_stripe(frac)
        self._initialized()

    def init_droplet(self, radius=0.2):
        self.lat.init_droplet(radius)
        self._initialized()

    def init_from_populations_slab(self, f_ghosted, g_ghosted):
        self.lat.init_from_populations_slab(f_ghosted, g_ghosted)
        _check(self.lat.lib.bflbm_halo_refresh_begin(self.lat.h))
        self._exchange()
        _check(self.lat.lib.bflbm_halo_refresh_end(self.lat.h))
        self._initialized()

    def init_from_staged(self):
        """The staged (ghosted) checkpoint of this slab + the halo refresh: init_from_populations_slab without the host."""
        self.lat.init_from_staged()
        _check(self.lat.lib.bflbm_halo_refresh_begin(self.lat.h))
        self._exchange()
        _check(self.lat.lib.bflbm_halo_refresh_end(self.lat.h))
        self._initialized()

    def init_from_global_populations(self, f, g):
        """Convenience for tests: every rank passes the WHOLE box (19, nz, ny, nx) and keeps its slab + ghost planes."""
        idx = [(z % self.nz_global) for z in range(self.z0 - 1, self.z0 + self.nzl + 1)]
        self.init_from_populations_slab(np.ascontiguousarray(f[:, idx]), np.ascontiguousarray(g[:, idx]))

    def step(self, n=1):
        lib, h = self.lat.lib, self.lat.h
        if self.peer and self.com is None:  # the whole loop runs inside the library: begin (pack = NVLink stores), end (wait, unpack)
            _check(lib.bflbm_step_slab(h, int(n)))
            return
        for _ in range(int(n)):
            _check(lib.bflbm_step_begin(h))
            self._exchange()
            _check(lib.bflbm_step_end(h))
            self._com_exchange()

    def host_checkpoint(self):
        """bench.py helper (untimed): this slab's populations as a ghosted host checkpoint, (2, 19, nz_local + 2, ny, nx), pinned
        if the host allows it.  The ghost planes come from the ring neighbours once, here -- like reading a checkpoint file
        that already has them."""
        import torch
        lat = self.lat
        f, g = lat.populations()
        try:
            fg = torch.empty((2, NVEL, self.nzl + 2, lat.ny, lat.nx), dtype=torch.float64, pin_memory=True).numpy()
        except Exception:
            fg = np.empty((2, NVEL, self.nzl + 2, lat.ny, lat.nx))
        fg[0, :, 1:-1], fg[1, :, 1:-1] = f, g
        lo_send = torch.from_numpy(np.ascontiguousarray(np.stack([f[:, 0], g[:, 0]]))).to(self.device)
        hi_send = torch.from_numpy(np.ascontiguousarray(np.stack([f[:, -1], g[:, -1]]))).to(self.device)
        del f, g
        lo_recv, hi_recv = torch.empty_like(lo_send), torch.empty_like(hi_send)
        exchange_ring(lo_send, hi_send, lo_recv, hi_recv, self.rank, self.world, self.group)
        fg[:, :, 0] = lo_recv.cpu().numpy()
        fg[:, :, -1] = hi_recv.cpu().numpy()
        torch.cuda.synchronize()
        return fg
