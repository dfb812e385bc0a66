"""Host mirror of FHDeX's StructFact as the reference driver uses it (main_run_job.cpp:299-310, 342-349, 50-54), over
include/bflbm_sf.h: the hydrodynamic fields are transformed and accumulated on the GPU, only the averaged spectra come back."""
from __future__ import annotations

import ctypes
import os

import numpy as np

from . import _build
from .lattice import BflbmError, Lattice

#: the reference's pair lists, main_run_job.cpp:301-306 (indices into hydrovs, VariableNames order)
REFERENCE_PAIRS = list(zip([0, 1, 0, 2, 3, 4, 6, 7, 8, 2, 9, 15, 16, 17, 15, 18, 19, 20, 21, 20, 20, 21],
                           [0, 1, 1, 2, 3, 4, 6, 7, 8, 6, 9, 15, 16, 17, 16, 18, 19, 20, 21, 21, 18, 18]))

_sf_lib = None


def _load():
    global _sf_lib
    if _sf_lib is None:
        if not os.path.exists(_build.SF_LIB):
            raise BflbmError(f"{_build.SF_LIB} not built: run bflbm_b200.build_sf() (there is no CPU fallback)")
        ctypes.CDLL(_build.LIB, mode=ctypes.RTLD_GLOBAL)
        lib = ctypes.CDLL(_build.SF_LIB)
        vp, ip, dpp = ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p
        lib.bflbm_sf_create.restype, lib.bflbm_sf_create.argtypes = ip, [vp, ip, dpp, dpp, dpp, ctypes.POINTER(vp)]
        lib.bflbm_sf_create_multi.restype, lib.bflbm_sf_create_multi.argtypes = ip, [vp, ip, dpp, dpp, dpp, ctypes.POINTER(vp)]
        lib.bflbm_sf_destroy.restype, lib.bflbm_sf_destroy.argtypes = ip, [vp]
        lib.bflbm_sf_accumulate.restype, lib.bflbm_sf_accumulate.argtypes = ip, [vp]
        lib.bflbm_sf_reset.restype, lib.bflbm_sf_reset.argtypes = ip, [vp]
        lib.bflbm_sf_samples.restype, lib.bflbm_sf_samples.argtypes = ctypes.c_longlong, [vp]
        lib.bflbm_sf_get.restype, lib.bflbm_sf_get.argtypes = ip, [vp, ip, dpp, dpp]
        sz = ctypes.POINTER(ctypes.c_size_t)
        ipp = ctypes.POINTER(ctypes.c_int)
        for name, res, args in (
                ("bflbm_sf_slab_create", ip, [vp, ip, ip, dpp, ip, dpp, dpp, dpp, ctypes.POINTER(vp)]),
                ("bflbm_sf_slab_destroy", ip, [vp]),
                ("bflbm_sf_slab_set_stream", ip, [vp, vp]),
                ("bflbm_sf_slab_rounds", ip, [vp]),
                ("bflbm_sf_slab_layout", ip, [vp, ip, sz, sz, sz, sz]),
                ("bflbm_sf_slab_send_buffer", vp, [vp]),
                ("bflbm_sf_slab_recv_buffer", vp, [vp]),
                ("bflbm_sf_slab_begin", ip, [vp, ip]),
                ("bflbm_sf_slab_end", ip, [vp, ip]),
                ("bflbm_sf_slab_reset", ip, [vp]),
                ("bflbm_sf_slab_samples", ctypes.c_longlong, [vp]),
                ("bflbm_sf_slab_kx_range", ip, [vp, ip, ipp, ipp]),
                ("bflbm_sf_slab_get", ip, [vp, ip, dpp, dpp])):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _sf_lib = lib
    return _sf_lib


class StructureFactor:
    """StructFact(ba, dm, var_names, var_scaling, pairA, pairB) for a whole-box Lattice or a MultiLattice (slabs on several GPUs)."""

    def __init__(self, lat: Lattice, pairs=REFERENCE_PAIRS, var_scaling=None):
        self.lib = _load()
        self.lat = lat
        self.pairs = [(int(a), int(b)) for a, b in pairs]
        a = np.ascontiguousarray([p[0] for p in self.pairs], dtype=np.int32)
        b = np.ascontiguousarray([p[1] for p in self.pairs], dtype=np.int32)
        sc = None if var_scaling is None else np.ascontiguousarray(var_scaling, dtype=np.float64)
        self.h = ctypes.c_void_p()
        create = self.lib.bflbm_sf_create_multi if hasattr(lat, "ngpus") else self.lib.bflbm_sf_create
        rc = create(lat.h, len(self.pairs), a.ctypes.data, b.ctypes.data, None if sc is None else sc.ctypes.data, ctypes.byref(self.h))
        if rc:
            raise BflbmError(f"bflbm_sf_create failed ({rc})")

    def close(self):
        if self.h:
            self.lib.bflbm_sf_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def fort_structure(self):
        """StructFact::FortStructure(hydrovs, 0): add the current state's A_k conj(B_k) of every pair."""
        rc = self.lib.bflbm_sf_accumulate(self.h)
        if rc:
            raise BflbmError(f"bflbm_sf_accumulate failed ({rc})")

    def reset(self):
        self.lib.bflbm_sf_reset(self.h)

    @property
    def samples(self) -> int:
        return int(self.lib.bflbm_sf_samples(self.h))

    def result(self, zero_avg: bool = True, imag: bool = False):
        """What StructFact::WritePlotFile writes: (npairs, nz, ny, nx) sample means on the shifted k grid."""
        shape = (len(self.pairs), self.lat.nz, self.lat.ny, self.lat.nx)
        re = np.empty(shape)
        im = np.empty(shape) if imag else None
        rc = self.lib.bflbm_sf_get(self.h, 1 if zero_avg else 0, re.ctypes.data, None if im is None else im.ctypes.data)
        if rc:
            raise BflbmError(f"bflbm_sf_get failed ({rc})")
        return (re, im) if imag else re


def _slab_check(rc: int, what: str):
    if rc:
        err = BflbmError(f"{what} failed ({rc})")
        err.code = rc
        raise err


class SlabStructureFactor:
    """StructFact for a box split along z (include/bflbm_sf_slab.h): every rank keeps its slab of the fields and its kx columns of
    k-space; one all-to-all per distinct variable moves the 2-D spectra between the ranks.

    `slab` is a distributed.SlabLattice (one rank per process; the blocks go through torch.distributed.all_to_all_single on the
    slab's stream, which its halo collectives use too) or a distributed.EmulatedSlabs (every slab of the box in this process on
    one GPU; the blocks move by device copies)."""

    def __init__(self, slab, pairs=REFERENCE_PAIRS, var_scaling=None):
        from .distributed import EmulatedSlabs, _device_tensor
        self.lib = _load()
        self.slab = slab
        self.pairs = [(int(a), int(b)) for a, b in pairs]
        self.emulated = isinstance(slab, EmulatedSlabs)
        if self.emulated:
            lats, ranks, bounds = slab.lats, list(range(slab.world)), slab.bounds
        else:
            from .distributed import slab_bounds
            lats, ranks = [slab.lat], [slab.rank]
            bounds = [slab_bounds(slab.nz_global, slab.world, r) for r in range(slab.world)]
        self.world = len(bounds)
        self.rank = 0 if self.emulated else slab.rank
        self.nx, self.ny, self.nz = lats[0].nx, lats[0].ny, slab.nz_global
        zsplit = np.ascontiguousarray([z0 for z0, _ in bounds] + [slab.nz_global], dtype=np.int32)
        a = np.ascontiguousarray([p[0] for p in self.pairs], dtype=np.int32)
        b = np.ascontiguousarray([p[1] for p in self.pairs], dtype=np.int32)
        sc = None if var_scaling is None else np.ascontiguousarray(var_scaling, dtype=np.float64)
        self.h = []
        for lat, r in zip(lats, ranks):
            h = ctypes.c_void_p()
            _slab_check(self.lib.bflbm_sf_slab_create(lat.h, self.world, r, zsplit.ctypes.data, len(self.pairs), a.ctypes.data,
                                                      b.ctypes.data, None if sc is None else sc.ctypes.data, ctypes.byref(h)),
                        "bflbm_sf_slab_create")
            self.h.append(h)
            _slab_check(self.lib.bflbm_sf_slab_set_stream(h, ctypes.c_void_p(slab.stream.cuda_stream)), "bflbm_sf_slab_set_stream")
        self.rounds = int(self.lib.bflbm_sf_slab_rounds(self.h[0]))
        # every round has the same layout (one variable); counts and displacements in doubles, per rank
        self.layout, self.send, self.recv = [], [], []
        for h in self.h:
            arrs = [(ctypes.c_size_t * self.world)() for _ in range(4)]
            _slab_check(self.lib.bflbm_sf_slab_layout(h, 0, *arrs), "bflbm_sf_slab_layout")
            sc_, sd, rc_, rd = ([int(v) for v in x] for x in arrs)
            self.layout.append((sc_, sd, rc_, rd))
            self.send.append(_device_tensor(self.lib.bflbm_sf_slab_send_buffer(h), sum(sc_), slab.device))
            self.recv.append(_device_tensor(self.lib.bflbm_sf_slab_recv_buffer(h), sum(rc_), slab.device))

    def close(self):
        for h in self.h:
            self.lib.bflbm_sf_slab_destroy(h)
        self.h = []

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def kx_range(self, rank: int) -> tuple[int, int]:
        """(kx0, nkx): the half-spectrum columns `rank` owns."""
        kx0, nkx = ctypes.c_int(), ctypes.c_int()
        _slab_check(self.lib.bflbm_sf_slab_kx_range(self.h[0], int(rank), ctypes.byref(kx0), ctypes.byref(nkx)), "bflbm_sf_slab_kx_range")
        return kx0.value, nkx.value

    def _collective(self) -> bool:
        """A SlabLattice of an initialised process group (of any size) exchanges through torch.distributed."""
        import torch.distributed as dist
        return not self.emulated and dist.is_initialized()

    def _exchange(self):
        import torch
        with torch.cuda.stream(self.slab.stream):
            if self.emulated:
                for s, (scnt, sdis, _, _) in enumerate(self.layout):
                    for d, (_, _, rcnt, rdis) in enumerate(self.layout):
                        self.recv[d][rdis[s]:rdis[s] + rcnt[s]].copy_(self.send[s][sdis[d]:sdis[d] + scnt[d]])
            elif not self._collective():
                self.recv[0].copy_(self.send[0])
            else:
                import torch.distributed as dist
                scnt, _, rcnt, _ = self.layout[0]
                dist.all_to_all_single(self.recv[0], self.send[0], output_split_sizes=rcnt, input_split_sizes=scnt,
                                       group=self.slab.group)

    def fort_structure(self):
        """StructFact::FortStructure(hydrovs, 0) on the decomposed box: one begin / exchange / end per distinct variable."""
        for v in range(self.rounds):
            for h in self.h:
                _slab_check(self.lib.bflbm_sf_slab_begin(h, v), "bflbm_sf_slab_begin")
            self._exchange()
            for h in self.h:
                _slab_check(self.lib.bflbm_sf_slab_end(h, v), "bflbm_sf_slab_end")

    def reset(self):
        for h in self.h:
            _slab_check(self.lib.bflbm_sf_slab_reset(h), "bflbm_sf_slab_reset")

    @property
    def samples(self) -> int:
        return int(self.lib.bflbm_sf_slab_samples(self.h[0]))

    def result(self, zero_avg: bool = True, imag: bool = False, root: int = 0):
        """What StructFact::WritePlotFile writes, (npairs, nz, ny, nx) sample means on the shifted k grid, on rank `root` of the
        slab's group (None on the other ranks).  Every rank fills the x columns it owns; the parts meet on the root through a sum
        reduction in which every value has exactly one non-zero contributor."""
        shape = (len(self.pairs), self.nz, self.ny, self.nx)
        re = np.zeros(shape)
        im = np.zeros(shape) if imag else None
        for h in self.h:
            _slab_check(self.lib.bflbm_sf_slab_get(h, 1 if zero_avg else 0, re.ctypes.data, None if im is None else im.ctypes.data),
                        "bflbm_sf_slab_get")
        if self._collective():
            import torch
            import torch.distributed as dist
            group = self.slab.group
            dst = root if group is None else dist.get_global_rank(group, root)
            with torch.cuda.stream(self.slab.stream):
                for arr in (re, im):
                    if arr is None:
                        continue
                    for p in range(shape[0]):  # one pair at a time bounds the device memory of the reduction
                        t = torch.from_numpy(arr[p]).to(self.slab.device)
                        dist.reduce(t, dst=dst, op=dist.ReduceOp.SUM, group=group)
                        if self.rank == root:
                            arr[p] = t.cpu().numpy()
            if self.rank != root:
                return None
        return (re, im) if imag else re
