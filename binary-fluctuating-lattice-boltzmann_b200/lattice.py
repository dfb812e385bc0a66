"""Host-side mirror of the reference's solver interface over the C ABI (include/bflbm.h).

The reference's boundary is a set of free functions on caller-owned MultiFabs
(LBM_binary.H:545-551, 598-605, 632-641, 664-668, 699-707) plus global parameters
(LBM_d3q19.H:10, LBM_binary.H:17-30).  `Lattice` bundles what those MultiFabs hold; the module-level
functions at the bottom keep the reference's names and argument meaning.

Every array is float64 with C shape (ncomp, nz_local, ny, nx) = AMReX FAB order.
There is no CPU path: constructing a Lattice without the CUDA library or a GPU raises.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass, asdict

import numpy as np

from . import _build

NVEL, NHYDRO, NHYDRO_BAR, NNORMALS = 19, 22, 9, 33

#: hydrovs component names, AMReX_FileIO.H:208-261
VARIABLE_NAMES = ["rho", "phi", "ufx", "ufy", "ufz", "p_bulk", "ugx", "ugy", "ugz", "afx", "afy", "afz",
                  "agx", "agy", "agz", "ubx", "uby", "ubz", "nfbarx", "ngbarx", "ufbarx", "ugbarx"]

#: fields of bflbm_debug_last_step, in its order (include/bflbm.h): algorithm 0 fused / 1 two-pass; fold_source 1 = staged from
#: the extended boxes, 0 = every plane from R; schedule 0 whole box / 1 slab on one stream / 2 slab overlapped
LAST_STEP_FIELDS = ("algorithm", "threads", "tile_x", "tile_y", "lz", "bx", "by", "bz", "full", "rate1", "noise",
                    "fold_source", "schedule", "graph")


class BflbmError(RuntimeError):
    pass


class _CParams(ctypes.Structure):
    _fields_ = [("kBT", ctypes.c_double), ("tau_f", ctypes.c_double), ("tau_g", ctypes.c_double),
                ("alpha0", ctypes.c_double), ("alpha1", ctypes.c_double), ("kappa", ctypes.c_double),
                ("rho_lo", ctypes.c_double), ("rho_hi", ctypes.c_double),
                ("seed", ctypes.c_ulonglong), ("step0", ctypes.c_longlong)]


@dataclass
class Params:
    """The reference's editable globals (defaults = shipped values)."""
    kBT: float = 0.0       # LBM_d3q19.H:10
    tau_f: float = 0.5     # LBM_binary.H:18
    tau_g: float = 0.5     # LBM_binary.H:19
    alpha0: float = 4.0    # LBM_binary.H:20
    alpha1: float = 0.0    # LBM_binary.H:21 (no effect in the reference; must stay 0)
    kappa: float = 4.0     # LBM_binary.H:30
    rho_lo: float = 0.0    # LBM_binary.H:25
    rho_hi: float = 1.0    # LBM_binary.H:26
    seed: int = 12345      # LBM_binary.H:17 / main_run_job.cpp:68
    step0: int = 0         # main_run_job.cpp:80 step_continue

    def _c(self) -> _CParams:
        return _CParams(**asdict(self))


_lib = None


def load_library() -> ctypes.CDLL:
    """Load libbflbm.so (built in-tree by `_build.build()`); raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("BFLBM_LIB") or _build.LIB  # BFLBM_LIB: A/B runs of two builds of the same library
    if not os.path.exists(path):
        raise BflbmError(f"CUDA library {path} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(there is no CPU fallback)")
    lib = ctypes.CDLL(path)
    vp, ip, dp = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    P = ctypes.POINTER(_CParams)
    sig = {
        "bflbm_params_default": (ip, [P]),
        "bflbm_create": (ip, [P, ip, ip, ip, ip, ctypes.POINTER(vp)]),
        "bflbm_create_slab": (ip, [P, ip, ip, ip, ip, ip, ip, ctypes.POINTER(vp)]),
        "bflbm_destroy": (ip, [vp]),
        "bflbm_set_params": (ip, [vp, P]),
        "bflbm_get_params": (ip, [vp, P]),
        "bflbm_set_stream": (ip, [vp, vp]),
        "bflbm_set_algorithm": (ip, [vp, ip]),
        "bflbm_set_tiling": (ip, [vp, ip]),
        "bflbm_init_mixture": (ip, [vp]),
        "bflbm_init_stripe": (ip, [vp, dp]),
        "bflbm_init_droplet": (ip, [vp, dp]),
        "bflbm_init_from_populations": (ip, [vp, vp, vp]),
        "bflbm_init_from_populations_slab": (ip, [vp, vp, vp]),
        "bflbm_stage_populations": (ip, [vp, vp, vp, ip]),
        "bflbm_stage_wait": (ip, [vp]),
        "bflbm_init_from_staged": (ip, [vp]),
        "bflbm_get_hydrovars_async": (ip, [vp, vp]),
        "bflbm_get_hydrovars_bar_async": (ip, [vp, vp]),
        "bflbm_download_wait": (ip, [vp]),
        "bflbm_release_staging": (ip, [vp]),
        "bflbm_step": (ip, [vp, ip]),
        "bflbm_sync": (ip, [vp]),
        "bflbm_step_count": (ctypes.c_longlong, [vp]),
        "bflbm_get_populations": (ip, [vp, vp, vp]),
        "bflbm_get_hydrovars": (ip, [vp, vp]),
        "bflbm_get_hydrovars_bar": (ip, [vp, vp]),
        "bflbm_get_noise": (ip, [vp, vp, vp]),
        "bflbm_get_normals": (ip, [vp, vp]),
        "bflbm_get_hydrovars_device": (ip, [vp, vp]),
        "bflbm_get_hydrovars_bar_device": (ip, [vp, vp]),
        "bflbm_get_hydrovars_device_into_global": (ip, [vp, vp]),
        "bflbm_get_device": (ip, [vp]),
        "bflbm_get_populations_device": (ip, [vp, vp, vp]),
        "bflbm_center_of_mass": (ip, [vp, vp, vp]),
        "bflbm_total_mass": (ip, [vp, vp, vp]),
        "bflbm_check_nan": (ip, [vp, ctypes.POINTER(ctypes.c_longlong)]),
        "bflbm_halo_doubles": (ctypes.c_size_t, [vp]),
        "bflbm_halo_send_buffer": (vp, [vp, ip]),
        "bflbm_halo_recv_buffer": (vp, [vp, ip]),
        "bflbm_step_begin": (ip, [vp]),
        "bflbm_step_end": (ip, [vp]),
        "bflbm_halo_refresh_begin": (ip, [vp]),
        "bflbm_halo_refresh_end": (ip, [vp]),
        "bflbm_set_profiling": (ip, [vp, ip]),
        "bflbm_get_profile": (ip, [vp, vp, ctypes.POINTER(ctypes.c_longlong)]),
        "bflbm_kernel_launches": (ctypes.c_longlong, [vp]),
        "bflbm_device_bytes": (ctypes.c_size_t, [vp]),
        "bflbm_get_dims": (ip, [vp] + [ctypes.POINTER(ip)] * 5),
        "bflbm_second_moments": (ip, [vp, vp]),
        "bflbm_droplet_covariance": (ip, [vp, vp, vp, vp]),
        "bflbm_debug_philox": (ip, [vp, vp, vp]),
        "bflbm_debug_last_step": (ip, [vp, vp]),
        "bflbm_debug_normal_statistics": (ip, [ctypes.c_ulonglong, ctypes.c_longlong, ctypes.c_longlong, ip, ip, dp, dp, vp, vp, vp]),
        "bflbm_covariance_from_moments": (ip, [vp, vp, vp, vp]),
        "bflbm_set_reference_state": (ip, [vp, vp, vp, vp]),
        "bflbm_fit_droplet": (ip, [vp, ip, dp, ip, dp, dp, dp, dp, dp, vp, ctypes.POINTER(ip)]),
        "bflbm_droplet_fit_terms": (ip, [vp, dp, dp, vp, vp]),
        "bflbm_debug_fit_coefficients": (ip, [dp, dp, dp, dp, dp, dp, vp]),
        "bflbm_multi_fit_droplet": (ip, [vp, ip, dp, ip, dp, dp, dp, dp, dp, vp, ctypes.POINTER(ip)]),
        "bflbm_get_reference_com": (ip, [vp, vp]),
        "bflbm_get_reference_shift": (ip, [vp, vp]),
        "bflbm_com_doubles": (ctypes.c_size_t, [vp]),
        "bflbm_com_buffer": (vp, [vp]),
        "bflbm_com_update": (ip, [vp]),
        "bflbm_multi_set_reference_state": (ip, [vp, vp, vp, vp]),
        "bflbm_init_from_global_populations": (ip, [vp, vp, vp]),
        "bflbm_get_populations_into_global": (ip, [vp, vp, vp]),
        "bflbm_get_hydrovars_into_global": (ip, [vp, vp]),
        "bflbm_get_hydrovars_bar_into_global": (ip, [vp, vp]),
        "bflbm_get_noise_into_global": (ip, [vp, vp, vp]),
        "bflbm_peer_mailbox_bytes": (ctypes.c_size_t, [vp]),
        "bflbm_peer_mailbox": (vp, [vp]),
        "bflbm_peer_ipc_handle": (ip, [vp, vp]),
        "bflbm_peer_connect": (ip, [vp, ip, vp, ip]),
        "bflbm_peer_connect_ipc": (ip, [vp, ip, vp]),
        "bflbm_peer_connected": (ip, [vp]),
        "bflbm_step_slab": (ip, [vp, ip]),
        "bflbm_halo_refresh": (ip, [vp]),
        "bflbm_halo_error": (ip, [vp, ctypes.POINTER(ip)]),
        "bflbm_multi_create": (ip, [P, ip, ip, ip, ip, ctypes.POINTER(ip), ip, ctypes.POINTER(vp)]),
        "bflbm_multi_destroy": (ip, [vp]),
        "bflbm_multi_count": (ip, [vp]),
        "bflbm_multi_slab": (vp, [vp, ip]),
        "bflbm_multi_set_params": (ip, [vp, P]),
        "bflbm_multi_init_mixture": (ip, [vp]),
        "bflbm_multi_init_stripe": (ip, [vp, dp]),
        "bflbm_multi_init_droplet": (ip, [vp, dp]),
        "bflbm_multi_init_from_populations": (ip, [vp, vp, vp]),
        "bflbm_multi_step": (ip, [vp, ip]),
        "bflbm_multi_sync": (ip, [vp]),
        "bflbm_multi_step_count": (ctypes.c_longlong, [vp]),
        "bflbm_multi_get_populations": (ip, [vp, vp, vp]),
        "bflbm_multi_get_hydrovars": (ip, [vp, vp]),
        "bflbm_multi_get_hydrovars_bar": (ip, [vp, vp]),
        "bflbm_multi_get_noise": (ip, [vp, vp, vp]),
        "bflbm_multi_total_mass": (ip, [vp, vp, vp]),
        "bflbm_multi_second_moments": (ip, [vp, vp]),
        "bflbm_multi_center_of_mass": (ip, [vp, vp]),
        "bflbm_multi_droplet_covariance": (ip, [vp, vp, vp, vp]),
        "bflbm_multi_check_nan": (ip, [vp, ctypes.POINTER(ctypes.c_longlong)]),
        "bflbm_multi_kernel_launches": (ctypes.c_longlong, [vp]),
        "bflbm_multi_device_bytes": (ctypes.c_size_t, [vp]),
        "bflbm_multi_last_error": (ctypes.c_char_p, []),
        "bflbm_last_error": (ctypes.c_char_p, []),
        "bflbm_version": (ctypes.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _check(rc: int):
    if rc != 0:
        raise BflbmError(f"bflbm error {rc}: {load_library().bflbm_last_error().decode()}")


def _host(a, shape, name):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.shape != tuple(shape):
        raise ValueError(f"{name}: expected shape {tuple(shape)}, got {a.shape}")
    return a


class Lattice:
    """Device-resident state of one box (or one z-slab of it): what fold, gold, hydrovs, hydrovsbar,
    fnoisevs, gnoisevs hold in the reference (main_run_job.cpp:205-212)."""

    def __init__(self, nx, ny=None, nz=None, params: Params | None = None, device: int = 0,
                 slab: tuple[int, int] | None = None):
        ny = nx if ny is None else ny
        nz = nx if nz is None else nz
        self.lib = load_library()
        self.params = params or Params()
        self.nx, self.ny, self.nz_global = int(nx), int(ny), int(nz)
        self.z0, self.nz = (0, self.nz_global) if slab is None else (int(slab[0]), int(slab[1]))
        self.shape = (self.nz, self.ny, self.nx)
        self.device = device
        h = ctypes.c_void_p()
        cp = self.params._c()
        if slab is None:
            _check(self.lib.bflbm_create(ctypes.byref(cp), self.nx, self.ny, self.nz_global, device, ctypes.byref(h)))
        else:
            _check(self.lib.bflbm_create_slab(ctypes.byref(cp), self.nx, self.ny, self.nz_global, self.z0, self.nz,
                                              device, ctypes.byref(h)))
        self.h = h
        self._staged_refs = None   # host arrays of transfers in flight are kept alive here
        self._download_ref = None

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.lib.bflbm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- parameters -------------------------------------------------------------------------------
    def set_params(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.params, k):
                raise AttributeError(k)
            setattr(self.params, k, v)
        cp = self.params._c()
        _check(self.lib.bflbm_set_params(self.h, ctypes.byref(cp)))

    def set_stream(self, cuda_stream: int | None):
        _check(self.lib.bflbm_set_stream(self.h, ctypes.c_void_p(cuda_stream or 0)))

    def set_algorithm(self, name: str):
        _check(self.lib.bflbm_set_algorithm(self.h, {"fused": 0, "twopass": 1}[name]))

    def set_tiling(self, lz: int):
        _check(self.lib.bflbm_set_tiling(self.h, int(lz)))

    # -- initial conditions -------------------------------------------------------------------------
    def init_mixture(self):
        _check(self.lib.bflbm_init_mixture(self.h))

    def init_stripe(self, frac=0.5):
        _check(self.lib.bflbm_init_stripe(self.h, float(frac)))

    def init_droplet(self, radius=0.2):
        _check(self.lib.bflbm_init_droplet(self.h, float(radius)))

    def init_from_populations(self, f, g):
        f = _host(f, (NVEL,) + self.shape, "f")
        g = _host(g, (NVEL,) + self.shape, "g")
        _check(self.lib.bflbm_init_from_populations(self.h, f.ctypes.data, g.ctypes.data))

    def init_from_populations_slab(self, f_ghosted, g_ghosted):
        shp = (NVEL, self.nz + 2, self.ny, self.nx)
        f = _host(f_ghosted, shp, "f_ghosted")
        g = _host(g_ghosted, shp, "g_ghosted")
        _check(self.lib.bflbm_init_from_populations_slab(self.h, f.ctypes.data, g.ctypes.data))

    # -- asynchronous host transfers (include/bflbm.h "asynchronous host transfers") -----------------------------------
    def stage_populations(self, f, g, ghosted=False):
        """Start the host -> device copy of a checkpoint next to whatever the lattice is doing.  The arrays are used in place
        (no conversion copy): they must be C-contiguous float64 of the right shape and stay alive and untouched until
        stage_wait() (pinned memory, e.g. torch.empty(..., pin_memory=True).numpy(), makes the copy asynchronous)."""
        shp = (NVEL, self.nz + (2 if ghosted else 0), self.ny, self.nx)
        for a, name in ((f, "f"), (g, "g")):
            if not (isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.c_contiguous and a.shape == shp):
                raise ValueError(f"{name}: need a C-contiguous float64 array of shape {shp}")
        _check(self.lib.bflbm_stage_populations(self.h, f.ctypes.data, g.ctypes.data, 1 if ghosted else 0))
        self._staged_refs = (f, g)

    def stage_wait(self):
        _check(self.lib.bflbm_stage_wait(self.h))
        self._staged_refs = None

    def init_from_staged(self):
        """init_from_populations[_slab] of the staged checkpoint, queued behind the copy on the lattice's stream."""
        _check(self.lib.bflbm_init_from_staged(self.h))

    def hydrovars_bar_async(self, out=None):
        """Observer now, device -> host copy next to the following steps; `out` is complete after download_wait()."""
        if out is None:
            out = np.empty((NHYDRO_BAR,) + self.shape)
        if not (out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (NHYDRO_BAR,) + self.shape):
            raise ValueError("out: need a C-contiguous float64 array of shape %r" % (((NHYDRO_BAR,) + self.shape),))
        _check(self.lib.bflbm_get_hydrovars_bar_async(self.h, out.ctypes.data))
        self._download_ref = out
        return out

    def hydrovars_async(self, out=None):
        if out is None:
            out = np.empty((NHYDRO,) + self.shape)
        if not (out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (NHYDRO,) + self.shape):
            raise ValueError("out: need a C-contiguous float64 array of shape %r" % (((NHYDRO,) + self.shape),))
        _check(self.lib.bflbm_get_hydrovars_async(self.h, out.ctypes.data))
        self._download_ref = out
        return out

    def download_wait(self):
        _check(self.lib.bflbm_download_wait(self.h))
        self._download_ref = None

    def release_staging(self):
        _check(self.lib.bflbm_release_staging(self.h))

    def init_from_global_populations(self, f_global, g_global):
        """Host arrays of the WHOLE box (19, nz_global, ny, nx); a slab takes its planes and the periodic neighbour planes."""
        shp = (NVEL, self.nz_global, self.ny, self.nx)
        f = _host(f_global, shp, "f_global")
        g = _host(g_global, shp, "g_global")
        _check(self.lib.bflbm_init_from_global_populations(self.h, f.ctypes.data, g.ctypes.data))

    def set_reference_state(self, rho_eq=None, phi_eq=None, rhot_eq=None):
        """USE_REF_STATE noise (LBM_binary.H:12, 92-107): amplitudes from these equilibrium profiles of the WHOLE box,
        (nz_global, ny, nx) also for a slab, at the COM-shifted cell; None switches back to the shipped behaviour.  A slab then
        needs the centre-of-mass exchange after every step and init (com_buffer, com_update; distributed.py does it)."""
        if rho_eq is None:
            _check(self.lib.bflbm_set_reference_state(self.h, None, None, None))
            return
        shp = (self.nz_global, self.ny, self.nx)
        a = [_host(v, shp, n) for v, n in ((rho_eq, "rho_eq"), (phi_eq, "phi_eq"), (rhot_eq, "rhot_eq"))]
        _check(self.lib.bflbm_set_reference_state(self.h, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data))

    def reference_com(self):
        c = np.empty(3)
        _check(self.lib.bflbm_get_reference_com(self.h, c.ctypes.data))
        return c

    def reference_shift(self):
        """the integer shift (x, y, z) the next step reads the equilibrium profiles with (synchronises the lattice's stream)"""
        s = (ctypes.c_int * 3)()
        _check(self.lib.bflbm_get_reference_shift(self.h, s))
        return np.array(s, dtype=np.int64)

    def com_buffer_pointer(self) -> int:
        """device address of the 4 * nz_global doubles of per-plane centre-of-mass sums (slabs: the caller sum-all-reduces them)"""
        return int(self.lib.bflbm_com_buffer(self.h) or 0)

    def com_update(self):
        _check(self.lib.bflbm_com_update(self.h))

    # -- peer mode (include/bflbm.h): the halo message goes straight into the neighbour's mailbox ----------------
    def peer_ipc_handle(self) -> bytes:
        buf = ctypes.create_string_buffer(64)
        _check(self.lib.bflbm_peer_ipc_handle(self.h, buf))
        return buf.raw

    def peer_connect_ipc(self, side: int, handle: bytes):
        _check(self.lib.bflbm_peer_connect_ipc(self.h, int(side), ctypes.c_char_p(handle)))

    def peer_connect(self, side: int, other: "Lattice"):
        _check(self.lib.bflbm_peer_connect(self.h, int(side), ctypes.c_void_p(self.lib.bflbm_peer_mailbox(other.h)), int(other.device)))

    @property
    def peer_connected(self) -> bool:
        return bool(self.lib.bflbm_peer_connected(self.h))

    def step_slab(self, n=1):
        _check(self.lib.bflbm_step_slab(self.h, int(n)))

    def halo_refresh(self):
        _check(self.lib.bflbm_halo_refresh(self.h))

    def halo_error(self) -> int:
        e = ctypes.c_int()
        _check(self.lib.bflbm_halo_error(self.h, ctypes.byref(e)))
        return e.value

    # -- time stepping --------------------------------------------------------------------------------
    def step(self, n=1):
        _check(self.lib.bflbm_step(self.h, int(n)))

    def sync(self):
        _check(self.lib.bflbm_sync(self.h))

    @property
    def step_count(self) -> int:
        return int(self.lib.bflbm_step_count(self.h))

    # -- outputs --------------------------------------------------------------------------------------
    def populations(self):
        f = np.empty((NVEL,) + self.shape)
        g = np.empty((NVEL,) + self.shape)
        _check(self.lib.bflbm_get_populations(self.h, f.ctypes.data, g.ctypes.data))
        return f, g

    def hydrovars(self):
        out = np.empty((NHYDRO,) + self.shape)
        _check(self.lib.bflbm_get_hydrovars(self.h, out.ctypes.data))
        return out

    def hydrovars_bar(self):
        out = np.empty((NHYDRO_BAR,) + self.shape)
        _check(self.lib.bflbm_get_hydrovars_bar(self.h, out.ctypes.data))
        return out

    def noise(self):
        fn = np.empty((NVEL,) + self.shape)
        gn = np.empty((NVEL,) + self.shape)
        _check(self.lib.bflbm_get_noise(self.h, fn.ctypes.data, gn.ctypes.data))
        return fn, gn

    def normals(self):
        out = np.empty(self.shape + (NNORMALS,))
        _check(self.lib.bflbm_get_normals(self.h, out.ctypes.data))
        return out

    def center_of_mass(self):
        com = (ctypes.c_double * 3)()
        sums = (ctypes.c_double * 4)()
        _check(self.lib.bflbm_center_of_mass(self.h, com, sums))
        return np.array(com), np.array(sums)

    def droplet_covariance(self):
        """(com[3], cov[3, 3], eigenvalues[3] ascending) of rho: fittingDropletCovariance, LBM_hydrovs.H:258-335."""
        com, c6, e = np.empty(3), np.empty(6), np.empty(3)
        _check(self.lib.bflbm_droplet_covariance(self.h, com.ctypes.data, c6.ctypes.data, e.ctypes.data))
        cov = np.array([[c6[0], c6[3], c6[4]], [c6[3], c6[1], c6[5]], [c6[4], c6[5], c6[2]]])
        return com, cov, e

    def total_mass(self):
        a, b = ctypes.c_double(), ctypes.c_double()
        _check(self.lib.bflbm_total_mass(self.h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def fit_droplet(self, W0, R0, step_window=20, undul_ratio=0.01, nstep=400, eta_W=0.2, eta_R=0.2, dt=0.02):
        """fittingDropletParams (LBM_hydrovs.H:160-213, defaults of the call at main_run_job.cpp:365): (W, R, undulation, converged)."""
        out = np.empty(3)
        ok = ctypes.c_int()
        _check(self.lib.bflbm_fit_droplet(self.h, int(step_window), float(undul_ratio), int(nstep), float(W0), float(R0), float(eta_W),
                                          float(eta_R), float(dt), out.ctypes.data, ctypes.byref(ok)))
        return float(out[0]), float(out[1]), float(out[2]), bool(ok.value)

    def check_nan(self) -> int:
        """Number of non-finite hydro values; raises BflbmError if any (the reference prints and exit(0)s,
        Debug.H:137-149)."""
        n = ctypes.c_longlong()
        rc = self.lib.bflbm_check_nan(self.h, ctypes.byref(n))
        _check(rc)
        return n.value

    def set_profiling(self, on):
        """False/0 off, True/1 events read back after every step, 2 deferred read-back (no host synchronisation per step)"""
        _check(self.lib.bflbm_set_profiling(self.h, int(on)))

    def profile(self):
        """(ms per step of {step kernel, density fold, halo pack, halo unpack}, steps accumulated)"""
        ms = (ctypes.c_double * 4)()
        n = ctypes.c_longlong()
        _check(self.lib.bflbm_get_profile(self.h, ms, ctypes.byref(n)))
        k = max(1, n.value)
        return [v / k for v in ms], n.value

    # -- bookkeeping ----------------------------------------------------------------------------------
    @property
    def kernel_launches(self) -> int:
        return int(self.lib.bflbm_kernel_launches(self.h))

    @property
    def device_bytes(self) -> int:
        return int(self.lib.bflbm_device_bytes(self.h))

    def last_step(self) -> dict:
        """Which compiled variant of the step kernel the last step launched (bflbm_debug_last_step): a dict of LAST_STEP_FIELDS."""
        out = (ctypes.c_int * len(LAST_STEP_FIELDS))()
        _check(self.lib.bflbm_debug_last_step(self.h, out))
        return dict(zip(LAST_STEP_FIELDS, (int(v) for v in out)))


class MultiLattice:
    """One periodic box on several GPUs of this process (include/bflbm.h, bflbm_multi_*): z-slabs ring-connected in peer mode,
    host arrays of the WHOLE box (ncomp, nz, ny, nx).  Mirrors Lattice."""

    def __init__(self, nx, ny=None, nz=None, params: Params | None = None, ngpus: int = 1, devices=None, brick_lz: int = 0):
        ny = nx if ny is None else ny
        nz = nx if nz is None else nz
        self.lib = load_library()
        self.params = params or Params()
        self.nx, self.ny, self.nz = int(nx), int(ny), int(nz)
        self.shape = (self.nz, self.ny, self.nx)
        self.ngpus = int(ngpus)
        h = ctypes.c_void_p()
        cp = self.params._c()
        dev = (ctypes.c_int * self.ngpus)(*devices) if devices is not None else None
        self._mcheck(self.lib.bflbm_multi_create(ctypes.byref(cp), self.nx, self.ny, self.nz, self.ngpus, dev, int(brick_lz), ctypes.byref(h)))
        self.h = h

    def _mcheck(self, rc):
        if rc != 0:
            raise BflbmError(f"bflbm error {rc}: {self.lib.bflbm_multi_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.bflbm_multi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_params(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.params, k):
                raise AttributeError(k)
            setattr(self.params, k, v)
        cp = self.params._c()
        self._mcheck(self.lib.bflbm_multi_set_params(self.h, ctypes.byref(cp)))

    def init_mixture(self):
        self._mcheck(self.lib.bflbm_multi_init_mixture(self.h))

    def init_stripe(self, frac=0.5):
        self._mcheck(self.lib.bflbm_multi_init_stripe(self.h, float(frac)))

    def init_droplet(self, radius=0.2):
        self._mcheck(self.lib.bflbm_multi_init_droplet(self.h, float(radius)))

    def init_from_populations(self, f, g):
        f = _host(f, (NVEL,) + self.shape, "f")
        g = _host(g, (NVEL,) + self.shape, "g")
        self._mcheck(self.lib.bflbm_multi_init_from_populations(self.h, f.ctypes.data, g.ctypes.data))

    def set_reference_state(self, rho_eq=None, phi_eq=None, rhot_eq=None):
        """Lattice.set_reference_state on every slab (whole-box arrays); steps and inits then exchange the centre of mass"""
        if rho_eq is None:
            self._mcheck(self.lib.bflbm_multi_set_reference_state(self.h, None, None, None))
            return
        a = [_host(v, self.shape, n) for v, n in ((rho_eq, "rho_eq"), (phi_eq, "phi_eq"), (rhot_eq, "rhot_eq"))]
        self._mcheck(self.lib.bflbm_multi_set_reference_state(self.h, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data))

    def reference_shift(self, slab: int = 0):
        """the reference-state shift held by slab `slab` (every slab holds the same one)"""
        s = (ctypes.c_int * 3)()
        _check(self.lib.bflbm_get_reference_shift(self.lib.bflbm_multi_slab(self.h, int(slab)), s))
        return np.array(s, dtype=np.int64)

    def step(self, n=1):
        self._mcheck(self.lib.bflbm_multi_step(self.h, int(n)))

    def sync(self):
        self._mcheck(self.lib.bflbm_multi_sync(self.h))

    @property
    def step_count(self) -> int:
        return int(self.lib.bflbm_multi_step_count(self.h))

    def populations(self):
        f, g = np.empty((NVEL,) + self.shape), np.empty((NVEL,) + self.shape)
        self._mcheck(self.lib.bflbm_multi_get_populations(self.h, f.ctypes.data, g.ctypes.data))
        return f, g

    def hydrovars(self):
        out = np.empty((NHYDRO,) + self.shape)
        self._mcheck(self.lib.bflbm_multi_get_hydrovars(self.h, out.ctypes.data))
        return out

    def hydrovars_bar(self):
        out = np.empty((NHYDRO_BAR,) + self.shape)
        self._mcheck(self.lib.bflbm_multi_get_hydrovars_bar(self.h, out.ctypes.data))
        return out

    def noise(self):
        fn, gn = np.empty((NVEL,) + self.shape), np.empty((NVEL,) + self.shape)
        self._mcheck(self.lib.bflbm_multi_get_noise(self.h, fn.ctypes.data, gn.ctypes.data))
        return fn, gn

    def total_mass(self):
        a, b = ctypes.c_double(), ctypes.c_double()
        self._mcheck(self.lib.bflbm_multi_total_mass(self.h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def droplet_covariance(self):
        com, c6, e = np.empty(3), np.empty(6), np.empty(3)
        self._mcheck(self.lib.bflbm_multi_droplet_covariance(self.h, com.ctypes.data, c6.ctypes.data, e.ctypes.data))
        cov = np.array([[c6[0], c6[3], c6[4]], [c6[3], c6[1], c6[5]], [c6[4], c6[5], c6[2]]])
        return com, cov, e

    def check_nan(self) -> int:
        n = ctypes.c_longlong()
        self._mcheck(self.lib.bflbm_multi_check_nan(self.h, ctypes.byref(n)))
        return n.value

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.bflbm_multi_kernel_launches(self.h))

    @property
    def device_bytes(self) -> int:
        return int(self.lib.bflbm_multi_device_bytes(self.h))


def philox4x32_10(ctr, key):
    """Device-side Philox4x32-10 block (known-answer test hook)."""
    lib = load_library()
    c = (ctypes.c_uint * 4)(*ctr)
    k = (ctypes.c_uint * 2)(*key)
    o = (ctypes.c_uint * 4)()
    _check(lib.bflbm_debug_philox(c, k, o))
    return tuple(int(v) for v in o)


# ---- the reference's function names (LBM_binary.H) ---------------------------------------------------
def LBM_init_mixture(lat: Lattice):
    """LBM_binary.H:598-629"""
    lat.init_mixture()


def LBM_init_stripe(frac: float, lat: Lattice):
    """LBM_binary.H:663-695"""
    lat.init_stripe(frac)


def LBM_init_droplet(r: float, lat: Lattice):
    """LBM_binary.H:698-742"""
    lat.init_droplet(r)


def LBM_init(lat: Lattice, f0, g0):
    """LBM_binary.H:631-661 (restart from populations)"""
    lat.init_from_populations(f0, g0)


def LBM_timestep(lat: Lattice, nsteps: int = 1):
    """LBM_binary.H:544-594"""
    lat.step(nsteps)


def LBM_hydrovars(lat: Lattice):
    """LBM_binary.H:297-313: the 22 real hydrodynamic fields"""
    return lat.hydrovars()


def LBM_hydrovars_density(lat: Lattice):
    """LBM_binary.H:342-354: hydrovsbar components 0..8"""
    return lat.hydrovars_bar()


def thermal_noise(lat: Lattice):
    """LBM_binary.H:73-132: (fnoise, gnoise) for the next collision"""
    return lat.noise()


def update_com(lat: Lattice):
    """LBM_hydrovs.H:26-60"""
    return lat.center_of_mass()[0]
