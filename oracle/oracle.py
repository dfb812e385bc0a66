"""TEST INFRASTRUCTURE ONLY -- ctypes loaders for the two CPU checkers.

* ``RefOracle``  : the reference's own headers (LBM_d3q19.H, LBM_binary.H) compiled
                   unchanged over oracle/shim (oracle/_ref/libbflbm_ref*.so, built by
                   oracle/Makefile in the container that has /root/reference).
* ``PortOracle`` : the plain-C restatement oracle/bflbm_oracle.c.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
leg may import this module.  The product (the package and its CUDA library) never does.

All arrays are float64, C-contiguous, shape (ncomp, nz, ny, nx): that is AMReX FAB
order (x fastest ... component slowest) for the valid region.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = ctypes.c_void_p
_d = ctypes.c_double
_i = ctypes.c_int


def build(quiet: bool = True) -> None:
    """Compile the checkers (port always; _ref only where /root/reference exists)."""
    subprocess.run(["make", "-C", _HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def _ptr(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


class _Base:
    prefix = ""
    lib = None

    def __init__(self, nx, ny, nz):
        self.nx, self.ny, self.nz = int(nx), int(ny), int(nz)
        self.shape = (self.nz, self.ny, self.nx)
        self._keep = None
        self.h = self._fn("create", _dp, [_i, _i, _i])(self.nx, self.ny, self.nz)

    def _fn(self, name, restype, argtypes):
        f = getattr(self.lib, self.prefix + name)
        f.restype, f.argtypes = restype, argtypes
        return f

    def close(self):
        if self.h:
            self._fn("destroy", None, [_dp])(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- inits ---------------------------------------------------------------
    def init_mixture(self):
        self._fn("init_mixture", None, [_dp])(self.h)

    def init_stripe(self, frac=0.5):
        self._fn("init_stripe", None, [_dp, _d])(self.h, frac)

    def init_droplet(self, radius=0.2):
        self._fn("init_droplet", None, [_dp, _d])(self.h, radius)

    def init_from_populations(self, f, g):
        f = np.ascontiguousarray(f, dtype=np.float64)
        g = np.ascontiguousarray(g, dtype=np.float64)
        assert f.shape == (19,) + self.shape and g.shape == f.shape
        self._fn("init_from_populations", None, [_dp, _dp, _dp])(self.h, _ptr(f), _ptr(g))

    def step(self, n=1):
        self._fn("step", None, [_dp, _i])(self.h, int(n))

    # -- outputs -------------------------------------------------------------
    def populations(self):
        f = np.empty((19,) + self.shape)
        g = np.empty((19,) + self.shape)
        self._fn("get_populations", None, [_dp, _dp, _dp])(self.h, _ptr(f), _ptr(g))
        return f, g

    def hydrovars(self):
        out = np.empty((22,) + self.shape)
        self._fn("get_hydrovars", None, [_dp, _dp])(self.h, _ptr(out))
        return out

    def hydrovars_bar(self):
        out = np.empty((9,) + self.shape)
        self._fn("get_hydrovars_bar", None, [_dp, _dp])(self.h, _ptr(out))
        return out

    def noise(self):
        fn = np.empty((19,) + self.shape)
        gn = np.empty((19,) + self.shape)
        self._fn("get_noise", None, [_dp, _dp, _dp])(self.h, _ptr(fn), _ptr(gn))
        return fn, gn

    # -- unit helpers ----------------------------------------------------------
    @classmethod
    def moments(cls, f19):
        f19 = np.ascontiguousarray(f19, dtype=np.float64)
        m = np.empty(19)
        fn = getattr(cls.lib, cls.prefix + "moments")
        fn.restype, fn.argtypes = None, [_dp, _dp]
        fn(_ptr(f19), _ptr(m))
        return m

    @classmethod
    def populations_from_moments(cls, m19):
        m19 = np.ascontiguousarray(m19, dtype=np.float64)
        f = np.empty(19)
        fn = getattr(cls.lib, cls.prefix + "populations")
        fn.restype, fn.argtypes = None, [_dp, _dp]
        fn(_ptr(m19), _ptr(f))
        return f

    @classmethod
    def constants(cls):
        c = np.empty((19, 3), dtype=np.int32)
        w = np.empty(19)
        b = np.empty(19)
        fn = getattr(cls.lib, cls.prefix + "constants")
        fn.restype, fn.argtypes = None, [_dp, _dp, _dp]
        fn(c.ctypes.data_as(_dp), _ptr(w), _ptr(b))
        return c, w, b


def _load(path):
    return ctypes.CDLL(path) if os.path.exists(path) else None


class PortOracle(_Base):
    """oracle/bflbm_oracle.c.  ``fast=True`` loads the -O3/OpenMP build (timing only)."""
    prefix = "oracle_"

    def __init__(self, nx, ny, nz, fast=False):
        path = os.path.join(_HERE, "libbflbm_oracle_fast.so" if fast else "libbflbm_oracle.so")
        if not os.path.exists(path):
            build()
        type(self).lib = ctypes.CDLL(path)
        super().__init__(nx, ny, nz)
        self.params = dict(kBT=0.0, tau_f=0.5, tau_g=0.5, alpha0=4.0, alpha1=0.0, kappa=4.0, rho_lo=0.0, rho_hi=1.0)

    def set_params(self, **kw):
        self.params.update(kw)
        p = self.params
        self._fn("set_params", None, [_dp] + [_d] * 8)(
            self.h, p["kBT"], p["tau_f"], p["tau_g"], p["alpha0"], p["alpha1"], p["kappa"], p["rho_lo"], p["rho_hi"])

    def num_threads(self):
        return self._fn("num_threads", _i, [])()

    def set_num_threads(self, n):
        self._fn("set_num_threads", None, [_i])(int(n))

    def set_equilibrium(self, rho_eq, phi_eq, rhot_eq):
        """USE_REF_STATE noise (LBM_binary.H:12, 92-107): amplitudes from these (nz, ny, nx) profiles, COM-shifted; None = off."""
        if rho_eq is None:
            self._fn("set_equilibrium", None, [_dp, _dp, _dp, _dp])(self.h, None, None, None)
            return
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (rho_eq, phi_eq, rhot_eq)]
        assert all(v.shape == self.shape for v in a)
        self._fn("set_equilibrium", None, [_dp, _dp, _dp, _dp])(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]))

    def set_ref_shift(self, shift):
        """the integer (x, y, z) shift the next reference-state noise generations read the equilibrium profiles with, in place
        of (int)(com - com_ref); None (the default) computes it again.  An oracle on a window of a larger box takes that
        box's shift this way (or shift 0 with profiles cut at window offset - shift)."""
        s = None if shift is None else (ctypes.c_int * 3)(*(int(v) for v in shift))
        self._fn("set_ref_shift", None, [_dp, _dp])(self.h, s)

    def set_normals(self, normals):
        """normals: (nz, ny, nx, 33) standard normals for the next noise generation, or None."""
        if normals is None:
            self._keep = None
            self._fn("set_normals", None, [_dp, _dp])(self.h, None)
        else:
            self._keep = np.ascontiguousarray(normals, dtype=np.float64)
            assert self._keep.shape == self.shape + (33,)
            self._fn("set_normals", None, [_dp, _dp])(self.h, _ptr(self._keep))


class RefOracle(_Base):
    """The reference headers themselves (oracle/_ref).  rho_lo/rho_hi are compile-time
    constants there (LBM_binary.H:25-26): other values enter through init_from_populations."""
    prefix = "ref_"

    @staticmethod
    def available(fast=False, ref_state=False):
        name = "libbflbm_ref_refstate.so" if ref_state else ("libbflbm_ref_fast.so" if fast else "libbflbm_ref.so")
        return os.path.exists(os.path.join(_HERE, "_ref", name))

    def __init__(self, nx, ny, nz, fast=False, ref_state=False):
        """ref_state: the build with -DUSE_REF_STATE (the reference's globals live in the library: one parameter set per build)."""
        name = "libbflbm_ref_refstate.so" if ref_state else ("libbflbm_ref_fast.so" if fast else "libbflbm_ref.so")
        path = os.path.join(_HERE, "_ref", name)
        self.lib = ctypes.CDLL(path)  # instance attribute: the USE_REF_STATE build is a different library
        if not ref_state:
            type(self).lib = self.lib
        super().__init__(nx, ny, nz)
        self.params = dict(kBT=0.0, tau_f=0.5, tau_g=0.5, alpha0=4.0, alpha1=0.0, kappa=4.0)
        self.set_rng(0, 12345)

    @property
    def rho_lo(self):
        return self._fn("rho_lo", _d, [])()

    @property
    def rho_hi(self):
        return self._fn("rho_hi", _d, [])()

    def set_params(self, **kw):
        kw.pop("rho_lo", None)
        kw.pop("rho_hi", None)
        self.params.update(kw)
        p = self.params
        self._fn("set_params", None, [_d] * 6)(p["kBT"], p["tau_f"], p["tau_g"], p["alpha0"], p["alpha1"], p["kappa"])

    def set_rng(self, mode, seed=12345, normals=None):
        if normals is not None:
            self._keep = np.ascontiguousarray(normals, dtype=np.float64)
            assert self._keep.shape == self.shape + (33,)
            ptr = _ptr(self._keep)
        else:
            self._keep, ptr = None, None
        self._fn("set_rng", None, [_i, ctypes.c_ulong, _dp])(int(mode), int(seed), ptr)

    def set_normals(self, normals):
        if normals is None:
            self.set_rng(0, 12345)
        else:
            self.set_rng(1, 12345, normals)

    def num_threads(self):
        return self._fn("num_threads", _i, [])()

    def set_num_threads(self, n):
        self._fn("set_num_threads", None, [_i])(int(n))

    def set_equilibrium(self, rho_eq, phi_eq, rhot_eq):
        a = [np.ascontiguousarray(v, dtype=np.float64) for v in (rho_eq, phi_eq, rhot_eq)]
        assert all(v.shape == self.shape for v in a)
        self._fn("set_equilibrium", None, [_dp, _dp, _dp, _dp])(self.h, _ptr(a[0]), _ptr(a[1]), _ptr(a[2]))

    def uses_ref_state(self):
        return bool(self._fn("uses_ref_state", _i, [])())


def stripe_populations(nx, ny, nz, frac, kappa, rho_lo, rho_hi):
    """Initial populations of LBM_init_stripe (LBM_binary.H:672-686) for arbitrary rho_lo/rho_hi,
    used to drive RefOracle (whose rho_lo/rho_hi are compile-time) through its restart entry."""
    p = PortOracle(nx, ny, nz)
    p.set_params(kappa=kappa, rho_lo=rho_lo, rho_hi=rho_hi)
    p.init_stripe(frac)
    return p.populations()


def droplet_populations(nx, ny, nz, radius, kappa, rho_lo, rho_hi):
    p = PortOracle(nx, ny, nz)
    p.set_params(kappa=kappa, rho_lo=rho_lo, rho_hi=rho_hi)
    p.init_droplet(radius)
    return p.populations()


class RefFit:
    """The reference's droplet (W, R) fit: externlib.H compiled unchanged (oracle/_ref/libbflbm_ref_fit.so, oracle/ref_fit_wrapper.cpp)."""

    @staticmethod
    def available():
        return os.path.exists(os.path.join(_HERE, "_ref", "libbflbm_ref_fit.so"))

    def __init__(self):
        self.lib = ctypes.CDLL(os.path.join(_HERE, "_ref", "libbflbm_ref_fit.so"))
        self.lib.ref_fit_coefficients.argtypes = [_d] * 6 + [_dp]
        self.lib.ref_fit_field_terms.argtypes = [_dp, _i, _i, _i, _d, _d, _dp]
        self.lib.ref_fit_droplet.argtypes = [_dp, _i, _i, _i, _i, _d, _i, _d, _d, _d, _d, _d, _d, _dp, _dp]
        self.lib.ref_fit_droplet.restype = _i

    def coefficients(self, W, R, eta_W=0.2, eta_R=0.2, dt=0.02, C0=1.0):
        out = np.empty(6)
        self.lib.ref_fit_coefficients(W, R, eta_W, eta_R, dt, C0, _ptr(out))
        return out

    def field_terms(self, rho, W, R):
        """(M_f(W), M_f(R), com[3]) of a (nz, ny, nx) density field, unit-cube coordinates."""
        rho = np.ascontiguousarray(rho, dtype=np.float64)
        nz, ny, nx = rho.shape
        out = np.empty(5)
        self.lib.ref_fit_field_terms(_ptr(rho), nx, ny, nz, W, R, _ptr(out))
        return out[0], out[1], out[2:]

    def fit(self, rho, W0, R0, step_window=20, undul_ratio=0.01, nstep=400, eta_W=0.2, eta_R=0.2, dt=0.02):
        """fittingDropletParams (LBM_hydrovs.H:160-213): (W, R, undulation, converged, trace[nstep, 2])."""
        rho = np.ascontiguousarray(rho, dtype=np.float64)
        nz, ny, nx = rho.shape
        out, trace = np.empty(3), np.empty((nstep, 2))
        rc = self.lib.ref_fit_droplet(_ptr(rho), nx, ny, nz, step_window, undul_ratio, nstep, W0, R0, eta_W, eta_R, dt, 1e-6, _ptr(out), _ptr(trace))
        return float(out[0]), float(out[1]), float(out[2]), rc == 0, trace
