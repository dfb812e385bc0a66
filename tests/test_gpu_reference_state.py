"""Reference-state noise (USE_REF_STATE, LBM_binary.H:12, 92-107) on the one-pass brick kernel and on z-slabs.

The amplitudes of the noise come from equilibrium profiles of the whole box read at the cell shifted by the integer part of
(centre of mass now - centre of mass of the profiles).  On the brick kernel that centre of mass is taken from per-plane sums
(k_com_chunks + k_com_fold_chunks) after every step; a slab contributes its own planes and the caller sum-all-reduces them.  Checked here:

* every reference-state instantiation k_step_fused<true, RATE1, FULL, NT, true> against the CPU oracle with injected normals,
  and the device's shift against the one the oracle's density implies, step by step;
* a drifting droplet whose shift changes during the run;
* emulated slabs (2, 3, 4, uneven cuts, copies and peer stores, both CTA sizes) and bflbm_multi bit for bit against the whole box
  on the brick kernel, shift included;
* graph replay, the two-pass kernels, switching the reference state off, and the calls made in the wrong order;
* (two or more GPUs) NCCL ranks and the C++ driver with ngpus = 2.
Test states keep (com - com_ref) at least 1e-9 away from an integer, so that the truncation cannot depend on rounding.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import rel_err
from test_gpu_kernel_variants import _asymmetric_state, _assert_parity, _params, expected_variant

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 1e-12
# D3Q19 velocities (d3q19.cuh)
C = np.array([[0, 1, -1, 0, 0, 0, 0, 1, -1, 1, -1, 0, 0, 0, 0, 1, -1, 1, -1],
              [0, 0, 0, 1, -1, 0, 0, 1, -1, -1, 1, 1, -1, 1, -1, 0, 0, 0, 0],
              [0, 0, 0, 0, 0, 1, -1, 0, 0, 0, 0, 1, -1, -1, 1, 1, -1, -1, 1]])


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def ref_profiles(shape, rho_state, offset=(2.3, -1.6, 3.3)):
    """equilibrium profiles whose centre of mass lies `offset` (x, y, z) cells below that of the density rho_state: a Gaussian
    drop of rho (1e-3 .. 2.9) inside the box, so that (com - com_ref) starts near `offset`, far from integers, and the shift
    is non-zero on all three axes"""
    target = com_of(rho_state) - np.array(offset)
    zz, yy, xx = np.meshgrid(*(np.arange(n, dtype=np.float64) for n in shape[::-1]), indexing="ij")
    s = 0.1 * min(shape)
    c = target.copy()
    for _ in range(20):  # the thin uniform background pulls the centre of mass towards the middle of the box: place the drop
        rho_eq = 1e-3 + 2.9 * np.exp(-((xx - c[0]) ** 2 + (yy - c[1]) ** 2 + (zz - c[2]) ** 2) / (2 * s * s))
        c += target - com_of(rho_eq)  # so that the profile's centre of mass lands on target
    phi_eq = 3.1 - rho_eq
    return rho_eq, phi_eq, rho_eq + phi_eq


def droplet_rho(oracle_mod, shape):
    """rho of LBM_init_droplet(0.3) with the test parameters"""
    return oracle_mod.droplet_populations(*shape, 0.3, 0.1, 0.1, 3.0)[0].sum(axis=0)


def com_of(rho):
    """(x, y, z) centre of mass in cell indices"""
    zz, yy, xx = np.meshgrid(*(np.arange(n) for n in rho.shape), indexing="ij")
    m = rho.sum()
    return np.array([(rho * xx).sum() / m, (rho * yy).sum() / m, (rho * zz).sum() / m])


def expected_shift(rho, com_ref):
    """(int)(com - com_ref) per axis, C truncation; refuses a state on an integer knife edge"""
    d = com_of(rho) - com_ref
    assert np.abs(d - np.round(d)).min() > 1e-9, f"com - com_ref = {d} is too close to an integer for a rounding-proof test"
    return np.trunc(d).astype(np.int64)


def dyadic(a):
    """the values rounded to multiples of 2^-24: every sum of a cell's populations is then exact, so the densities a restart
    builds do not depend on where the box is cut into slabs"""
    return np.round(a * 2.0 ** 24) / 2.0 ** 24


def whole_box_ref(bflbm, shape, prm, eq, lz):
    """whole box with the reference state on the brick kernel"""
    lat = bflbm.Lattice(*shape, params=prm)
    lat.set_reference_state(*eq)
    lat.set_algorithm("fused")
    lat.set_tiling(lz)
    return lat


# ---- 1. the eight reference-state instantiations against the oracle --------------------------------------------------------
REF_SHAPES = [  # (NT, shape, brick height): FULL and partial tiles at both CTA sizes
    (256, (64, 16, 24), 8),
    (256, (40, 19, 20), 6),
    (128, (64, 8, 24), 8),
    (128, (40, 10, 20), 6),
]
TAUS = [(0.5, 0.5), (0.7, 0.55)]


@pytest.mark.parametrize("tau", TAUS, ids=["rate1", "general"])
@pytest.mark.parametrize("nt,shape,lz", REF_SHAPES, ids=[f"nt{nt}-{'x'.join(map(str, s))}" for nt, s, _ in REF_SHAPES])
def test_reference_state_brick_kernel_matches_oracle(bflbm, oracle_mod, monkeypatch, nt, shape, lz, tau):
    monkeypatch.setenv("BFLBM_CTA_THREADS", str(nt))
    prm = _params(1e-5, tau)
    f0, g0 = _asymmetric_state(oracle_mod, shape, seed=sum(shape) + nt)
    eq = ref_profiles(shape, f0.sum(axis=0))
    want = expected_variant("fused", nt, shape, lz, 1e-5, tau)
    assert want["noise"] == 1 and want["rate1"] == int(tau == (0.5, 0.5))
    with whole_box_ref(bflbm, shape, bflbm.Params(**prm, seed=31, step0=5), eq, lz) as lat:
        lat.init_from_populations(f0, g0)
        com_ref = lat.reference_com()
        O = oracle_mod.PortOracle(*shape)
        O.set_params(**prm)
        O.set_equilibrium(*eq)
        O.set_normals(lat.normals())
        O.init_from_populations(f0, g0)
        shift = lat.reference_shift()
        assert np.array_equal(shift, expected_shift(O.hydrovars()[0], com_ref)) and np.all(shift != 0), shift
        for s in range(4):
            fn, gn = lat.noise()
            fo, go = O.noise()
            tol = TOL if s == 0 else 10 * TOL
            assert rel_err(fn, fo) <= tol and rel_err(gn, go) <= tol, f"noise amplitudes before step {s + 1}"
            lat.step(1)
            O.set_normals(lat.normals())
            O.step(1)
            _assert_parity(lat, O, tol, f"REF nt{nt} {shape} tau {tau} step {s + 1}", want)
            assert lat.last_step() == (want if s else {**want, "fold_source": 0}), f"step {s + 1}"
            assert np.array_equal(lat.reference_shift(), expected_shift(O.hydrovars()[0], com_ref)), f"shift after step {s + 1}"


# ---- 2. the shift changes during the run --------------------------------------------------------------------------------
def test_shift_follows_a_drifting_droplet(bflbm, oracle_mod):
    """a droplet moving with u = (0.04, 0, 0.04) drifts 1.6 cells in 40 steps: its shift changes in x and z, and the device's
    sequence equals the one the oracle's densities give"""
    shape, lz = (24, 16, 20), 4
    prm = _params(1e-5, (0.5, 0.5))
    f, g = oracle_mod.droplet_populations(*shape, 0.3, 0.1, 0.1, 3.0)
    boost = (1 + 3 * (C.T @ np.array([0.04, 0.0, 0.04])))[:, None, None, None]
    f, g = f * boost, g * boost
    eq = ref_profiles(shape, f.sum(axis=0))
    with whole_box_ref(bflbm, shape, bflbm.Params(**prm, seed=5), eq, lz) as lat:
        lat.init_from_populations(f, g)
        com_ref = lat.reference_com()
        O = oracle_mod.PortOracle(*shape)
        O.set_params(**prm)
        O.set_equilibrium(*eq)
        O.set_normals(lat.normals())
        O.init_from_populations(f, g)
        gpu, cpu = [], []
        for _ in range(40):
            lat.step(1)
            O.set_normals(lat.normals())
            O.step(1)
            gpu.append(tuple(lat.reference_shift()))
            cpu.append(tuple(expected_shift(O.hydrovars()[0], com_ref)))
        assert gpu == cpu
        assert len({s[0] for s in gpu}) >= 2 and len({s[2] for s in gpu}) >= 2, gpu
        assert rel_err(lat.populations()[0], O.populations()[0]) <= 1e-10


# ---- 3. slabs bit for bit against the whole box ---------------------------------------------------------------------------
SLAB_SHAPE, SLAB_LZ = (32, 16, 48), 4
SLAB_CASES = [  # (slabs, zsplit, peer, NT, init, tau)
    (2, None, False, 256, "droplet", (0.5, 0.5)),
    (2, None, True, 128, "populations", (0.7, 0.55)),
    (3, (0, 12, 28, 48), False, 128, "droplet", (0.5, 0.5)),
    (3, (0, 12, 28, 48), True, 256, "populations", (0.5, 0.5)),
    (4, (0, 8, 20, 36, 48), False, 256, "populations", (0.7, 0.55)),
    (4, None, True, 128, "droplet", (0.7, 0.55)),
]


@pytest.mark.parametrize("nslabs,zsplit,peer,nt,init,tau", SLAB_CASES,
                         ids=[f"{c[0]}slabs-{'uneven' if c[1] else 'even'}-{'peer' if c[2] else 'copies'}-nt{c[3]}-{c[4]}"
                              for c in SLAB_CASES])
def test_slabs_bitwise_equal_to_whole_box(bflbm, oracle_mod, monkeypatch, nslabs, zsplit, peer, nt, init, tau):
    """the shift is the same on every slab and step as on the whole box, and after 20 steps populations and noise are the same
    bits; the equilibrium lies ~3 planes off in z, so the shifted reads cross the slab faces"""
    from bflbm_b200.distributed import EmulatedSlabs
    monkeypatch.setenv("BFLBM_CTA_THREADS", str(nt))
    prm = bflbm.Params(**_params(1e-5, tau), seed=99)
    eq = ref_profiles(SLAB_SHAPE, droplet_rho(oracle_mod, SLAB_SHAPE))
    with whole_box_ref(bflbm, SLAB_SHAPE, prm, eq, SLAB_LZ) as W:
        S = EmulatedSlabs(*SLAB_SHAPE, nslabs, params=prm, brick_lz=SLAB_LZ, peer=peer, zsplit=zsplit)
        try:
            S.set_reference_state(*eq)
            if init == "droplet":  # absolute centre of mass for the first step (LBM_binary.H:623-625)
                W.init_droplet(0.3)
                S.init_droplet(0.3)
            else:                  # restart: com - com_ref
                f0, g0 = (dyadic(a) for a in _asymmetric_state(oracle_mod, SLAB_SHAPE, seed=7 + nslabs))
                W.init_from_populations(f0, g0)
                S.init_from_global_populations(f0, g0)
            shifts = set()
            for s in range(21):
                sw = W.reference_shift()
                shifts.add(int(sw[2]))
                for r, lat in enumerate(S.lats):
                    assert np.array_equal(lat.reference_shift(), sw), f"slab {r} before step {s + 1}"
                if s == 20:
                    break
                W.step(1)
                S.step(1)
            assert 0 not in shifts, shifts
            fw, gw = W.populations()
            fs, gs = S.gather("populations")
            assert np.array_equal(fw, fs) and np.array_equal(gw, gs)
            nw, ns = W.noise(), S.gather("noise")
            assert np.array_equal(nw[0], ns[0]) and np.array_equal(nw[1], ns[1])
            assert W.last_step()["threads"] == nt and all(lat.last_step()["noise"] == 1 for lat in S.lats)
            if peer:
                assert all(lat.halo_error() == 0 for lat in S.lats)
        finally:
            S.close()


def test_slabs_keep_the_shift_current_at_kbt0_then_raise_kbt(bflbm, oracle_mod):
    """kBT = 0: the plain kernels run, but every step still takes the centre of mass and its exchange.  After set_params raises
    kBT mid-run the reference-state kernels start from a current shift: slabs and whole box agree bit for bit throughout, and
    the shift is the one the whole box's density gives"""
    from bflbm_b200.distributed import EmulatedSlabs
    prm = bflbm.Params(**_params(0.0, (0.5, 0.5)), seed=21)
    eq = ref_profiles(SLAB_SHAPE, droplet_rho(oracle_mod, SLAB_SHAPE))
    with whole_box_ref(bflbm, SLAB_SHAPE, prm, eq, SLAB_LZ) as W:
        S = EmulatedSlabs(*SLAB_SHAPE, 3, params=prm, brick_lz=SLAB_LZ)
        try:
            S.set_reference_state(*eq)
            W.init_droplet(0.3)
            S.init_droplet(0.3)
            com_ref = W.reference_com()
            for s in range(10):
                if s == 5:
                    W.set_params(kBT=1e-5)
                    for lat in S.lats:
                        lat.set_params(kBT=1e-5)
                W.step(1)
                S.step(1)
                assert W.last_step()["noise"] == int(s >= 5)
                sw = W.reference_shift()
                assert np.array_equal(sw, expected_shift(W.hydrovars()[0], com_ref)), f"step {s + 1}"
                assert all(np.array_equal(lat.reference_shift(), sw) for lat in S.lats), f"step {s + 1}"
            fw, gw = W.populations()
            fs, gs = S.gather("populations")
            assert np.array_equal(fw, fs) and np.array_equal(gw, gs)
            assert np.array_equal(W.noise()[0], S.gather("noise")[0])
        finally:
            S.close()


def test_whole_box_stepped_like_a_slab(bflbm, oracle_mod):
    """a whole box on the reference-state brick kernel stepped through bflbm_step_begin / bflbm_step_end (the centre of mass is
    then taken in step_end) gives the bits and the shifts of bflbm_step"""
    shape = (32, 16, 24)
    prm = bflbm.Params(**_params(1e-5, (0.7, 0.55)), seed=33)
    eq = ref_profiles(shape, droplet_rho(oracle_mod, shape))
    with whole_box_ref(bflbm, shape, prm, eq, 4) as A, whole_box_ref(bflbm, shape, prm, eq, 4) as B:
        for lat in (A, B):
            lat.init_droplet(0.3)
        lib = B.lib
        for s in range(6):
            A.step(1)
            assert lib.bflbm_step_begin(B.h) == 0 and lib.bflbm_step_end(B.h) == 0
            assert np.array_equal(A.reference_shift(), B.reference_shift()), f"step {s + 1}"
        for a, b in zip(A.populations() + A.noise(), B.populations() + B.noise()):
            assert np.array_equal(a, b)


# ---- 4. bflbm_multi ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("devices", [(0, 0, 0), (0, 1)], ids=["3slabs-one-gpu", "2gpus"])
def test_multi_lattice_bitwise_equal_to_whole_box(bflbm, oracle_mod, devices):
    if max(devices) + 1 > _ngpus():
        pytest.skip(f"needs {max(devices) + 1} GPUs")
    shape, lz = (32, 16, 16 * len(devices)), 4
    prm = bflbm.Params(**_params(1e-5, (0.7, 0.55)), seed=4711)
    eq = ref_profiles(shape, droplet_rho(oracle_mod, shape))
    with whole_box_ref(bflbm, shape, prm, eq, lz) as W, \
            bflbm.MultiLattice(*shape, params=prm, ngpus=len(devices), devices=list(devices), brick_lz=lz) as M:
        M.set_reference_state(*eq)
        W.init_droplet(0.3)
        M.init_droplet(0.3)
        for _ in range(4):
            W.step(5)
            M.step(5)
            for r in range(len(devices)):
                assert np.array_equal(M.reference_shift(r), W.reference_shift())
        fw, gw = W.populations()
        fm, gm = M.populations()
        assert np.array_equal(fw, fm) and np.array_equal(gw, gm)
        assert np.array_equal(W.noise()[0], M.noise()[0])
        # restart from exactly summable populations, then step again
        f0, g0 = dyadic(fw), dyadic(gw)
        W.init_from_populations(f0, g0)
        M.init_from_populations(f0, g0)
        W.step(6)
        M.step(6)
        assert np.array_equal(W.populations()[1], M.populations()[1])
        assert np.array_equal(M.reference_shift(len(devices) - 1), W.reference_shift())
        assert M.check_nan() == 0


# ---- 5. graphs, two-pass kernels, switching off ---------------------------------------------------------------------------
def test_graph_replay_bitwise_equal_to_plain_launches(bflbm, oracle_mod, monkeypatch):
    shape = (32, 32, 32)
    prm = bflbm.Params(**_params(1e-5, (0.5, 0.5)), seed=2024)
    eq = ref_profiles(shape, droplet_rho(oracle_mod, shape))
    monkeypatch.setenv("BFLBM_GRAPH", "0")
    with whole_box_ref(bflbm, shape, prm, eq, 0) as P:
        monkeypatch.delenv("BFLBM_GRAPH")
        with whole_box_ref(bflbm, shape, prm, eq, 0) as Gr:
            for lat in (P, Gr):
                lat.init_droplet(0.3)
            for n in (1, 23, 2, 16):
                P.step(n)
                Gr.step(n)
                assert np.array_equal(P.reference_shift(), Gr.reference_shift())
                fp, gp = P.populations()
                fg, gg = Gr.populations()
                assert np.array_equal(fp, fg) and np.array_equal(gp, gg), f"graph replay differs after a call of {n} steps"
            assert Gr.last_step()["graph"] == 1 and P.last_step()["graph"] == 0 and Gr.last_step()["algorithm"] == 0


@pytest.mark.parametrize("tau", TAUS, ids=["rate1", "general"])
def test_brick_and_two_pass_kernels_agree(bflbm, oracle_mod, tau):
    shape = (24, 20, 28)
    prm = bflbm.Params(**_params(1e-5, tau), seed=8)
    f0, g0 = _asymmetric_state(oracle_mod, shape, seed=3)
    eq = ref_profiles(shape, f0.sum(axis=0))
    with whole_box_ref(bflbm, shape, prm, eq, 4) as B, bflbm.Lattice(*shape, params=prm) as T:
        T.set_reference_state(*eq)  # a whole box: the two-pass kernels
        for lat in (B, T):
            lat.init_from_populations(f0, g0)
        for s in range(4):
            assert np.array_equal(B.reference_shift(), T.reference_shift()), f"before step {s + 1}"
            B.step(1)
            T.step(1)
            assert T.last_step()["algorithm"] == 1 and B.last_step()["algorithm"] == 0
            for a, b in zip(B.populations(), T.populations()):
                assert rel_err(a, b) <= 10 * TOL
            for a, b in zip(B.noise(), T.noise()):
                assert rel_err(a, b) <= 10 * TOL
        assert np.array_equal(B.reference_shift(), T.reference_shift())


def test_reference_state_off_gives_the_shipped_noise(bflbm, oracle_mod):
    shape = (32, 16, 24)
    prm = bflbm.Params(**_params(1e-5, (0.5, 0.5)), seed=12)
    eq = ref_profiles(shape, droplet_rho(oracle_mod, shape))
    with whole_box_ref(bflbm, shape, prm, eq, 4) as A, bflbm.Lattice(*shape, params=prm) as B:
        A.init_droplet(0.3)
        A.step(3)
        bytes_on = A.device_bytes
        A.set_reference_state(None)
        assert bytes_on - A.device_bytes == 24 * np.prod(shape)
        f, g = A.populations()
        B.set_algorithm("fused")
        B.set_tiling(4)
        for lat in (A, B):
            lat.init_from_populations(f, g)
            lat.step(2)
        assert A.last_step() == B.last_step()
        for a, b in zip(A.populations() + A.noise(), B.populations() + B.noise()):
            assert np.array_equal(a, b)


# ---- 6. calls in the wrong order ------------------------------------------------------------------------------------------
def test_state_errors(bflbm, oracle_mod):
    from bflbm_b200.distributed import EmulatedSlabs
    shape = (16, 16, 16)
    eq = ref_profiles(shape, droplet_rho(oracle_mod, shape))
    prm = bflbm.Params(**_params(1e-5, (0.5, 0.5)))
    S = EmulatedSlabs(*shape, 2, params=prm, brick_lz=4, peer=True)
    try:
        lib = S.lats[0].lib
        for lat in S.lats:
            lat.set_reference_state(*eq)  # no exchange: done by hand below
            assert lib.bflbm_com_doubles(lat.h) == 4 * shape[2]
            lat.init_droplet(0.3)
        assert lib.bflbm_step_begin(S.lats[0].h) == -3 and "pending" in lib.bflbm_last_error().decode()
        assert lib.bflbm_step_slab(S.lats[0].h, 1) == -3 and "bflbm_com_update" in lib.bflbm_last_error().decode()
        with pytest.raises(bflbm.BflbmError, match="no centre of mass pending"):
            S.lats[0].com_update()
            S.lats[0].com_update()
        a = np.ascontiguousarray(eq[0])
        assert lib.bflbm_set_reference_state(S.lats[1].h, a.ctypes.data, None, None) == -1
        assert lib.bflbm_set_reference_state(S.lats[1].h, a.ctypes.data, a.ctypes.data, None) == -1
        with pytest.raises(ValueError):
            S.lats[1].set_reference_state(eq[0][:8], eq[1][:8], eq[2][:8])  # a slab takes the whole box
    finally:
        S.close()
    with bflbm.Lattice(*shape, params=prm) as W:
        with pytest.raises(bflbm.BflbmError, match="no reference state"):
            W.reference_shift()


# ---- 7. several GPUs ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["nccl", "peer"])
def test_nccl_ranks_bitwise_equal_to_whole_box(mode):
    world = 2
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29680 + (1 if mode == "peer" else 0)), os.path.join(HERE, "mp_refstate_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, MP_PEER="1" if mode == "peer" else "0"))
    assert r.returncode == 0 and f"MP_REFSTATE_OK {world} {mode}" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def _plotfiles(root):
    """{relative path: float64 data} of the Cell_D files of the fluctuating run under root"""
    out = {}
    for dirpath, _, files in os.walk(root):
        for fn in files:
            if fn.startswith("Cell_D") and "_continue" in dirpath:
                raw = open(os.path.join(dirpath, fn), "rb").read()
                out[os.path.relpath(os.path.join(dirpath, fn), root)] = np.frombuffer(raw[raw.index(b"\n") + 1:], dtype="<f8")
    return out


def test_driver_reference_state_on_two_gpus(bflbm, tmp_path):
    """the driver's use_ref_state job with ngpus = 2 (brick kernel on slabs) against ngpus = 1 (two-pass kernels), both on the
    equilibrium profiles of one kBT = 0 run: the same plotfiles to 1e-10"""
    if _ngpus() < 2:
        pytest.skip("needs 2 GPUs")
    import shutil
    from bflbm_b200 import host_driver
    exe = host_driver.build()
    common = "system = droplet\nnx = 24\nny = 16\nnz = 32\nalpha0 = 1.5\nkappa = 0.1\nrho_lo = 0.1\nrho_hi = 3.\nradius = 0.3\n" \
             "plot_int = 10\nprint_int = 10\nout_step = 0\nplot_fields = hydrovars\n"
    eq = tmp_path / "eq"
    eq.mkdir()
    (eq / "Parameters").write_text(common + f"kBT = 0\nnsteps = 20\nroot_path = {eq}\nngpus = 1\n")
    r = subprocess.run([exe, str(eq / "Parameters")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    outs = []
    for n in (1, 2):
        root = tmp_path / f"run{n}"
        shutil.copytree(eq, root)  # the equilibrium_* profiles of the kBT = 0 run
        (root / "Parameters").write_text(common + f"kBT = 1e-5\nnsteps = 30\nroot_path = {root}\nngpus = {n}\nuse_ref_state = 1\n")
        r = subprocess.run([exe, str(root / "Parameters")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr + r.stdout
        outs.append(_plotfiles(root))
    assert len(outs[0]) >= 4 and outs[0].keys() == outs[1].keys()
    for k, a in outs[0].items():
        b = outs[1][k]
        assert a.shape == b.shape and np.abs(a - b).max() <= 1e-10 * np.abs(a).max(), k
