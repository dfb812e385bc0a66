"""Reference-state noise on large planes and at 512^3, against the oracle and exact centre-of-mass sums.

tests/test_gpu_reference_state.py checks the reference-state noise on boxes whose planes hold at most 1024 cells.  The code that
exists for large boxes does not run there:

* k_com_chunks sums each plane in chunks of COM_CHUNK = 8192 cells: a second chunk, a partial last chunk and a chunk boundary
  inside a row need planes of more than 8192 cells, and k_com_fold_chunks adds the chunks of a plane in order;
* k_com_fold_chunks runs (nz_global + 127) / 128 CTAs: more than one needs nz_global > 128;
* k_com_shift (two-pass kernels) has thread t add the k_diag block partials t, t + 256, ...: the loop runs more than once only
  with more than 256 blocks;
* at 512^3 the equilibrium profiles pass 2^31 bytes, the host sums com_ref over 1.3e8 cells, and the first shift after an
  analytic init is the absolute centre of mass (~255 per axis), so that about half the cells wrap on each axis.

Checked here: mid-size boxes that reach every one of these paths against the oracle with injected normals, the per-plane sums in
bflbm_com_buffer against numpy after every init and step; emulated slabs with large planes bit for bit against the whole box;
and the 512^3 box restarted from the periodically tiled state of tests/test_gpu_tiled_fullsize.py, whose shift and plane sums
are checked against numpy and whose populations are checked on three 64^3 windows against oracles that take the big box's
shift through PortOracle.set_ref_shift.  The CPU tests pin that hook and show that the case table reaches each path.
"""
import resource
import time

import numpy as np
import pytest

from conftest import rel_err
from test_gpu_kernel_variants import _asymmetric_state, _assert_parity, _params, ceil_div, expected_variant, twopass_block
from test_gpu_reference_state import C, com_of, dyadic, expected_shift, whole_box_ref
from test_gpu_tiled_fullsize import (BENCH_VARIANT, LZ, N, T, WINDOWS, W, _assert_windows, _bench_params, _cut, _device_download,
                                     _free_device, _settle, _tile, _tiled, _window_normals)

TOL = 1e-12
KBT = 1e-5
OFFSET = (2.3, -1.6, 3.3)  # com(state) - com(profiles): far from integers, non-zero shift on every axis
TAUS = [(0.5, 0.5), (0.7, 0.55)]


# ---- references ----------------------------------------------------------------------------------------------------------
def plane_sums(rho):
    """(nz, 4): {sum rho, sum rho x, sum rho y, sum rho z} of every plane of a (nz, ny, nx) density, cell indices as coordinates:
    what the device's com_buffer holds on a whole box after every step and init"""
    nz, ny, nx = rho.shape
    m = rho.sum(axis=(1, 2))
    sx = rho.sum(axis=1) @ np.arange(nx, dtype=np.float64)
    sy = rho.sum(axis=2) @ np.arange(ny, dtype=np.float64)
    return np.stack([m, sx, sy, m * np.arange(nz, dtype=np.float64)], axis=1)


def com_of_planes(planes):
    s = planes.sum(axis=0)
    return s[1:] / s[0]


def shift_of_planes(planes, com_ref=None):
    """expected_shift from plane sums: (int)(com - com_ref), or (int)com after an analytic init (com_ref None)"""
    d = com_of_planes(planes) - (0.0 if com_ref is None else com_ref)
    assert np.abs(d - np.round(d)).min() > 1e-9, f"com - com_ref = {d} is too close to an integer for a rounding-proof test"
    return np.trunc(d).astype(np.int64)


def com_buffer(lat):
    """the device's (nz_global, 4) per-plane sums behind the shift (bflbm_com_buffer)"""
    from bflbm_b200.distributed import _device_tensor
    import torch
    lat.sync()
    nz = lat.nz_global
    return _device_tensor(lat.com_buffer_pointer(), 4 * nz, torch.device("cuda", lat.device)).cpu().numpy().reshape(nz, 4)


def plane_errors(got, want):
    """per plane: max |got - want| over the four sums, relative to the plane's largest entry"""
    return np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)


def assert_plane_sums(got, want, tol, what):
    e = plane_errors(got, want)
    z = int(np.argmax(e))
    assert e[z] <= tol, f"{what}: com_buffer plane {z} off by {e[z]:.3e} of its largest entry ({got[z]} vs {want[z]})"


def drop_profiles(shape, target):
    """ref_profiles' Gaussian drop (rho 1e-3 .. 2.9) with its centre of mass on target, but 0.1 of the box wide on each axis
    rather than 0.1 of its shortest edge: on a thin box such as 512 x 40 x 12 a 1.2-cell drop weighs less than the background
    and cannot carry the centre of mass to target.  Placed with 1-D sums of the separable drop, so that 512^3 costs one pass."""
    axes = [np.arange(n, dtype=np.float64) for n in shape]
    cells = float(np.prod(shape))
    c = np.array(target, dtype=np.float64)
    for _ in range(30):
        g = [np.exp(-(a - ci) ** 2 / (2 * (0.1 * len(a)) ** 2)) for a, ci in zip(axes, c)]
        m1 = [gi.sum() for gi in g]
        mass = 1e-3 * cells + 2.9 * np.prod(m1)
        com = np.array([(1e-3 * cells / shape[d] * axes[d].sum() + 2.9 * (axes[d] * g[d]).sum() * np.prod(m1) / m1[d]) / mass
                        for d in range(3)])
        c += target - com
    rho_eq = g[2][:, None, None] * g[1][None, :, None] * g[0][None, None, :]
    rho_eq *= 2.9
    rho_eq += 1e-3
    phi_eq = 3.1 - rho_eq
    return rho_eq, phi_eq, rho_eq + phi_eq


def profiles_below(rho_state):
    """drop_profiles whose centre of mass lies OFFSET below that of rho_state"""
    return drop_profiles(rho_state.shape[::-1], com_of(rho_state) - np.array(OFFSET))


# ---- restatement of the centre-of-mass launches (kernels.cuh, capi.cu update_ref_shift) --------------------------------------
COM_THREADS, COM_CHUNK = 256, 32 * 256


def com_chunks(shape):
    """[c0, c1) cell ranges of k_com_chunks in one plane"""
    plane = shape[0] * shape[1]
    return [(c0, min(c0 + COM_CHUNK, plane)) for c0 in range(0, plane, COM_CHUNK)]


def fold_ctas(shape):
    """CTAs of k_com_fold_chunks: one thread per global plane, 128 per CTA"""
    return ceil_div(shape[2], 128)


def diag_blocks(shape):
    """blocks of k_diag (the two-pass kernels' cell grid) whose partials k_com_shift adds"""
    bx, by = twopass_block(shape[0])
    return ceil_div(shape[0], bx) * ceil_div(shape[1], by) * shape[2]


# ---- cases ---------------------------------------------------------------------------------------------------------------------
MID = [  # (shape, brick height, what it covers)
    ((136, 72, 20), 6, "2 chunks, the second partial; the chunk boundary inside row 60; partial tiles"),
    ((512, 40, 12), 4, "3 chunks on a thin box, 512-wide rows as at 512^3; full tiles"),
    ((96, 96, 136), 8, "nz > 128: k_com_fold_chunks runs 2 CTAs; 1.25 M cells"),
]
MID_CASES = ([("fused", nt, shape, lz, tau) for shape, lz, _ in MID for nt in (256, 128) for tau in TAUS]
             + [("twopass", 256, shape, 0, tau) for shape, _, _ in MID for tau in TAUS])
SLAB_SHAPE, SLAB_CUTS, SLAB_LZ = (136, 72, 48), (0, 8, 28, 48), 4
DRIFT_SHAPE = (512, 40, 12)


def _case_id(c):
    algo, nt, shape, lz, tau = c
    return f"{algo}-nt{nt}-{'x'.join(map(str, shape))}-tau{tau[0]:g}_{tau[1]:g}"


# ---- CPU: the premises ---------------------------------------------------------------------------------------------------------
def test_cases_reach_the_large_box_paths():
    """the case table runs every centre-of-mass path that planes of <= 1024 cells and nz <= 128 never reach"""
    shapes = [s for s, _, _ in MID]
    chunks = {s: com_chunks(s) for s in shapes + [SLAB_SHAPE]}
    assert all(len(c) >= 2 for c in chunks.values()), chunks
    assert any(len(c) >= 3 for c in chunks.values())
    assert any(c[-1][1] - c[-1][0] < COM_CHUNK for c in chunks.values()), "a partial last chunk"
    assert any(c0 % s[0] != 0 for s, c in chunks.items() for c0, _ in c[1:]), "a chunk boundary inside a row"
    assert com_chunks((136, 72, 20))[1][0] // 136 == 60
    assert max(fold_ctas(s) for s in shapes) >= 2, "more than one CTA of k_com_fold_chunks"
    assert all(diag_blocks(s) > 256 for s in shapes), [diag_blocks(s) for s in shapes]
    # the brick cases span the reference-state instantiations: both CTA sizes x full / partial tiles x both rates
    fused = [expected_variant("fused", nt, shape, lz, KBT, tau) for algo, nt, shape, lz, tau in MID_CASES if algo == "fused"]
    assert {(v["threads"], v["full"], v["rate1"]) for v in fused} == {(nt, f, r) for nt in (128, 256) for f in (0, 1) for r in (0, 1)}
    assert all(v["noise"] == 1 for v in fused)
    # the 512^3 box: 32 chunks per plane, 4 fold CTAs, ~5e5 k_diag blocks
    assert (len(com_chunks((N, N, N))), fold_ctas((N, N, N)), diag_blocks((N, N, N))) == (32, 4, 524288)


def _small_oracles(oracle_mod, shape, prm):
    f0, g0 = _asymmetric_state(oracle_mod, shape, seed=11)
    eq = profiles_below(f0.sum(axis=0))
    rng = np.random.default_rng(5)
    normals = [rng.standard_normal(shape[::-1] + (33,)) for _ in range(4)]
    A, B = oracle_mod.PortOracle(*shape), oracle_mod.PortOracle(*shape)
    for O in (A, B):
        O.set_params(**prm)
        O.set_equilibrium(*eq)
    return A, B, f0, g0, eq, normals


def _assert_same_bits(A, B, what):
    for a, b in zip(A.populations() + A.noise(), B.populations() + B.noise()):
        assert np.array_equal(a, b), what


def test_oracle_forced_shift_equal_to_computed_one_gives_the_same_bits(oracle_mod):
    """forcing the shift the oracle computes anyway changes no bit of populations and noise; None computes it again"""
    shape = (14, 10, 12)
    A, B, f0, g0, eq, normals = _small_oracles(oracle_mod, shape, _params(KBT, (0.7, 0.55)))
    com_ref = com_of(eq[0])
    s = expected_shift(f0.sum(axis=0), com_ref)
    assert np.all(s != 0), s
    for O in (A, B):
        O.set_normals(normals[0])
    B.set_ref_shift(s)
    A.init_from_populations(f0, g0)
    B.init_from_populations(f0, g0)
    _assert_same_bits(A, B, "after the restart")
    for k in (1, 2):
        # the noise of a step is drawn from its post-step density, which B reaches with the same bits as A: A steps first
        A.set_normals(normals[k])
        A.step(1)
        s = expected_shift(A.hydrovars()[0], com_ref)
        B.set_ref_shift(s)
        B.set_normals(normals[k])
        B.step(1)
        _assert_same_bits(A, B, f"step {k}")
    B.set_ref_shift(None)
    for O in (A, B):
        O.set_normals(normals[3])
        O.step(1)
    _assert_same_bits(A, B, "after set_ref_shift(None)")
    # a wrong forced shift does change the noise
    B.set_ref_shift(s + np.array([1, 0, 0]))
    for O in (A, B):
        O.step(1)
    assert not np.array_equal(A.noise()[0], B.noise()[0])


def test_oracle_forced_zero_shift_on_rolled_profiles_gives_the_same_bits(oracle_mod):
    """shift 0 with the profiles rolled by s reads eq[x - s] at every cell: the bits of the unforced run, whose shift is s"""
    shape = (14, 10, 12)
    A, B, f0, g0, eq, normals = _small_oracles(oracle_mod, shape, _params(KBT, (0.5, 0.5)))
    com_ref = com_of(eq[0])
    B.set_ref_shift((0, 0, 0))

    def roll_for(rho):
        s = expected_shift(rho, com_ref)
        B.set_equilibrium(*(np.roll(a, (s[2], s[1], s[0]), axis=(0, 1, 2)) for a in eq))
        return s

    s = roll_for(f0.sum(axis=0))
    assert np.all(s != 0), s
    for O in (A, B):
        O.set_normals(normals[0])
        O.init_from_populations(f0, g0)
    _assert_same_bits(A, B, "after the restart")
    for k in (1, 2, 3):
        A.set_normals(normals[k])
        A.step(1)
        roll_for(A.hydrovars()[0])  # the shift of the noise drawn at the end of this step
        B.set_normals(normals[k])
        B.step(1)
        _assert_same_bits(A, B, f"step {k}")


# ---- a. mid-size boxes against the oracle -----------------------------------------------------------------------------------
def _ref_lattice(bflbm, algo, shape, prm, eq, lz):
    if algo == "fused":
        return whole_box_ref(bflbm, shape, prm, eq, lz)
    lat = bflbm.Lattice(*shape, params=prm)
    lat.set_reference_state(*eq)  # a whole box: the two-pass kernels
    return lat


def _check_com_buffer(lat, rho_oracle, what):
    """com_buffer against numpy's plane sums of the device's own density (the reduction alone: 1e-13) and of the oracle's (the
    densities themselves differ in the last bits after a step)"""
    got = com_buffer(lat)
    assert_plane_sums(got, plane_sums(lat.hydrovars()[0]), 1e-13, f"{what}, device density")
    assert_plane_sums(got, plane_sums(rho_oracle), 1e-12, f"{what}, oracle density")


@pytest.mark.gpu
@pytest.mark.parametrize("algo,nt,shape,lz,tau", MID_CASES, ids=[_case_id(c) for c in MID_CASES])
def test_large_planes_match_oracle(bflbm, oracle_mod, monkeypatch, algo, nt, shape, lz, tau):
    """3 steps with injected normals: noise, populations, variant, shift and (brick) the per-plane sums after every step"""
    monkeypatch.setenv("BFLBM_CTA_THREADS", str(nt))
    prm = _params(KBT, tau)
    f0, g0 = _asymmetric_state(oracle_mod, shape, seed=sum(shape) + nt)
    eq = profiles_below(f0.sum(axis=0))
    want = expected_variant(algo, nt, shape, lz, KBT, tau)
    brick = algo == "fused"
    with _ref_lattice(bflbm, algo, shape, bflbm.Params(**prm, seed=31, step0=5), eq, lz) as lat:
        lat.init_from_populations(f0, g0)
        com_ref = lat.reference_com()
        O = oracle_mod.PortOracle(*shape)
        O.set_params(**prm)
        O.set_equilibrium(*eq)
        O.set_normals(lat.normals())
        O.init_from_populations(f0, g0)
        shift = lat.reference_shift()
        assert np.array_equal(shift, expected_shift(O.hydrovars()[0], com_ref)) and np.all(shift != 0), shift
        if brick:
            _check_com_buffer(lat, O.hydrovars()[0], "after the restart")
        for s in range(3):
            fn, gn = lat.noise()
            fo, go = O.noise()
            tol = TOL if s == 0 else 10 * TOL
            assert rel_err(fn, fo) <= tol and rel_err(gn, go) <= tol, f"noise amplitudes before step {s + 1}"
            lat.step(1)
            O.set_normals(lat.normals())
            O.step(1)
            _assert_parity(lat, O, tol, f"REF {_case_id((algo, nt, shape, lz, tau))} step {s + 1}", want)
            assert lat.last_step() == (want if s else {**want, "fold_source": 0}), f"step {s + 1}"
            rho = O.hydrovars()[0]
            assert np.array_equal(lat.reference_shift(), expected_shift(rho, com_ref)), f"shift after step {s + 1}"
            if brick:
                _check_com_buffer(lat, rho, f"after step {s + 1}")
        v = lat.last_step()
        if not brick:
            assert v["bx"] * v["by"] * v["bz"] == diag_blocks(shape) > 256


@pytest.mark.gpu
def test_shift_follows_a_drifting_blob_on_wide_planes(bflbm, oracle_mod):
    """a density blob on 512 x 40 x 12 moving with u = (0.04, 0, 0) drifts 1.6 cells in x in 40 steps: the x shift changes, and
    the device's sequence of shifts equals the one the oracle's densities give"""
    shape = DRIFT_SHAPE
    nx, ny, nz = shape
    prm = _params(KBT, (0.5, 0.5))
    _, w, _ = oracle_mod.PortOracle.constants()
    x, y = np.arange(nx, dtype=np.float64), np.arange(ny, dtype=np.float64)
    blob = np.exp(-(x[None, :] - 200.0) ** 2 / (2 * 30.0 ** 2) - (y[:, None] - 17.0) ** 2 / (2 * 8.0 ** 2))
    rho = np.broadcast_to(0.1 + 2.9 * blob, (nz, ny, nx))
    boost = (1 + 3 * (C.T @ np.array([0.04, 0.0, 0.0])))[:, None, None, None]
    f = w[:, None, None, None] * rho[None] * boost
    g = w[:, None, None, None] * (3.1 - rho)[None] * boost
    eq = profiles_below(f.sum(axis=0))
    with whole_box_ref(bflbm, shape, bflbm.Params(**prm, seed=5), eq, 4) as lat:
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
        assert len({s[0] for s in gpu}) >= 2 and all(s[1] != 0 and s[2] != 0 for s in gpu), gpu
        assert lat.last_step()["noise"] == 1 and lat.last_step()["algorithm"] == 0
        assert rel_err(lat.populations()[0], O.populations()[0]) <= 1e-10


# ---- b. slabs with large planes ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("peer,nt", [(False, 256), (True, 128)], ids=["copies-nt256", "peer-nt128"])
def test_slabs_with_large_planes_bitwise_equal_to_whole_box(bflbm, oracle_mod, monkeypatch, peer, nt):
    """3 uneven slabs of 136 x 72 planes (2 chunks each): after every init and step each slab's all-reduced com_buffer is the
    whole box's bit for bit, and so is the shift; populations after 4 steps are the same bits"""
    from bflbm_b200.distributed import EmulatedSlabs
    monkeypatch.setenv("BFLBM_CTA_THREADS", str(nt))
    prm = bflbm.Params(**_params(KBT, (0.7, 0.55)), seed=77)
    f0, g0 = (dyadic(a) for a in _asymmetric_state(oracle_mod, SLAB_SHAPE, seed=17))
    eq = profiles_below(f0.sum(axis=0))
    with whole_box_ref(bflbm, SLAB_SHAPE, prm, eq, SLAB_LZ) as Wb:
        S = EmulatedSlabs(*SLAB_SHAPE, len(SLAB_CUTS) - 1, params=prm, brick_lz=SLAB_LZ, peer=peer, zsplit=SLAB_CUTS)
        try:
            S.set_reference_state(*eq)
            Wb.init_from_populations(f0, g0)
            S.init_from_global_populations(f0, g0)
            for s in range(5):
                sw, cw = Wb.reference_shift(), com_buffer(Wb)
                assert np.all(sw != 0), sw
                assert_plane_sums(cw, plane_sums(Wb.hydrovars()[0]), 1e-13, f"whole box before step {s + 1}")
                for r, lat in enumerate(S.lats):
                    assert np.array_equal(lat.reference_shift(), sw), f"slab {r} shift before step {s + 1}"
                    assert np.array_equal(com_buffer(lat), cw), f"slab {r} com_buffer before step {s + 1}"
                if s == 4:
                    break
                Wb.step(1)
                S.step(1)
            fw, gw = Wb.populations()
            fs, gs = S.gather("populations")
            assert np.array_equal(fw, fs) and np.array_equal(gw, gs)
            assert all(lat.last_step()["noise"] == 1 and lat.last_step()["threads"] == nt for lat in S.lats)
            if peer:
                assert all(lat.halo_error() == 0 for lat in S.lats)
        finally:
            S.close()


# ---- c. the 512^3 box --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_eq(oracle_mod):
    """profiles whose centre of mass lies OFFSET below the tiled state's: the tile's centre of mass + 240 (16 periods of 32)"""
    f0, _ = _tile(oracle_mod)
    target = com_of(f0.sum(axis=0)) + (N - T) / 2 - np.array(OFFSET)
    eq = drop_profiles((N, N, N), target)
    planes = plane_sums(eq[0])
    com = com_of_planes(planes)
    assert np.abs(com - target).max() < 1e-6, (com, target)
    return eq, planes, serial_com(eq[0])


def serial_com(rho):
    """the centre of mass summed cell by cell, x fastest, like bflbm_set_reference_state's host loop (update_com): over 1.3e8
    cells that order is ~5e-11 (relative) away from the pairwise sums of plane_sums, so the host's com_ref is checked against
    this restatement bit for bit.  Premise: the host loop rounds r * i before adding it (no FMA contraction).  That holds for
    the x86-64 build without -march; a host build with FMA in its baseline and contraction on (aarch64, or -march=native
    under GCC's default -ffp-contract=fast) would differ in the last bits with no bug present."""
    x = np.arange(max(rho.shape), dtype=np.float64)
    m = np.cumsum(rho, axis=None)[-1]
    return np.array([np.cumsum(rho * c, axis=None)[-1] / m
                     for c in (x[None, None, :rho.shape[2]], x[None, :rho.shape[1], None], x[:rho.shape[0], None, None])])


def _device_rho(lat):
    """rho of the whole box through the device hydro download (one 1 GiB host array instead of 22)"""
    (h,) = _device_download(lat, "hydrovars", 22, 1)
    rho = h[0].cpu().numpy()
    del h
    _free_device()
    return rho


def _check_big(lat, com_ref, brick, what, relative=True):
    """the device's shift against numpy's from the downloaded rho, and (brick) com_buffer against its plane sums"""
    shift = lat.reference_shift()
    planes = plane_sums(_device_rho(lat))
    want = shift_of_planes(planes, com_ref if relative else None)
    print(f"\n[{what}] shift {tuple(shift)}, numpy {tuple(want)}", flush=True)
    assert np.array_equal(shift, want), f"{what}: device shift {shift}, numpy {want}"
    if brick:
        e = plane_errors(com_buffer(lat), planes)
        print(f"[{what}] com_buffer: largest plane error {e.max():.2e}", flush=True)
        assert e.max() <= 1e-13, f"{what}: com_buffer plane {int(np.argmax(e))} off by {e.max():.3e}"
    return shift


def _window_oracle(oracle_mod, prm, eq, off, shift, nrm, state):
    """64^3 oracle on the window at off: forced shift 0 on profiles cut at off - shift, so that it reads the big box's eq[x - s]"""
    O = oracle_mod.PortOracle(W, W, W)
    O.set_params(**prm)
    O.set_ref_shift((0, 0, 0))
    _window_profiles(O, eq, off, shift)
    O.set_normals(nrm)
    O.init_from_populations(*state)
    return O


def _window_profiles(O, eq, off, shift):
    O.set_equilibrium(*(_cut(a[None], tuple(o - s for o, s in zip(off, shift)), N)[0] for a in eq))


def _report(what, t0, lat_bytes):
    import torch
    print(f"\n[{what}] {time.time() - t0:.1f} s; library device bytes {lat_bytes / 1e9:.2f} GB, torch peak "
          f"{torch.cuda.max_memory_allocated() / 1e9:.2f} GB, peak host RSS "
          f"{resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6:.1f} GB", flush=True)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["fused", "twopass"], ids=["brick-bench", "twopass"])
def test_512cubed_restart_against_numpy_and_window_oracles(bflbm, oracle_mod, monkeypatch, big_eq, algo):
    """512^3 restarted from the tiled state with profiles OFFSET below it: reference_com against numpy, after the restart and
    after each of 2 noisy steps the shift (and on the brick kernel com_buffer) against numpy's from the downloaded density;
    noise before the first step on all cells, populations after 1 and 2 steps at margins 1 and 3 of three 64^3 windows"""
    import torch
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    monkeypatch.setenv("BFLBM_CTA_THREADS", "256")
    eq, eq_planes, eq_serial = big_eq
    brick = algo == "fused"
    prm, seed = _bench_params(KBT)
    f0, g0 = _tile(oracle_mod)
    want = BENCH_VARIANT if brick else expected_variant("twopass", 256, (N, N, N), 0, KBT, (0.5, 0.5))
    with bflbm.Lattice(N, N, N, params=bflbm.Params(**prm, seed=seed)) as lat:
        lat.set_reference_state(*eq)
        if brick:
            lat.set_algorithm("fused")
            lat.set_tiling(LZ)
        com_ref = lat.reference_com()
        assert np.array_equal(com_ref, eq_serial), (com_ref, eq_serial)
        assert rel_err(com_ref, com_of_planes(eq_planes)) <= 1e-10, (com_ref, com_of_planes(eq_planes))
        ft, gt = _tiled(f0, N // T), _tiled(g0, N // T)
        lat.init_from_populations(ft, gt)
        del ft, gt
        s0 = lat.step_count
        shift = _check_big(lat, com_ref, brick, f"{algo} restart")
        assert np.all(shift != 0), shift
        nrm = _window_normals(bflbm, prm, seed, (s0, s0 + 1, s0 + 2))
        oracles = {name: _window_oracle(oracle_mod, prm, eq, off, shift, nrm[name, s0], [_cut(a, off, T) for a in (f0, g0)])
                   for name, off in WINDOWS.items()}
        fn, gn = lat.noise()
        for name, off in WINDOWS.items():
            for s, got, ref in zip("fg", (fn, gn), oracles[name].noise()):
                e = rel_err(_cut(got, off, N), ref)
                print(f"[{algo} restart] noise {s} window {name}: rel err {e:.2e} on all cells", flush=True)
                assert e <= TOL, f"noise {s} before the first step, window {name}: rel err {e:.3e}"
        del fn, gn
        for k, (m, tol) in enumerate(((1, TOL), (3, 10 * TOL)), start=1):
            lat.step(1)
            assert lat.last_step() == (want if k > 1 else {**want, "fold_source": 0}), f"step {k}"
            shift = _check_big(lat, com_ref, brick, f"{algo} step {k}")
            for name, off in WINDOWS.items():
                O = oracles[name]
                _window_profiles(O, eq, off, shift)
                O.set_normals(nrm[name, s0 + k])
                O.step(1)
            _settle(lat)
            _assert_windows(lat, oracles, m, tol, f"{algo} noisy step {k}")
        v = lat.last_step()
        if not brick:
            assert v["bx"] * v["by"] * v["bz"] == diag_blocks((N, N, N))
        _report(f"512^3 restart, {algo}", t0, lat.device_bytes)


@pytest.mark.gpu
def test_512cubed_droplet_init_takes_the_absolute_centre_of_mass(bflbm, big_eq, monkeypatch):
    """init_droplet(0.3) on the bench's brick: the first shift is (int)com (~255 on every axis: about half the cells wrap), the
    one after a step (int)(com - com_ref); both against numpy, com_buffer too"""
    import torch
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    monkeypatch.setenv("BFLBM_CTA_THREADS", "256")
    eq = big_eq[0]
    prm, seed = _params(KBT, (0.5, 0.5)), 2024  # rho_lo = 0.1: with the bench's rho_lo = 0 the droplet's com is 256 - 1e-40
    with bflbm.Lattice(N, N, N, params=bflbm.Params(**prm, seed=seed)) as lat:
        lat.set_reference_state(*eq)
        lat.set_algorithm("fused")
        lat.set_tiling(LZ)
        lat.init_droplet(0.3)
        com_ref = lat.reference_com()
        shift = _check_big(lat, com_ref, True, "droplet init", relative=False)
        assert np.all(shift >= N // 2 - 8), shift
        lat.step(1)
        assert lat.last_step() == {**BENCH_VARIANT, "fold_source": 0}
        shift = _check_big(lat, com_ref, True, "droplet step 1")
        assert np.all(np.abs(shift) < 16), shift
        _report("512^3 droplet init", t0, lat.device_bytes)
