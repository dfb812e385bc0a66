"""Structure factors of a box split into z-slabs (include/bflbm_sf_slab.h): slab FFT with one all-to-all per variable.
  * emulated slabs (every slab in this process on one GPU, blocks moved by device copies) against the whole-box accumulator
    bflbm_sf and against the numpy restatements of tests/slab_fft.py;
  * same bits run to run; documented error codes; the device-memory budget at 512^3;
  * real ranks over NCCL (tests/mp_sf_slab_worker.py, skipped with fewer GPUs than ranks)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import slab_fft

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

SHAPE = (20, 11, 24)  # nx, ny (odd), nz
LZ = 4                # brick height: divides every slab below, so the slabs step bit-identically to the whole box
SPLITS = {2: [0, 8, 24], 3: [0, 8, 20, 24], 4: [0, 4, 12, 16, 24]}
PRM = dict(kBT=1e-5, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0, tau_f=0.7, tau_g=0.55, seed=21)
ERR_ARG, ERR_STATE = -1, -3


def _scaling(bflbm):
    return np.linspace(0.5, 2.0, len(bflbm.REFERENCE_PAIRS))


def _emulated_run(bflbm, nslabs, snapshots=None):
    """4 samples of the emulated slabs; returns {zero_avg: (re, im)} and the accumulator's samples before / after reset."""
    from bflbm_b200.distributed import EmulatedSlabs
    S = EmulatedSlabs(*SHAPE, nslabs, params=bflbm.Params(**PRM), brick_lz=LZ, zsplit=SPLITS[nslabs])
    try:
        S.init_droplet(0.3)
        with bflbm.SlabStructureFactor(S, bflbm.REFERENCE_PAIRS, _scaling(bflbm)) as sf:
            assert sf.rounds == len({c for p in bflbm.REFERENCE_PAIRS for c in p})
            nx, ny = SHAPE[0], SHAPE[1]
            for r in range(nslabs):
                assert sf.kx_range(r) == slab_fft.kx_split(nx // 2 + 1, nslabs)[r]
                assert tuple(sf.layout[r]) == slab_fft.layout(nx, ny, SPLITS[nslabs], r)
            for _ in range(4):
                S.step(3)
                sf.fort_structure()
                if snapshots is not None:
                    snapshots.append(S.gather("hydrovars"))
            out = {za: sf.result(zero_avg=za, imag=True) for za in (True, False)}
            samples = sf.samples
            sf.reset()
            return out, samples, sf.samples
    finally:
        S.close()


@pytest.mark.parametrize("nslabs", [2, 3, 4])
def test_emulated_slabs_equal_the_whole_box_accumulator(bflbm, nslabs):
    bflbm.build_sf()
    pairs = bflbm.REFERENCE_PAIRS
    whole_snaps = []
    with bflbm.Lattice(*SHAPE, params=bflbm.Params(**PRM)) as W:
        W.set_tiling(LZ)
        W.init_droplet(0.3)
        with bflbm.StructureFactor(W, pairs, _scaling(bflbm)) as sw:
            for _ in range(4):
                W.step(3)
                sw.fort_structure()
                whole_snaps.append(W.hydrovars())
            want = {za: sw.result(zero_avg=za, imag=True) for za in (True, False)}
    snaps = []
    got, samples, after_reset = _emulated_run(bflbm, nslabs, snaps)
    assert samples == 4 and after_reset == 0
    assert all(np.array_equal(a, b) for a, b in zip(snaps, whole_snaps)), "slabs must see the whole box's fields"
    for za in (True, False):
        (gr, gi), (wr, wi) = got[za], want[za]
        scale = np.abs(wr + 1j * wi).max(axis=(1, 2, 3), keepdims=True)
        assert (np.abs(gr - wr) / scale).max() <= 1e-12
        assert (np.abs(gi - wi) / scale).max() <= 1e-12
        ref = slab_fft.whole_box_reference(snaps, pairs, _scaling(bflbm), zero_avg=za)
        assert (np.abs(gr - ref.real) / scale).max() <= 1e-11
        assert (np.abs(gi - ref.imag) / scale).max() <= 1e-11
        for p, (a, b) in enumerate(pairs):
            if a == b:
                assert np.abs(gi[p]).max() <= 1e-12 * scale[p].max()
    nz, ny, nx = SHAPE[2], SHAPE[1], SHAPE[0]
    assert (got[True][0][:, nz // 2, ny // 2, nx // 2] == 0).all()


def test_emulated_slabs_same_bits_run_to_run(bflbm):
    bflbm.build_sf()
    a, _, _ = _emulated_run(bflbm, 3)
    b, _, _ = _emulated_run(bflbm, 3)
    for za in (True, False):
        assert np.array_equal(a[za][0], b[za][0]) and np.array_equal(a[za][1], b[za][1])


def test_slab_structure_factor_error_codes(bflbm):
    from bflbm_b200 import structure_factor
    from bflbm_b200.distributed import EmulatedSlabs
    bflbm.build_sf()
    lib = structure_factor._load()
    pa = np.zeros(1, dtype=np.int32)

    def create(lat, nranks, rank, zsplit, pairs=pa):
        z = np.ascontiguousarray(zsplit, dtype=np.int32)
        h = ctypes.c_void_p()
        rc = lib.bflbm_sf_slab_create(lat.h, nranks, rank, z.ctypes.data, len(pairs), pairs.ctypes.data, pairs.ctypes.data, None,
                                      ctypes.byref(h))
        if rc == 0:
            lib.bflbm_sf_slab_destroy(h)
        return rc

    prm = bflbm.Params(**PRM)
    with bflbm.Lattice(16, 9, 24, params=prm, slab=(0, 8)) as lat:
        assert create(lat, 3, 0, [0, 8, 16, 24]) == 0
        assert create(lat, 2, 0, [0, 12, 24]) == ERR_ARG      # zsplit does not match the lattice's planes
        assert create(lat, 3, 1, [0, 8, 16, 24]) == ERR_ARG   # another rank's planes
        assert create(lat, 3, 0, [0, 8, 16, 20]) == ERR_ARG   # does not end at nz
        assert create(lat, 3, 0, [0, 8, 16, 24], np.array([22], dtype=np.int32)) == ERR_ARG  # pair index outside hydrovs
    with bflbm.Lattice(6, 9, 10, params=prm, slab=(0, 2)) as lat:
        assert create(lat, 5, 0, [0, 2, 4, 6, 8, 10]) == ERR_ARG  # nx/2 + 1 = 4 < 5 ranks
    S = EmulatedSlabs(*SHAPE, 2, params=prm, brick_lz=LZ, zsplit=SPLITS[2])
    try:
        S.init_droplet(0.3)
        with bflbm.SlabStructureFactor(S, [(0, 0), (1, 1)]) as sf:
            h = sf.h[0]
            out = np.zeros((2,) + SHAPE[::-1])
            assert lib.bflbm_sf_slab_get(h, 1, out.ctypes.data, None) == ERR_STATE  # no samples yet
            assert lib.bflbm_sf_slab_end(h, 0) == ERR_STATE                         # end before begin
            assert lib.bflbm_sf_slab_begin(h, 1) == ERR_STATE                       # rounds out of order
            assert lib.bflbm_sf_slab_begin(h, 2) == ERR_ARG                         # no such round
            with pytest.raises(bflbm.BflbmError) as e:
                sf.result()
            assert e.value.code == ERR_STATE
            sf.fort_structure()  # the accumulator is still usable after refused calls
            assert sf.samples == 1
    finally:
        S.close()


def test_slab_structure_factor_memory_budget_512cubed(bflbm):
    """The accumulator must fit beside a 512^3 lattice: <= 560 B per local cell for create + one accumulate, cuFFT work area
    included, measured after the lattice's own observer staging exists."""
    import torch
    from bflbm_b200 import structure_factor
    bflbm.build_sf()
    lib = structure_factor._load()
    n = 512
    pairs = bflbm.REFERENCE_PAIRS
    with bflbm.Lattice(n, n, n, params=bflbm.Params(kBT=1e-5, alpha0=0.0, seed=3)) as lat:
        lat.init_mixture()
        tmp = torch.empty(22 * n ** 3, dtype=torch.float64, device="cuda")
        assert lat.lib.bflbm_get_hydrovars_device(lat.h, ctypes.c_void_p(tmp.data_ptr())) == 0
        del tmp
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free0, _ = torch.cuda.mem_get_info()
        a = np.ascontiguousarray([p[0] for p in pairs], dtype=np.int32)
        b = np.ascontiguousarray([p[1] for p in pairs], dtype=np.int32)
        z = np.array([0, n], dtype=np.int32)
        h = ctypes.c_void_p()
        assert lib.bflbm_sf_slab_create(lat.h, 1, 0, z.ctypes.data, len(pairs), a.ctypes.data, b.ctypes.data, None, ctypes.byref(h)) == 0
        try:
            from bflbm_b200.distributed import _device_tensor
            cnt = (ctypes.c_size_t * 1)()
            assert lib.bflbm_sf_slab_layout(h, 0, cnt, None, None, None) == 0
            send = _device_tensor(lib.bflbm_sf_slab_send_buffer(h), cnt[0], torch.device("cuda", 0))
            recv = _device_tensor(lib.bflbm_sf_slab_recv_buffer(h), cnt[0], torch.device("cuda", 0))
            for v in range(lib.bflbm_sf_slab_rounds(h)):
                assert lib.bflbm_sf_slab_begin(h, v) == 0
                torch.cuda.synchronize()
                recv.copy_(send)
                torch.cuda.synchronize()
                assert lib.bflbm_sf_slab_end(h, v) == 0
            torch.cuda.synchronize()
            assert lib.bflbm_sf_slab_samples(h) == 1
            used = free0 - torch.cuda.mem_get_info()[0]
            print(f"slab structure factor at 512^3, 22 pairs: {used / n ** 3:.1f} B per cell")
            assert used <= 560 * n ** 3, f"{used / n ** 3:.1f} B per cell"
        finally:
            lib.bflbm_sf_slab_destroy(h)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_slab_structure_factor_over_processes_equals_whole_box(world):
    import torch
    if (torch.cuda.device_count() if torch.cuda.is_available() else 0) < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29700 + world), os.path.join(HERE, "mp_sf_slab_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and f"MP_SF_SLAB_OK {world}" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
