"""CPU tests of the slab-decomposed structure factor (include/bflbm_sf_slab.h): the numpy restatement of its decomposition
(tests/slab_fft.py) equals the whole-box transform of tests/stats.py, and the library exports and binds every symbol."""
import ctypes
import os
import re

import numpy as np
import pytest

import slab_fft
import stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS = [(0, 0), (1, 1), (0, 1), (2, 6), (15, 16), (5, 5)]


def _fields(shape, seed):
    rng = np.random.default_rng(seed)
    f = rng.standard_normal((22,) + shape)
    f[0] += 1.0  # a mean, so that the k = 0 bin matters
    return f


@pytest.mark.parametrize("shape,zsplit", [
    ((8, 6, 10), [0, 8]),                       # P = 1: even nx, ny
    ((7, 5, 9), [0, 3, 7]),                     # P = 2: odd nx, ny, uneven z
    ((9, 6, 12), [0, 2, 5, 9]),                 # P = 3: nxh = 6, odd nx
    ((11, 7, 8), [0, 3, 5, 7, 11]),             # P = 4: nxh = 5 not divisible by 4
    ((13, 6, 9), [0, 2, 4, 6, 9, 13]),          # P = 5: nxh = 7, odd ny
    ((12, 5, 8), [0, 4, 6, 8, 10, 12]),         # P = 5: even nx, nxh = 7
    ((10, 4, 8), [0, 2, 4, 6, 8, 10]),          # P = 5 = nx/2 + 1: one column per rank
])
def test_slab_decomposition_equals_whole_box(shape, zsplit):
    nz, ny, nx = shape
    P = len(zsplit) - 1
    scaling = np.linspace(0.5, 2.0, len(PAIRS))
    dec = slab_fft.SlabStructureFactor(shape, zsplit, PAIRS, var_scaling=scaling)
    ref = stats.StructureFactor(PAIRS)
    snaps = [_fields(shape, s) for s in range(3)]
    for f in snaps:
        dec.add(f)
        ref.add(f)
    assert dec.rounds() == len({c for p in PAIRS for c in p})
    for zero_avg in (True, False):
        got_re, got_im, owner = dec.get(zero_avg=zero_avg)
        # every output column has exactly one owner
        assert (owner >= 0).all() and len(owner) == nx
        want = slab_fft.whole_box_reference(snaps, PAIRS, scaling, zero_avg=zero_avg)
        scale = np.abs(want).max(axis=(1, 2, 3), keepdims=True)
        assert (np.abs(got_re - want.real) / scale).max() <= 1e-12
        assert (np.abs(got_im - want.imag) / scale).max() <= 1e-12
    # stats.StructureFactor (mean removed, k = 0 zeroed, real part) is the same thing unscaled
    got_re, _, _ = dec.get(zero_avg=True)
    want = ref.result() * scaling[:, None, None, None]
    assert (np.abs(got_re - want) / np.abs(want).max(axis=(1, 2, 3), keepdims=True)).max() <= 1e-12
    # the kx split covers the half spectrum in order; the blocks of the layout tile the send and receive buffers
    split = slab_fft.kx_split(nx // 2 + 1, P)
    assert split[0][0] == 0 and sum(n for _, n in split) == nx // 2 + 1
    assert all(split[r][0] + split[r][1] == split[r + 1][0] for r in range(P - 1))
    assert max(n for _, n in split) - min(n for _, n in split) <= 1
    for r in range(P):
        sc, sd, rc, rd = slab_fft.layout(nx, ny, zsplit, r)
        assert sd[0] == 0 and rd[0] == 0
        assert all(sd[i] + sc[i] == sd[i + 1] and rd[i] + rc[i] == rd[i + 1] for i in range(P - 1))
        assert sum(sc) == 2 * (zsplit[r + 1] - zsplit[r]) * ny * (nx // 2 + 1)
        assert sum(rc) == 2 * nz * ny * split[r][1]
        # what rank r sends to d is what d receives from r
        for d in range(P):
            assert sc[d] == slab_fft.layout(nx, ny, zsplit, d)[2][r]


def test_kx_split_needs_a_column_per_rank():
    with pytest.raises(ValueError):
        slab_fft.kx_split(4, 5)
    assert slab_fft.kx_split(5, 5) == [(0, 1), (1, 1), (2, 1), (3, 1), (4, 1)]
    assert slab_fft.kx_split(257, 8)[0] == (0, 33) and slab_fft.kx_split(257, 8)[-1] == (225, 32)


def _slab_header_symbols():
    src = open(os.path.join(ROOT, "include", "bflbm_sf_slab.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bflbm_sf_slab_[a-z0-9_]+)\s*\(", src)))


def test_slab_structure_factor_library_exports_and_binds_its_header(bflbm):
    bflbm.build_sf()
    names = _slab_header_symbols()
    assert len(names) == 13
    ctypes.CDLL(bflbm.LIB, mode=ctypes.RTLD_GLOBAL)
    raw = ctypes.CDLL(bflbm.SF_LIB)
    assert not [n for n in names if not hasattr(raw, n)]
    from bflbm_b200 import structure_factor
    lib = structure_factor._load()
    assert not [n for n in names if getattr(lib, n).argtypes is None]
