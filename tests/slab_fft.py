"""TEST INFRASTRUCTURE -- the slab-decomposed structure factor of include/bflbm_sf_slab.h, restated in numpy.

Every step of the library's algorithm is written out on plain arrays, so that tests can check it against the whole-box
transform of stats.StructureFactor and against the library's layout:
  kx split (remainder to the low ranks), 2-D r2c per plane, pack into one block per destination, all-to-all of the blocks,
  1-D transform along z on the received [z][ky][kx_local] array, running sums of A_k conj(B_k) / N per pair, and the
  expansion of each rank's half-spectrum columns into the x columns of the shifted full grid it owns.
"""
from __future__ import annotations

import numpy as np


def kx_split(nxh: int, nranks: int):
    """[(kx0, nkx)] per rank: contiguous ranges of [0, nxh), sizes differ by at most one, remainder to the low ranks."""
    if nxh < nranks:
        raise ValueError("nx/2 + 1 < nranks")
    base, rem = divmod(nxh, nranks)
    return [(r * base + min(r, rem), base + (1 if r < rem else 0)) for r in range(nranks)]


def layout(nx: int, ny: int, zsplit, rank: int):
    """(send_counts, send_displs, recv_counts, recv_displs) of `rank` in doubles: bflbm_sf_slab_layout."""
    P = len(zsplit) - 1
    split = kx_split(nx // 2 + 1, P)
    nzl = zsplit[rank + 1] - zsplit[rank]
    nkx = split[rank][1]
    sc = [2 * nzl * ny * n for _, n in split]
    sd = [2 * nzl * ny * k0 for k0, _ in split]
    rc = [2 * (zsplit[s + 1] - zsplit[s]) * ny * nkx for s in range(P)]
    rd = [2 * zsplit[s] * ny * nkx for s in range(P)]
    return sc, sd, rc, rd


def owned_columns(nx: int, kx0: int, nkx: int):
    """Shifted x columns a rank with half-spectrum columns [kx0, kx0 + nkx) writes: x holds kx = x - nx/2 (mod nx), read from
    the half spectrum at kx, or (Hermitian partner) at nx - kx when kx >= nx/2 + 1."""
    nxh = nx // 2 + 1
    out = []
    for x in range(nx):
        kx = (x + nx - nx // 2) % nx
        k = kx if kx < nxh else nx - kx
        if kx0 <= k < kx0 + nkx:
            out.append(x)
    return out


class SlabStructureFactor:
    """Running sums of the slab algorithm, all ranks in one object.  fields: (22, nz, ny, nx) snapshots of the whole box."""

    def __init__(self, shape, zsplit, pairs, var_scaling=None):
        self.nz, self.ny, self.nx = shape
        self.zsplit = list(zsplit)
        self.P = len(zsplit) - 1
        self.pairs = list(pairs)
        self.scale = np.ones(len(pairs)) if var_scaling is None else np.asarray(var_scaling, dtype=float)
        self.vars = []
        for a, b in self.pairs:
            for v in (a, b):
                if v not in self.vars:
                    self.vars.append(v)
        self.nxh = self.nx // 2 + 1
        self.split = kx_split(self.nxh, self.P)
        self.acc = [np.zeros((len(pairs), self.nz, self.ny, n), dtype=complex) for _, n in self.split]
        self.samples = 0

    def rounds(self):
        return len(self.vars)

    def add(self, fields):
        P, ny, nx, nz = self.P, self.ny, self.nx, self.nz
        spec = [dict() for _ in range(P)]
        for v in self.vars:  # one round per distinct variable
            sends = []
            for s in range(P):
                z0, z1 = self.zsplit[s], self.zsplit[s + 1]
                out2d = np.fft.rfft2(fields[v][z0:z1], axes=(1, 2))  # [z][ky][kx], kx < nxh
                send = np.concatenate([out2d[:, :, k0:k0 + n].ravel() for k0, n in self.split])
                sends.append(send)
            for d in range(P):
                _, _, rc, rd = layout(nx, ny, self.zsplit, d)
                parts = []
                for s in range(P):
                    sc, sd, _, _ = layout(nx, ny, self.zsplit, s)
                    blk = sends[s][sd[d] // 2:(sd[d] + sc[d]) // 2]
                    assert blk.size * 2 == rc[s]
                    parts.append(blk)
                recv = np.concatenate(parts)
                assert recv.size * 2 == rd[-1] + rc[-1]
                spec[d][v] = np.fft.fft(recv.reshape(nz, ny, self.split[d][1]), axis=0)
        n = nx * ny * nz
        for d in range(P):
            for p, (a, b) in enumerate(self.pairs):
                self.acc[d][p] += self.scale[p] * spec[d][a] * np.conj(spec[d][b]) / n
        self.samples += 1

    def get(self, zero_avg=True):
        """(re, im), (npairs, nz, ny, nx), assembled from every rank's owned columns; also returns the owner of each column."""
        nz, ny, nx, nxh = self.nz, self.ny, self.nx, self.nxh
        out = np.zeros((len(self.pairs), nz, ny, nx), dtype=complex)
        owner = np.full(nx, -1)
        z = np.arange(nz)
        y = np.arange(ny)
        kz = (z + nz - nz // 2) % nz
        ky = (y + ny - ny // 2) % ny
        for d, (k0, nk) in enumerate(self.split):
            for x in owned_columns(nx, k0, nk):
                assert owner[x] == -1, f"column {x} has two owners"
                owner[x] = d
                kx = (x + nx - nx // 2) % nx
                if kx < nxh:
                    col = self.acc[d][:, kz][:, :, ky][:, :, :, kx - k0]
                else:
                    col = np.conj(self.acc[d][:, (nz - kz) % nz][:, :, (ny - ky) % ny][:, :, :, nx - kx - k0])
                out[:, :, :, x] = col
        if zero_avg:
            out[:, nz // 2, ny // 2, nx // 2] = 0
        out /= self.samples
        return out.real, out.imag, owner


def whole_box_reference(snapshots, pairs, var_scaling=None, zero_avg=True):
    """Complex S of the whole-box transform (AMReX_DFT.H convention), shifted: (npairs, nz, ny, nx)."""
    scale = np.ones(len(pairs)) if var_scaling is None else np.asarray(var_scaling, dtype=float)
    acc = None
    for f in snapshots:
        n = f[0].size
        ft = {c: np.fft.fftn(f[c]) for c in {c for p in pairs for c in p}}
        cur = np.stack([scale[p] * ft[a] * np.conj(ft[b]) / n for p, (a, b) in enumerate(pairs)])
        acc = cur if acc is None else acc + cur
    s = np.fft.fftshift(acc / len(snapshots), axes=(1, 2, 3))
    nz, ny, nx = s.shape[1:]
    if zero_avg:
        s[:, nz // 2, ny // 2, nx // 2] = 0
    return s
