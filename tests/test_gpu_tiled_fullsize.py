"""The 512^3 step, and every chunked transfer around it, against the oracle through periodic tiling.

The oracle is too slow for the 512^3 box that bench.py times, but that box can be checked against a small one:

* A deterministic step (kBT = 0) has no position-dependent input, so a state that is periodic with period 32^3 stays periodic.
  A 32^3 "twin" lattice stepped with the same kernel, the same switches and a brick of the same shape puts every cell at
  the same place in its brick as the big box does, so every one of the 4096 periods of the big box must equal the twin bit
  for bit after any number of steps, while the twin itself is checked against the oracle.  The comparison goes through
  every chunked download (each moves at most 1 GiB per chunk, so at 512^3 they run 10 to 40 chunks) and, on slabs, through
  the chunked upload of whole-box host arrays.
* With noise the normals are keyed by global cell and the state stops being periodic.  After one step the populations of a
  cell depend on the state and the normals of its neighbours only, and every step widens that by the two-cell reach of the
  density gradients.  A 64^3 oracle window cut out of the periodic state, with the big box's normals of its cells injected,
  must therefore give the big box's populations on every window cell at least 1 from the window's faces after one noisy
  step and at least 3 after two; the CPU tests below show that these margins are tight.

The tile is a droplet times (1 + 1e-3 u) (no mirror symmetry) rounded to multiples of 2^-24, so that the densities a restart
builds as (local part + neighbour part) on slab-face planes are exact sums wherever the box is cut.
"""
import importlib.util
import os
import time

import numpy as np
import pytest

from conftest import assert_hydro_close, rel_err
from test_gpu_kernel_variants import _asymmetric_state, _assert_parity, ceil_div, expected_variant
from test_gpu_reference_state import dyadic

HERE = os.path.dirname(os.path.abspath(__file__))
N, T = 512, 32          # the bench's box per GPU and the period of the tiled state (one brick in x and z)
LZ = 32                 # the brick height the bench's box gets automatically
NVEL, PLANE = 19, N * N
TOL = 1e-12
KBT = 1e-5

# what the bench's step launches at 512^3 (bflbm_debug_last_step)
BENCH_VARIANT = dict(algorithm=0, threads=256, tile_x=32, tile_y=8, lz=32, bx=16, by=64, bz=16, full=1, rate1=1, noise=1,
                     fold_source=1, schedule=0, graph=0)

# ---- restatement of the transfer chunking (capi.cu) ------------------------------------------------------------------------
STAGE_DOUBLES = 128 << 20  # chunk_planes / upload_populations: a staged chunk holds at most 1 GiB


def chunk_planes(ncomp, nzl=N):
    return max(1, min(nzl, STAGE_DOUBLES // (ncomp * PLANE)))


def download_chunks(ncomp, nzl=N):
    """chunks of an observer download of ncomp components (observe / observe_pair / bflbm_get_populations_device); also the
    chunks of the whole-box population upload (ncomp = 38)"""
    return ceil_div(nzl, chunk_planes(ncomp, nzl))


def global_upload_chunks(z0, nzl):
    """chunks of bflbm_init_from_global_populations on a slab (upload_populations mode 2): the source planes z0 - 1 .. z0 + nzl,
    the lower ghost plane a chunk of its own, and no chunk crosses the periodic wrap of the host array"""
    nsrc = nzl + 2
    cp = max(1, min(nsrc, STAGE_DOUBLES // (2 * NVEL * PLANE)))
    z = n = 0
    while z < nsrc:
        zc = 1 if z == 0 else min(cp, nsrc - z, N - (z0 - 1 + z) % N)
        z += zc
        n += 1
    return n


# ---- cases -------------------------------------------------------------------------------------------------------------------
A_CASES = [  # (id, algorithm, threads per CTA, (tau_f, tau_g))
    ("bench-kernel", "fused", 256, (0.5, 0.5)),
    ("general-rates", "fused", 256, (0.7, 0.55)),
    ("nt128", "fused", 128, (0.5, 0.5)),
    ("twopass", "twopass", 256, (0.5, 0.5)),
]
B_CASES = [((0, 192, 512), False), ((0, 160, 352, 512), True)]  # (z cuts, peer stores)
WINDOWS = {  # 64^3 windows at (x, y, z) offsets that are no multiple of the 32 x 8 x 32 brick
    "origin": (499, 507, 505),          # contains x = 0, y = 0 and z = 0
    "interior": (203, 157, 229),        # crosses interior brick faces in x, y and z
    "last-bricks": (461, 459, 455),     # covers the last brick in x and y and the last brick row in z
}
W = 64


def _bench_params(kbt, tau=(0.5, 0.5)):
    """bench.py's PARAMS (without the seed) at the given kBT and relaxation times"""
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(HERE), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    prm = dict(bench.PARAMS, kBT=kbt, tau_f=tau[0], tau_g=tau[1])
    return {k: v for k, v in prm.items() if k != "seed"}, bench.PARAMS["seed"]


def _tile(oracle_mod):
    return tuple(dyadic(a) for a in _asymmetric_state(oracle_mod, (T, T, T), seed=2048))


def _tiled(a, reps):
    return np.tile(a, (1, reps, reps, reps))


def _window(offset, period, n=W):
    """open-mesh (z, y, x) indices of the n^3 window at (x, y, z) offset of a periodic box of the given period"""
    ox, oy, oz = offset
    return np.ix_(*((o + np.arange(n)) % period for o in (oz, oy, ox)))


def _cut(a, offset, period, n=W):
    """the (c, n, n, n) window of a (c, period, period, period) array"""
    return a[(slice(None),) + _window(offset, period, n)]


def _inner(a, m):
    """cells at least m from the faces of a (c, n, n, n) window"""
    return a[:, m:a.shape[1] - m, m:a.shape[2] - m, m:a.shape[3] - m]


def _configure(lat, algo):
    lat.set_algorithm(algo)
    if algo == "fused":
        lat.set_tiling(LZ)


# ---- CPU: the premises, on the oracle ---------------------------------------------------------------------------------------
def test_chunk_counts_at_512cubed():
    """the restated chunking gives the transfer table of the 512^3 box: (planes per chunk, chunks, planes of the last chunk)"""
    table = {38: (13, 40, 5), 22: (23, 23, 6), 9: (56, 10, 8), 33: (15, 35, 2)}
    for ncomp, want in table.items():
        cp, n = chunk_planes(ncomp), download_chunks(ncomp)
        assert (cp, n, N - (n - 1) * cp) == want, ncomp
    # slab uploads of the two slab cases: one chunk for the lower ghost plane, one more where the upper ghost plane wraps to 0
    got = {(z0, z1 - z0): global_upload_chunks(z0, z1 - z0) for cuts, _ in B_CASES for z0, z1 in zip(cuts, cuts[1:])}
    assert got == {(0, 192): 16, (192, 320): 27, (0, 160): 14, (160, 192): 16, (352, 160): 15}


def test_twins_share_the_brick_of_the_big_box():
    """the bench's automatic choice at 512^3 is the variant declared above, and each 32^3 twin gets the tile, brick height,
    fold source and kernel of its 512^3 box"""
    assert expected_variant("fused", 256, (N, N, N), 0, KBT, (0.5, 0.5)) == BENCH_VARIANT
    for _, algo, nt, tau in A_CASES:
        # the two-pass kernels are thread-per-cell: their launch block (32 x 8 on the twin, 128 x 2 at 512^3) cannot matter
        same = ("algorithm", "rate1", "noise") + (("threads", "tile_x", "tile_y", "lz", "full", "fold_source") if algo == "fused" else ())
        lz = LZ if algo == "fused" else 0
        big, twin = (expected_variant(algo, nt, (n, n, n), lz, 0.0, tau) for n in (N, T))
        assert {k: big[k] for k in same} == {k: twin[k] for k in same}, (algo, nt, tau)
        assert big["fold_source"] == int(algo == "fused")


def test_tiled_oracle_is_the_tile_repeated(oracle_mod):
    """a 32^3 tile repeated 2 x 2 x 2: after 5 deterministic steps the 64^3 oracle holds the tile's own result, repeated"""
    prm, _ = _bench_params(0.0)
    f0, g0 = _tile(oracle_mod)
    small, big = oracle_mod.PortOracle(T, T, T), oracle_mod.PortOracle(2 * T, 2 * T, 2 * T)
    for O, reps in ((small, 1), (big, 2)):
        O.set_params(**prm)
        O.init_from_populations(_tiled(f0, reps), _tiled(g0, reps))
        O.step(5)
    for a, b in zip(big.populations() + (big.hydrovars(),), small.populations() + (small.hydrovars(),)):
        assert np.array_equal(a, _tiled(b, 2))


def test_window_oracle_matches_inside_tight_margins(oracle_mod):
    """a 96^3 oracle started from the tile repeated 3 x 3 x 3 with seeded random normals, and a 32^3 oracle on a window of it
    (offset not a multiple of the tile, wrapping around the box) with the same normals: equal on cells at least 1 from the
    window's faces after one step (populations, noise) and at least 3 after two; hydro fields at least 2 after one.  One
    cell less and they differ."""
    prm, _ = _bench_params(KBT)
    n, w, off = 3 * T, T, (77, 41, 83)
    f0, g0 = _tile(oracle_mod)
    rng = np.random.default_rng(96)
    normals = [rng.standard_normal((n, n, n, 33)) for _ in range(3)]
    win_normals = [a[_window(off, n, w)] for a in normals]
    big, win = oracle_mod.PortOracle(n, n, n), oracle_mod.PortOracle(w, w, w)
    for O, state, nrm in ((big, [_tiled(a, 3) for a in (f0, g0)], normals), (win, [_cut(a, off, T, w) for a in (f0, g0)], win_normals)):
        O.set_params(**prm)
        O.set_normals(nrm[0])
        O.init_from_populations(*state)
    views = {}
    for s in (1, 2):
        for O, nrm in ((big, normals), (win, win_normals)):
            O.set_normals(nrm[s])
            O.step(1)
        views[s] = {"populations": [(_cut(a, off, n, w), b) for a, b in zip(big.populations(), win.populations())],
                    "noise": [(_cut(a, off, n, w), b) for a, b in zip(big.noise(), win.noise())],
                    "hydrovars": [(_cut(big.hydrovars(), off, n, w), win.hydrovars())]}

    def equal_at(pairs, m):
        return all(np.array_equal(_inner(a, m), _inner(b, m)) for a, b in pairs)

    for s, what, m in ((1, "populations", 1), (1, "noise", 1), (1, "hydrovars", 2), (2, "populations", 3)):
        assert equal_at(views[s][what], m), f"{what} after {s} step(s) differ at margin {m}"
        assert not equal_at(views[s][what], m - 1), f"{what} after {s} step(s) already agree at margin {m - 1}"


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------------
def _run_twin(bflbm, oracle_mod, algo, tau, long=True):
    """the 32^3 twin from the tile: 1 step, checked against the oracle like the variant matrix (1e-12 on the populations), then
    70 more replayed from 64 + 4 + 2-step graphs (the 22 fields within 1e-10 of the oracle).  Returns the populations after
    the first step and (populations, hydrovars, hydrovars_bar) after the last."""
    prm, seed = _bench_params(0.0, tau)
    nt = int(os.environ.get("BFLBM_CTA_THREADS", "256"))
    want = expected_variant(algo, nt, (T, T, T), LZ if algo == "fused" else 0, 0.0, tau)
    f0, g0 = _tile(oracle_mod)
    with bflbm.Lattice(T, T, T, params=bflbm.Params(**prm, seed=seed)) as tw:
        _configure(tw, algo)
        tw.init_from_populations(f0, g0)
        O = oracle_mod.PortOracle(T, T, T)
        O.set_params(**prm)
        O.init_from_populations(f0, g0)
        tw.step(1)
        O.step(1)
        _assert_parity(tw, O, TOL, f"{algo} twin, tau {tau}, step 1", want)
        first = tw.populations()
        if not long:
            return first, None
        tw.step(70)
        O.step(70)
        assert_hydro_close(tw.hydrovars(), O.hydrovars(), 1e-10, f"{algo} twin, tau {tau}, step 71")
        assert tw.last_step() == {**want, "graph": 1}
        return first, tw.populations() + (tw.hydrovars(), tw.hydrovars_bar())


def _periodic_mismatch(big, tile):
    """None if every 32^3 period of big (c, N, N, N; host array or device tensor) equals the twin's (c, 32, 32, 32) bit for bit,
    else where the first difference is"""
    r = N // T
    dev = not isinstance(big, np.ndarray)
    if dev:
        import torch
        tile = torch.from_numpy(np.ascontiguousarray(tile)).to(big.device)
    for c in range(big.shape[0]):
        v = big[c].reshape(r, T, r, T, r, T)
        t = tile[c].reshape(1, T, 1, T, 1, T)
        bad = v != t
        if bool(bad.any()):
            if dev:
                bad, v, t = bad.cpu().numpy(), v.cpu().numpy(), t.cpu().numpy()
            i = np.unravel_index(int(np.argmax(bad)), bad.shape)
            periods = int(np.count_nonzero(bad.any(axis=(1, 3, 5))))
            return (f"component {c} differs from the twin in {periods} of {r ** 3} periods; first at (x, y, z) = "
                    f"({i[4] * T + i[5]}, {i[2] * T + i[3]}, {i[0] * T + i[1]}), ({i[5]}, {i[3]}, {i[1]}) in its period: "
                    f"{v[i]:.17g} vs {t[0, i[1], 0, i[3], 0, i[5]]:.17g}")
    return None


def _download_mismatch(get, lats, chunks, tiles):
    """downloads through get() and returns what differs: the observer launches of each lattice against its chunk count, then
    every array period by period against the twin's; None if nothing does"""
    n0 = [lat.kernel_launches for lat in lats]
    outs = get()
    n = [lat.kernel_launches - a for lat, a in zip(lats, n0)]
    if n != list(chunks):
        return f"{n} observer launches, expected one per chunk: {list(chunks)}"
    for i, (o, t) in enumerate(zip(outs, tiles)):
        m = _periodic_mismatch(o, t)
        if m:
            return f"array {i}: {m}"
    return None


def _free_device():
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _assert_download_periodic(get, lats, chunks, tiles, what):
    """_download_mismatch, asserted once the downloaded arrays (10 to 41 GB) are gone, so that a failure keeps none alive"""
    msg = _download_mismatch(get, lats, chunks, tiles)
    _free_device()
    assert msg is None, f"{what}: {msg}"


def _device_download(lat, name, ncomp_each, nout):
    """bflbm_get_<name>_device into torch tensors of (ncomp_each, nz, ny, nx)"""
    import torch
    from bflbm_b200.lattice import _check
    outs = [torch.empty((ncomp_each,) + lat.shape, dtype=torch.float64, device=torch.device("cuda", lat.device)) for _ in range(nout)]
    _check(getattr(lat.lib, f"bflbm_get_{name}_device")(lat.h, *(o.data_ptr() for o in outs)))
    return outs


def _counted(lat, fn, *a):
    n0 = lat.kernel_launches
    out = fn(*a)
    return out, lat.kernel_launches - n0


def _settle(lat):
    """complete the densities R the way the first observer after a step would (ensure_full_R, here inside total_mass), so that
    every download below launches exactly one observer per chunk and nothing else"""
    lat.total_mass()


def _report(what, t0, lat_bytes):
    import torch
    print(f"\n[{what}] {time.time() - t0:.1f} s; library device bytes {lat_bytes / 1e9:.2f} GB, torch peak "
          f"{torch.cuda.max_memory_allocated() / 1e9:.2f} GB", flush=True)


# ---- A. deterministic, whole box ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,algo,nt,tau", A_CASES, ids=[c[0] for c in A_CASES])
def test_whole_box_periods_equal_the_twin(bflbm, oracle_mod, monkeypatch, name, algo, nt, tau):
    """512^3 from the tile repeated 16 x 16 x 16, 1 step then 70 replayed from graphs: every period equals the 32^3 twin bit for
    bit (the bench's kernel after both, the others after the last), read through the device population download; for the bench's
    kernel also through every other chunked download of the deterministic state, each with its chunk count."""
    import torch
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    monkeypatch.setenv("BFLBM_CTA_THREADS", str(nt))
    first, last = _run_twin(bflbm, oracle_mod, algo, tau)
    prm, seed = _bench_params(0.0, tau)
    want = expected_variant(algo, nt, (N, N, N), LZ if algo == "fused" else 0, 0.0, tau)
    bench = name == "bench-kernel"
    if bench:
        assert want == {**BENCH_VARIANT, "noise": 0}
    f0, g0 = _tile(oracle_mod)
    with bflbm.Lattice(N, N, N, params=bflbm.Params(**prm, seed=seed)) as lat:
        _configure(lat, algo)
        ft, gt = _tiled(f0, N // T), _tiled(g0, N // T)
        _, n = _counted(lat, lat.init_from_populations, ft, gt)
        del ft, gt
        assert n == download_chunks(2 * NVEL) + 3, "upload chunks + density partials, halo pack and unpack of the restart"
        lat.step(1)
        assert lat.last_step() == {**want, "fold_source": 0}  # the first step after an upload stages every plane from R
        pop_chunks = download_chunks(2 * NVEL)
        if bench:
            _settle(lat)
            _assert_download_periodic(lambda: _device_download(lat, "populations", NVEL, 2), [lat], [pop_chunks], first,
                                      f"{name} step 1, device populations")
        lat.step(70)
        assert lat.last_step() == {**want, "graph": 1}
        _settle(lat)
        downloads = [(lambda: _device_download(lat, "populations", NVEL, 2), pop_chunks, last[:2], "device populations")]
        if bench:
            downloads += [(lambda: _device_download(lat, "hydrovars", 22, 1), download_chunks(22), last[2:3], "device hydrovars"),
                          (lat.populations, pop_chunks, last[:2], "populations()"),
                          (lambda: (lat.hydrovars(),), download_chunks(22), last[2:3], "hydrovars()"),
                          (lambda: (lat.hydrovars_bar(),), download_chunks(9), last[3:4], "hydrovars_bar()")]
        for get, chunks, tiles, what in downloads:
            _assert_download_periodic(get, [lat], [chunks], tiles, f"{name} step 71, {what}")
        assert lat.step_count == 71
        _report(name, t0, lat.device_bytes)


# ---- B. slabs on one GPU --------------------------------------------------------------------------------------------------
def _init_slabs_from_global(S, f, g):
    """bflbm_init_from_global_populations on every slab (the chunked upload of whole-box host arrays; in peer mode it also runs
    the first half of the halo refresh), then the rest of the halo refresh.  Returns each slab's kernel launches of the upload."""
    from bflbm_b200.lattice import _check
    counts = [_counted(lat, lat.init_from_global_populations, f, g)[1] for lat in S.lats]
    if not S.peer:
        for lat in S.lats:
            _check(lat.lib.bflbm_halo_refresh_begin(lat.h))
        S._exchange()
    for lat in S.lats:
        _check(lat.lib.bflbm_halo_refresh_end(lat.h))
    return counts


def _into_global(S, name, ncomp_each, nout):
    """bflbm_get_<name>_into_global of every slab into whole-box host arrays (ncomp_each, N, N, N)"""
    from bflbm_b200.lattice import _check
    outs = [np.empty((ncomp_each, N, N, N)) for _ in range(nout)]
    for lat in S.lats:
        _check(getattr(lat.lib, f"bflbm_get_{name}_into_global")(lat.h, *(o.ctypes.data for o in outs)))
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize("cuts,peer", B_CASES, ids=["2slabs-copies", "3slabs-peer"])
def test_slabs_periods_equal_the_twin(bflbm, oracle_mod, monkeypatch, cuts, peer):
    """512^3 in emulated z-slabs cut at multiples of the brick height, restarted from the tiled whole-box arrays, 1 + 70 steps,
    read back into whole-box arrays: every period equals the bench kernel's twin bit for bit"""
    import torch
    from bflbm_b200.distributed import EmulatedSlabs
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    monkeypatch.setenv("BFLBM_CTA_THREADS", "256")
    _, last = _run_twin(bflbm, oracle_mod, "fused", (0.5, 0.5))
    prm, seed = _bench_params(0.0)
    f0, g0 = _tile(oracle_mod)
    S = EmulatedSlabs(N, N, N, len(cuts) - 1, params=bflbm.Params(**prm, seed=seed), brick_lz=LZ, peer=peer, zsplit=cuts)
    try:
        ft, gt = _tiled(f0, N // T), _tiled(g0, N // T)
        counts = _init_slabs_from_global(S, ft, gt)
        del ft, gt
        assert counts == [global_upload_chunks(z0, nzl) + (2 if peer else 0) for z0, nzl in S.bounds]
        S.step(1)
        S.step(70)
        for lat, (_, nzl) in zip(S.lats, S.bounds):
            assert lat.last_step() == expected_variant("fused", 256, (N, N, nzl), LZ, 0.0, (0.5, 0.5), schedule=2)
            _settle(lat)
        for name, ncomp, nout, tiles in (("populations", NVEL, 2, last[:2]), ("hydrovars", 22, 1, last[2:3])):
            _assert_download_periodic(lambda: _into_global(S, name, ncomp, nout), S.lats,
                                      [download_chunks(nout * ncomp, nzl) for _, nzl in S.bounds], tiles, f"slabs {cuts}, {name}")
        assert all(lat.halo_error() == 0 for lat in S.lats)
        assert all(lat.step_count == 71 for lat in S.lats)
        _report(f"slabs {cuts}{' peer' if peer else ''}", t0, sum(lat.device_bytes for lat in S.lats))
    finally:
        S.close()


# ---- C. the fluctuating bench kernel --------------------------------------------------------------------------------------
def _z_runs(oz, n=W):
    """the planes oz .. oz + n - 1 (mod N) as contiguous (z0, nz) runs"""
    first = min(n, N - oz)
    return [(oz, first)] + ([(0, n - first)] if first < n else [])


def _slab_normals(bflbm, prm, seed, z0, nz, steps, pick=lambda a: a):
    """{step: pick(normals)} of the global planes z0 .. z0 + nz - 1 at each step, from a thin slab lattice (slabs and the whole
    box key the normals by global cell and step alike; a whole-box normals() download holds 35 GB)"""
    out = {}
    with bflbm.Lattice(N, N, N, params=bflbm.Params(**prm, seed=seed), slab=(z0, nz)) as s:
        for k in steps:
            s.set_params(step0=k)
            s.init_mixture()  # an init sets the step counter to step0
            out[k] = pick(s.normals())
    return out


def _window_normals(bflbm, prm, seed, steps):
    """{(window, step): (64, 64, 64, 33)} normals of each window's cells"""
    out = {}
    for name, (ox, oy, oz) in WINDOWS.items():
        yi, xi = ((o + np.arange(W)) % N for o in (oy, ox))
        runs = [_slab_normals(bflbm, prm, seed, z0, nz, steps, lambda a: a[:, yi[:, None], xi[None, :]]) for z0, nz in _z_runs(oz)]
        for k in steps:
            out[name, k] = np.concatenate([r[k] for r in runs], axis=0)
    return out


def _window_errors(lat, oracles, m):
    """(launches of the device population download, {(window, species): rel err of the big box's populations against the
    window's oracle on the cells at least m from the window's faces}); gathered on the device"""
    import torch
    (f, g), n = _counted(lat, _device_download, lat, "populations", NVEL, 2)
    errs = {}
    for name, off in WINDOWS.items():
        idx = (slice(None),) + tuple(torch.as_tensor(i, device=f.device) for i in _window(off, N))
        for s, got, want in zip("fg", (f, g), oracles[name].populations()):
            errs[name, s] = rel_err(_inner(got[idx].cpu().numpy(), m), _inner(want, m))
    return n, errs


def _assert_windows(lat, oracles, m, tol, what):
    n, errs = _window_errors(lat, oracles, m)
    _free_device()
    print(f"\n[{what}] populations rel err on cells >= {m} from the window faces: "
          + ", ".join(f"{w} {s} {e:.2e}" for (w, s), e in errs.items()), flush=True)
    assert n == download_chunks(2 * NVEL)
    bad = {k: e for k, e in errs.items() if e > tol}
    assert not bad, f"{what}: rel err above {tol:.0e} on cells >= {m} from the window faces: {bad}"


def _host_downloads_mismatch(lat, oracles, normals, z_tail, tail):
    """after the first noisy step: hydrovars() on the windows at margin 2, noise() at margin 1, the whole-box normals() on the
    windows and in its last two chunks, each download with its chunk count; returns the first failure, or None"""
    h, n = _counted(lat, lat.hydrovars)
    if n != download_chunks(22):
        return f"hydrovars(): {n} observer launches"
    for name, off in WINDOWS.items():
        try:
            assert_hydro_close(_inner(_cut(h, off, N), 2), _inner(oracles[name].hydrovars(), 2), 100 * TOL, f"hydrovars(), window {name}")
        except AssertionError as e:
            return str(e)
    del h
    (fn, gn), n = _counted(lat, lat.noise)
    if n != download_chunks(2 * NVEL):
        return f"noise(): {n} observer launches"
    for name, off in WINDOWS.items():
        for s, got, want in zip("fg", (fn, gn), oracles[name].noise()):
            e = rel_err(_inner(_cut(got, off, N), 1), _inner(want, 1))
            if e > TOL:
                return f"noise() {s}, window {name}: rel err {e:.3e} on cells >= 1 from the window faces"
    del fn, gn
    nr, n = _counted(lat, lat.normals)
    if n != download_chunks(33):
        return f"normals(): {n} observer launches"
    if not np.array_equal(nr[z_tail:], tail):
        return "normals() in its last two chunks differs from a slab's normals of the same planes"
    for name, off in WINDOWS.items():
        if not np.array_equal(nr[_window(off, N)], normals[name]):
            return f"normals() on window {name} differs from a slab's normals of the same cells"
    return None


@pytest.mark.gpu
def test_fluctuating_bench_kernel_on_windows(bflbm, oracle_mod, monkeypatch):
    """512^3 from the tile, one deterministic step (still periodic), then kBT = 1e-5: two steps of exactly the bench's kernel
    against oracles on three 64^3 windows with the big box's normals injected (1e-12 at margin 1, then 1e-11 at margin 3);
    after the first, hydro fields (margin 2), noise (margin 1) and the whole-box normals through the chunked host downloads"""
    import torch
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    monkeypatch.setenv("BFLBM_CTA_THREADS", "256")
    first, _ = _run_twin(bflbm, oracle_mod, "fused", (0.5, 0.5), long=False)
    det, seed = _bench_params(0.0)
    noisy, _ = _bench_params(KBT)
    f0, g0 = _tile(oracle_mod)
    with bflbm.Lattice(N, N, N, params=bflbm.Params(**det, seed=seed)) as lat:
        _configure(lat, "fused")
        ft, gt = _tiled(f0, N // T), _tiled(g0, N // T)
        lat.init_from_populations(ft, gt)
        del ft, gt
        lat.step(1)  # the twin's first step, repeated (test_whole_box_periods_equal_the_twin)
        lat.set_params(kBT=KBT)
        s1 = lat.step_count
        nrm = _window_normals(bflbm, noisy, seed, (s1, s1 + 1, s1 + 2))
        z_tail = (download_chunks(33) - 2) * chunk_planes(33)  # first plane of the last two chunks of normals()
        tail = _slab_normals(bflbm, noisy, seed, z_tail, N - z_tail, (s1 + 1,))[s1 + 1]
        oracles = {}
        for name, off in WINDOWS.items():
            O = oracle_mod.PortOracle(W, W, W)
            O.set_params(**noisy)
            O.set_normals(nrm[name, s1])
            O.init_from_populations(*(_cut(a, off, T) for a in first))
            O.set_normals(nrm[name, s1 + 1])  # the normals of the noise generated at the end of the step
            O.step(1)
            oracles[name] = O

        lat.step(1)
        assert lat.last_step() == BENCH_VARIANT
        _settle(lat)
        _assert_windows(lat, oracles, 1, TOL, "first noisy step")
        msg = _host_downloads_mismatch(lat, oracles, {name: nrm[name, s1 + 1] for name in WINDOWS}, z_tail, tail)
        assert msg is None, msg

        for name, O in oracles.items():
            O.set_normals(nrm[name, s1 + 2])
            O.step(1)
        lat.step(1)
        assert lat.last_step() == BENCH_VARIANT
        _settle(lat)
        _assert_windows(lat, oracles, 3, 10 * TOL, "second noisy step")
        assert lat.step_count == s1 + 2
        _report("fluctuating bench kernel", t0, lat.device_bytes)
