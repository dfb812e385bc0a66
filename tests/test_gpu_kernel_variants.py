"""Every compiled variant of the step kernels against the CPU oracle.

The library compiles 16 instantiations of the fused brick kernel, k_step_fused<NOISE, RATE1, FULL, NT>, and 4 of the
thread-per-cell two-pass kernel, k_step_twopass<NOISE, RATE1>, whose launch block is 8x32 ... 128x2 depending on nx.
Which one a step runs follows from the box, the relaxation times, kBT, the brick height and the switches read at
bflbm_create (BFLBM_CTA_THREADS, BFLBM_RATE1, BFLBM_FOLD_IN_STAGING, BFLBM_OVERLAP); so do the fold source (the
brick-interior planes staged from the extended boxes E of the step before, or every plane from R after a full k_fold<0>
pass) and, for slabs, the schedule.  CASES declares the inputs of each case and the tile and CTA counts it must get; the
whole expected variant comes from a Python restatement of make_brick_grid / fold_in_staging_ok (fused.cuh) and of the
two-pass block rule (create_common, capi.cu).

* Without a GPU: the restatement reproduces the declared tiles, and the table spans every instantiation, every two-pass
  block width, every fold source and every schedule.
* On the GPU: each case is stepped next to the C oracle from a droplet with a seeded random perturbation (no mirror symmetry
  that could hide swapped neighbours), with the GPU's normals injected when kBT > 0 -- which also checks that every variant
  keys its in-kernel generator like the normals observer.  Lattice.last_step() must report the declared variant, so a
  case cannot pass on a kernel other than the one it names.  Slab schedules are compared bit for bit with the whole box.
"""
import itertools
from dataclasses import dataclass

import numpy as np
import pytest

from conftest import assert_hydro_close, rel_err

TOL = 1e-12
KBTS = (0.0, 1e-5)
TAUS = ((0.5, 0.5), (0.7, 0.55))


# ---- restatement of the kernel choice ----------------------------------------------------------------------------------
def ceil_div(a, b):
    return -(-a // b)


def brick_grid(shape, nt, lz=0):
    """make_brick_grid (fused.cuh): (tx, ty, bx, by, bz, lz) of the fused kernel with nt threads per CTA; lz = 0 is the
    automatic brick height."""
    nx, ny, nz = shape
    tx = 8
    while tx < nx and tx < 32:
        tx <<= 1
    ty = nt // tx
    bx, by = ceil_div(nx, tx), ceil_div(ny, ty)
    if lz <= 0:
        slots = 148 * 2
        lz = 4
        for c in (32, 16, 8):
            ctas = bx * by * ceil_div(nz, c)
            if (slots * 8) // 10 <= ctas <= slots or ctas >= 2 * slots:
                lz = c
                break
    lz = max(2, min(lz, nz))
    return tx, ty, bx, by, ceil_div(nz, lz), lz


def fold_in_staging_ok(shape, tx, ty, bx, by):
    """fold_in_staging_ok (fused.cuh): the last brick is at least two cells wide in x and y (the 2^31 bound on E is far away
    for these boxes)."""
    nx, ny, _ = shape
    return nx - (bx - 1) * tx >= 2 and ny - (by - 1) * ty >= 2 and (tx + 2) * (ty + 2) <= 2 * tx * ty


def twopass_block(nx):
    """launch block of the two-pass kernels (create_common, capi.cu)"""
    bx = 8
    while bx < nx and bx < 128:
        bx <<= 1
    return bx, 256 // bx


def expected_variant(algo, nt, shape, lz, kbt, tau, env=(), schedule=0):
    """What Lattice.last_step() reports in steady state (from the second step after an upload on)."""
    env = dict(env)
    nx, ny, nz = shape
    rate1 = int(tuple(tau) == (0.5, 0.5) and env.get("BFLBM_RATE1") != "0")
    noise = int(kbt > 0)
    if algo == "twopass":
        bx, by = twopass_block(nx)
        return dict(algorithm=1, threads=bx * by, tile_x=bx, tile_y=by, lz=1, bx=ceil_div(nx, bx), by=ceil_div(ny, by), bz=nz,
                    full=0, rate1=rate1, noise=noise, fold_source=0, schedule=0, graph=0)
    tx, ty, bx, by, bz, lz = brick_grid(shape, nt, lz)
    staged = env.get("BFLBM_FOLD_IN_STAGING") != "0" and fold_in_staging_ok(shape, tx, ty, bx, by)
    return dict(algorithm=0, threads=tx * ty, tile_x=tx, tile_y=ty, lz=lz, bx=bx, by=by, bz=bz, full=int(nx % tx == 0 and ny % ty == 0),
                rate1=rate1, noise=noise, fold_source=int(staged), schedule=schedule, graph=0)


# ---- the case table ----------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    algo: str      # "fused" or "twopass"
    nt: int        # BFLBM_CTA_THREADS
    shape: tuple   # (nx, ny, nz)
    lz: int        # brick height passed to set_tiling (fused)
    kbt: float
    tau: tuple     # (tau_f, tau_g)
    tile: tuple    # declared (tx, ty) of the fused tile, or the two-pass block
    ctas: tuple    # declared CTAs per axis: (bx, by, bz) bricks, or the two-pass grid
    env: tuple = ()  # further switches, ((name, value), ...)

    def __str__(self):
        env = "".join(f"-{k[6:].lower()}{v}" for k, v in self.env)
        return (f"{self.algo}-nt{self.nt}-{'x'.join(map(str, self.shape))}-lz{self.lz}-kbt{self.kbt:g}"
                f"-tau{self.tau[0]:g}_{self.tau[1]:g}{env}")

    def variant(self):
        return expected_variant(self.algo, self.nt, self.shape, self.lz, self.kbt, self.tau, self.env)

    @property
    def fold(self):
        """where the step kernel's densities come from"""
        if self.algo == "twopass":
            return "two-pass density pass"
        if dict(self.env).get("BFLBM_FOLD_IN_STAGING") == "0":
            return "fold pass (switch)"
        return "staged from E" if self.variant()["fold_source"] else "fold pass (one-cell-wide last brick)"

    @property
    def graph_capable(self):
        """bflbm_step replays graphs only for kernels that do not need the full fold pass (graph_ok, capi.cu)"""
        v = self.variant()
        return v["algorithm"] == 1 or v["fold_source"] == 1


# (NT, shape, brick height, declared tile, declared bricks): each at kBT x tau in KBTS x TAUS
FUSED_SHAPES = [
    (256, (64, 16, 24), 8, (32, 8), (2, 2, 3)),    # FULL; shells cross brick faces in x, y and z
    (256, (64, 16, 70), 32, (32, 8), (2, 2, 3)),   # FULL; the bench's brick height, a 6-plane last row
    (256, (40, 19, 20), 6, (32, 8), (2, 3, 4)),    # partial in x, y and z
    (256, (16, 32, 16), 4, (16, 16), (1, 2, 4)),   # FULL
    (256, (13, 21, 18), 5, (16, 16), (1, 2, 4)),   # partial
    (256, (8, 64, 12), 4, (8, 32), (1, 2, 3)),     # FULL (the tile of the 8 x 256 x 64 job)
    (256, (7, 45, 10), 4, (8, 32), (1, 2, 3)),     # partial
    (256, (33, 17, 12), 4, (32, 8), (2, 3, 3)),    # one-cell-wide last brick in x and y: k_fold<0> every step
    (128, (64, 8, 24), 8, (32, 4), (2, 2, 3)),     # FULL
    (128, (40, 10, 20), 6, (32, 4), (2, 3, 4)),    # partial
    (128, (16, 16, 16), 4, (16, 8), (1, 2, 4)),    # FULL
    (128, (13, 11, 18), 5, (16, 8), (1, 2, 4)),    # partial
    (128, (8, 32, 12), 4, (8, 16), (1, 2, 3)),     # FULL
    (128, (7, 21, 10), 4, (8, 16), (1, 2, 3)),     # partial
    (128, (33, 9, 12), 4, (32, 4), (2, 3, 3)),     # one-cell-wide last brick
]
# two-pass: one box per block width; declared block and grid
TWOPASS_SHAPES = [
    ((5, 40, 9), (8, 32), (1, 2, 9)),
    ((12, 20, 11), (16, 16), (1, 2, 11)),
    ((24, 14, 10), (32, 8), (1, 2, 10)),
    ((48, 9, 8), (64, 4), (1, 3, 8)),
    ((100, 6, 7), (128, 2), (1, 3, 7)),
]
# the FULL 32-wide shape of each NT, with the separate fold pass forced or the general relaxation code at rate 1
SWITCH_SHAPES = [(256, (64, 16, 24), 8, (32, 8), (2, 2, 3)), (128, (64, 8, 24), 8, (32, 4), (2, 2, 3))]

CASES = (
    [Case("fused", nt, shape, lz, kbt, tau, tile, ctas) for nt, shape, lz, tile, ctas in FUSED_SHAPES for kbt in KBTS for tau in TAUS]
    + [Case("twopass", 256, shape, 0, kbt, tau, tile, ctas) for shape, tile, ctas in TWOPASS_SHAPES for kbt in KBTS for tau in TAUS]
    + [Case("fused", nt, shape, lz, kbt, tau, tile, ctas, (("BFLBM_FOLD_IN_STAGING", "0"),))
       for nt, shape, lz, tile, ctas in SWITCH_SHAPES for kbt in KBTS for tau in TAUS]
    + [Case("fused", nt, shape, lz, kbt, (0.5, 0.5), tile, ctas, (("BFLBM_RATE1", "0"),))
       for nt, shape, lz, tile, ctas in SWITCH_SHAPES for kbt in KBTS]
)

# slab schedules: nz = 48 in 3 emulated slabs of 16 planes, brick height 4 (4 brick rows per slab, slab faces = brick faces)
SLABS, SLAB_LZ = 3, 4
SLAB_SHAPES = [  # (NT, shape, tau): FULL at the shipped tau = 1/2, partial at general rates
    (256, (64, 16, 48), (0.5, 0.5)),
    (256, (40, 19, 48), (0.7, 0.55)),
    (128, (64, 8, 48), (0.5, 0.5)),
    (128, (40, 10, 48), (0.7, 0.55)),
]
SLAB_OVERLAP = [True, False]


def slab_variant(nt, shape, tau, overlap, kbt):
    nx, ny, nz = shape
    return expected_variant("fused", nt, (nx, ny, nz // SLABS), SLAB_LZ, kbt, tau, schedule=2 if overlap else 1)


# ---- CPU: the table -----------------------------------------------------------------------------------------------------
def test_restated_rules_give_the_declared_tiles():
    for c in CASES:
        v = c.variant()
        assert (v["tile_x"], v["tile_y"]) == c.tile and (v["bx"], v["by"], v["bz"]) == c.ctas, str(c)
        assert v["threads"] == (256 if c.algo == "twopass" else c.nt), str(c)
    # the automatic brick height: 32 planes from 128^3 upwards (DESIGN section 6), 4 on small boxes
    assert brick_grid((128, 128, 128), 256) == (32, 8, 4, 16, 4, 32)
    assert brick_grid((512, 512, 512), 256) == (32, 8, 16, 64, 16, 32)
    assert brick_grid((32, 32, 32), 128) == (32, 4, 1, 8, 8, 4)
    for nt, shape, tau in SLAB_SHAPES:
        v = slab_variant(nt, shape, tau, True, 1e-5)
        assert v["bz"] == 4 and v["fold_source"] == 1, "the overlapped schedule needs >= 3 brick rows and fold-in-staging"


def test_case_table_spans_every_variant():
    fused = [c.variant() for c in CASES if c.algo == "fused"]
    twopass = [c.variant() for c in CASES if c.algo == "twopass"]
    assert {(v["noise"], v["rate1"], v["full"], v["threads"]) for v in fused} == set(itertools.product((0, 1), (0, 1), (0, 1), (128, 256)))
    assert {(v["noise"], v["rate1"], v["tile_x"]) for v in twopass} == set(itertools.product((0, 1), (0, 1), (8, 16, 32, 64, 128)))
    folds = {c.fold for c in CASES} | {"overlapped slab fold" if ov else "staged from E" for ov in SLAB_OVERLAP}
    assert folds == {"staged from E", "fold pass (switch)", "fold pass (one-cell-wide last brick)", "two-pass density pass",
                     "overlapped slab fold"}
    schedules = {c.variant()["schedule"] for c in CASES} | {slab_variant(*s, ov, 1e-5)["schedule"] for s in SLAB_SHAPES for ov in SLAB_OVERLAP}
    assert schedules == {0, 1, 2}
    assert len({str(c) for c in CASES}) == len(CASES)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _params(kbt, tau):
    return dict(kBT=kbt, tau_f=tau[0], tau_g=tau[1], alpha0=1.5, alpha1=0.0, kappa=0.1, rho_lo=0.1, rho_hi=3.0)


def _set_switches(monkeypatch, nt, env=()):
    monkeypatch.setenv("BFLBM_CTA_THREADS", str(nt))
    for k, v in env:
        monkeypatch.setenv(k, v)


def _asymmetric_state(oracle_mod, shape, seed):
    """a centred droplet's populations times (1 + 1e-3 u), u uniform on [0, 1): no mirror or axis-swap symmetry left"""
    f, g = oracle_mod.droplet_populations(*shape, 0.3, 0.1, 0.1, 3.0)
    rng = np.random.default_rng(seed)
    return f * (1 + 1e-3 * rng.random(f.shape)), g * (1 + 1e-3 * rng.random(g.shape))


def _assert_parity(lat, O, tol, what, v):
    """populations (max-norm relative error) and the 22 hydro fields; on failure names the worst component and cell and where
    the cell sits in its tile, so that errors on brick faces or tile edges show"""
    for name, got, want in zip("fg", lat.populations(), O.populations()):
        e = rel_err(got, want)
        if e > tol:
            c, z, y, x = np.unravel_index(np.argmax(np.abs(got - want)), got.shape)
            pytest.fail(f"{what}: {name} rel err {e:.3e} > {tol:.0e}; worst {name}[{c}] at (x, y, z) = ({x}, {y}, {z}), "
                        f"position in its tile ({x % v['tile_x']}, {y % v['tile_y']}, {z % v['lz']}) of "
                        f"({v['tile_x']}, {v['tile_y']}, {v['lz']})")
    # The velocities of this perturbed state are ~1e-4 (VEL_FLOOR), so 1e-12 of them is below one ulp of the population
    # sums they are made of: measured up to 1.5e-12 after one step and 1.5e-10 after four while the populations agree to
    # the bars above.  The fields take 100 x the population bar; the populations are what a wrong variant moves.
    assert_hydro_close(lat.hydrovars(), O.hydrovars(), 100 * tol, what)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=str)
def test_variant_matches_oracle(bflbm, oracle_mod, monkeypatch, case):
    """4 single steps against the oracle (1e-12 after the first, 1e-11 after later ones), the launched variant reported
    by every step, and at kBT = 0 six more steps replayed from graphs (4 + 2) where the variant allows it."""
    _set_switches(monkeypatch, case.nt, case.env)
    prm = _params(case.kbt, case.tau)
    want = case.variant()
    noise = case.kbt > 0
    f0, g0 = _asymmetric_state(oracle_mod, case.shape, seed=sum(case.shape) + case.nt)
    with bflbm.Lattice(*case.shape, params=bflbm.Params(**prm, seed=31, step0=5)) as lat:
        lat.set_algorithm(case.algo)
        if case.algo == "fused":
            lat.set_tiling(case.lz)
        lat.init_from_populations(f0, g0)
        O = oracle_mod.PortOracle(*case.shape)
        O.set_params(**prm)
        if noise:
            O.set_normals(lat.normals())
        O.init_from_populations(f0, g0)
        for s in range(4):
            lat.step(1)
            if noise:
                O.set_normals(lat.normals())  # normals of the noise generated at the end of this step
            O.step(1)
            _assert_parity(lat, O, TOL if s == 0 else 10 * TOL, f"{case} step {s + 1}", want)
            # the first step after an upload stages every plane from R
            assert lat.last_step() == (want if s else {**want, "fold_source": 0}), f"step {s + 1}"
        if not noise:
            lat.step(6)
            O.step(6)
            _assert_parity(lat, O, 10 * TOL, f"{case} 6 steps in one call", want)
            assert lat.last_step() == {**want, "graph": int(case.graph_capable)}
        assert lat.step_count == 5 + (4 if noise else 10)


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", SLAB_OVERLAP, ids=["overlapped", "one-stream"])
@pytest.mark.parametrize("peer", [False, True], ids=["copies", "peer"])
@pytest.mark.parametrize("nt,shape,tau", SLAB_SHAPES, ids=[f"nt{nt}-{'x'.join(map(str, s))}" for nt, s, _ in SLAB_SHAPES])
def test_slab_schedules_bitwise_equal_to_whole_box(bflbm, monkeypatch, nt, shape, tau, peer, overlap):
    """Three emulated slabs against the whole box with the same brick height: same bits for populations, hydro fields and
    normals, with the interior rows overlapping the exchange and with BFLBM_OVERLAP=0, at both CTA sizes."""
    from bflbm_b200.distributed import EmulatedSlabs
    _set_switches(monkeypatch, nt, () if overlap else (("BFLBM_OVERLAP", "0"),))
    kbt = 1e-5
    prm = bflbm.Params(**_params(kbt, tau), seed=99)
    want = slab_variant(nt, shape, tau, overlap, kbt)
    with bflbm.Lattice(*shape, params=prm) as whole:
        whole.set_algorithm("fused")
        whole.set_tiling(SLAB_LZ)
        whole.init_droplet(0.3)
        S = EmulatedSlabs(*shape, SLABS, params=prm, brick_lz=SLAB_LZ, peer=peer)
        try:
            S.init_droplet(0.3)
            for _ in range(3):
                whole.step(2)
                S.step(2)
                fw, gw = whole.populations()
                fs, gs = S.gather("populations")
                assert np.array_equal(fw, fs) and np.array_equal(gw, gs)
                assert np.array_equal(whole.hydrovars(), S.gather("hydrovars"))
                assert all(lat.last_step() == want for lat in S.lats), [lat.last_step() for lat in S.lats]
            assert whole.last_step()["schedule"] == 0
            assert np.array_equal(whole.normals(), S.gather("normals"))
            if peer:
                assert all(lat.halo_error() == 0 for lat in S.lats)
        finally:
            S.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kbt", KBTS)
def test_graph_replay_bitwise_equal_to_single_launches_128_threads(bflbm, monkeypatch, kbt):
    """The NT = 128 kernels replayed from CUDA graphs (device-side step counter in the noise key) give the bits of plain
    launches (BFLBM_GRAPH=0), whatever the split into calls; automatic brick height."""
    shape = (32, 32, 32)
    prm = bflbm.Params(**_params(kbt, (0.5, 0.5)), seed=2024)
    want = expected_variant("fused", 128, shape, 0, kbt, (0.5, 0.5))
    assert want["full"] == 1 and want["threads"] == 128
    _set_switches(monkeypatch, 128, (("BFLBM_GRAPH", "0"),))
    with bflbm.Lattice(*shape, params=prm) as P:
        monkeypatch.delenv("BFLBM_GRAPH")
        with bflbm.Lattice(*shape, params=prm) as Gr:
            for lat in (P, Gr):
                lat.set_algorithm("fused")
                lat.init_droplet(0.3)
            for n in (1, 87, 2, 5, 64):  # 87 = 64 + 16 + 4 + 2 + 1
                P.step(n)
                Gr.step(n)
                fp, gp = P.populations()
                fg, gg = Gr.populations()
                assert np.array_equal(fp, fg) and np.array_equal(gp, gg), f"graph replay differs after a call of {n} steps"
                assert np.array_equal(P.hydrovars(), Gr.hydrovars())
            assert P.last_step() == want
            assert Gr.last_step() == {**want, "graph": 1}
            assert Gr.step_count == P.step_count == 159


@pytest.mark.gpu
def test_last_step_before_the_first_step(bflbm):
    with bflbm.Lattice(8) as lat:
        lat.init_mixture()
        with pytest.raises(bflbm.BflbmError, match="no step"):
            lat.last_step()
        lat.step(1)
        assert lat.last_step()["algorithm"] == 1  # a small whole box takes the two-pass kernels by default
