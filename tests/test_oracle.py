"""CPU tests (no GPU): the plain-C oracle is pinned against
 (1) the committed fixtures in tests/golden/ (outputs of the reference's own headers, see make_golden.py),
 (2) oracle/_ref itself when it is present (this container), bit for bit,
 (3) textbook properties of the D3Q19 moment basis.
"""
import glob
import os

import numpy as np
import pytest

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def load_case(path):
    d = np.load(path)
    params = {k[2:]: float(d[k]) for k in d.files if k.startswith("p_")}
    return d, params


def drive(oracle, d, params, steps_cb):
    """Replays a fixture on an oracle-like object (PortOracle / RefOracle)."""
    normals = d["normals"] if "normals" in d.files else None
    k = 0

    def feed():
        nonlocal k
        if normals is not None:
            oracle.set_normals(normals[k])
            k += 1

    oracle.set_params(**params)
    feed()
    oracle.init_from_populations(d["f0"], d["g0"])
    done = 0
    for s in [int(x) for x in d["steps"]]:
        while done < s:
            feed()
            oracle.step(1)
            done += 1
        steps_cb(s)


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_port_matches_golden_bitwise(oracle_mod, path):
    d, params = load_case(path)
    nx, ny, nz = [int(v) for v in d["shape"]]
    P = oracle_mod.PortOracle(nx, ny, nz)

    def check(s):
        f, g = P.populations()
        assert np.array_equal(f, d[f"f_{s}"]) and np.array_equal(g, d[f"g_{s}"]), f"populations differ at step {s}"
        assert np.array_equal(P.hydrovars(), d[f"h_{s}"]), f"hydrovs differ at step {s}"
        assert np.array_equal(P.hydrovars_bar(), d[f"hb_{s}"]), f"hydrovsbar differ at step {s}"
        fn, gn = P.noise()
        assert np.array_equal(fn, d[f"fn_{s}"]) and np.array_equal(gn, d[f"gn_{s}"]), f"noise differs at step {s}"

    drive(P, d, params, check)
    assert np.array_equal(d["h0"].shape, (22, nz, ny, nx))


@pytest.mark.parametrize("init,arg,shape", [("stripe", 0.5, (8, 6, 12)), ("droplet", 0.3, (10, 10, 10)), ("mixture", None, (6, 6, 6))])
def test_port_analytic_inits_match_golden(oracle_mod, init, arg, shape):
    name = {"stripe": "stripe_default_8x6x12", "droplet": "droplet_default_10x10x10", "mixture": "mixture_default_6x6x6"}[init]
    d, params = load_case(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    P = oracle_mod.PortOracle(*shape)
    P.set_params(**params, rho_lo=0.0, rho_hi=1.0)
    getattr(P, "init_" + init)(*([] if arg is None else [arg]))
    f, g = P.populations()
    assert np.array_equal(f, d["f0"]) and np.array_equal(g, d["g0"])
    assert np.array_equal(P.hydrovars(), d["h0"])
    assert np.array_equal(P.hydrovars_bar(), d["hb0"])


def test_port_matches_reference_headers_bitwise(oracle_mod):
    if not oracle_mod.RefOracle.available():
        pytest.skip("oracle/_ref not built from the original project's source tree: make -C oracle ref REFERENCE=<that tree>")
    rng = np.random.default_rng(3)
    shape = (7, 9, 8)
    for params in (dict(kBT=0.0, tau_f=0.5, tau_g=0.5, alpha0=4.0, alpha1=0.0, kappa=4.0),
                   dict(kBT=3e-5, tau_f=0.65, tau_g=1.1, alpha0=1.5, alpha1=0.0, kappa=0.1)):
        R = oracle_mod.RefOracle(*shape)
        P = oracle_mod.PortOracle(*shape)
        R.set_params(**params)
        P.set_params(**params, rho_lo=R.rho_lo, rho_hi=R.rho_hi)
        for o in (R, P):
            o.set_normals(None)
        n0 = rng.standard_normal(R.shape + (33,))
        R.set_normals(n0)
        P.set_normals(n0)
        R.init_droplet(0.3)
        P.init_droplet(0.3)
        for _ in range(4):
            n = rng.standard_normal(R.shape + (33,))
            R.set_normals(n)
            P.set_normals(n)
            R.step(1)
            P.step(1)
        for a, b in zip(R.populations() + R.noise(), P.populations() + P.noise()):
            assert np.array_equal(a, b)
        assert np.array_equal(R.hydrovars(), P.hydrovars())
        assert np.array_equal(R.hydrovars_bar(), P.hydrovars_bar())


def test_lattice_constants_and_basis(oracle_mod):
    """c, w, b (LBM_d3q19.H:12-76) and the DSL basis: M is orthogonal under the weights with norms b."""
    c, w, b = oracle_mod.PortOracle.constants()
    assert c.shape == (19, 3) and abs(w.sum() - 1.0) < 1e-15
    assert np.allclose((w[:, None] * c).sum(0), 0) and np.allclose((w[:, None, None] * c[:, :, None] * c[:, None, :]).sum(0), np.eye(3) / 3)
    M = np.stack([oracle_mod.PortOracle.moments(np.eye(19)[i]) for i in range(19)], axis=1)  # M[k, i]
    assert np.allclose(M, np.round(M)), "basis vectors are integer"
    G = (M * w[None, :]) @ M.T
    assert np.allclose(G, np.diag(b), atol=1e-14)
    # inverse transform is the inverse
    rng = np.random.default_rng(0)
    f = rng.random(19)
    m = oracle_mod.PortOracle.moments(f)
    assert np.allclose(oracle_mod.PortOracle.populations_from_moments(m), f, atol=1e-15)
    assert np.allclose(m, M @ f, atol=1e-14)
    if oracle_mod.RefOracle.available():
        oracle_mod.RefOracle(2, 2, 2)
        cr, wr, br = oracle_mod.RefOracle.constants()
        assert np.array_equal(c, cr) and np.array_equal(w, wr) and np.array_equal(b, br)
        assert np.array_equal(oracle_mod.RefOracle.moments(f), m)


def test_conservation_and_reference_invariants(oracle_mod):
    """Mass of each species and total momentum noise: SURVEY.md 3.2b (meq_0 = rho_s, Phi_0 = 0, xi^g = -xi^f)."""
    P = oracle_mod.PortOracle(8, 8, 8)
    P.set_params(kBT=1e-5, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0)
    rng = np.random.default_rng(5)
    P.set_normals(rng.standard_normal(P.shape + (33,)))
    P.init_droplet(0.3)
    hb0 = P.hydrovars_bar()
    for _ in range(5):
        P.set_normals(rng.standard_normal(P.shape + (33,)))
        P.step(1)
    hb = P.hydrovars_bar()
    assert abs(hb[0].sum() - hb0[0].sum()) < 1e-11 * hb0[0].sum()
    assert abs(hb[1].sum() - hb0[1].sum()) < 1e-11 * hb0[1].sum()
    fn, gn = P.noise()
    assert np.array_equal(gn[1:4], -fn[1:4]) and not fn[0].any() and not gn[0].any()


def test_tau_half_forgets_nonconserved_moments(oracle_mod):
    """SURVEY.md section 9 item 10: at tau = 1/2 the post-collision state does not depend on the incoming
    non-conserved moments."""
    P = oracle_mod.PortOracle(6, 6, 6)
    P.set_params(alpha0=1.5, kappa=0.5, rho_lo=0.1, rho_hi=2.0)
    P.init_droplet(0.3)
    f, g = P.populations()
    rng = np.random.default_rng(2)
    # add a pure ghost-mode perturbation (mode 16) that leaves rho and j unchanged
    e16 = np.array([P.populations_from_moments(np.eye(19)[16])]).reshape(19, 1, 1, 1)
    f2 = f + 1e-3 * rng.random(f.shape[1:]) * e16
    A = oracle_mod.PortOracle(6, 6, 6); A.set_params(**P.params); A.init_from_populations(f, g); A.step(1)
    B = oracle_mod.PortOracle(6, 6, 6); B.set_params(**P.params); B.init_from_populations(f2, g); B.step(1)
    assert np.abs(A.populations()[0] - B.populations()[0]).max() < 1e-15


def test_port_reference_state_noise_matches_ref_build_bitwise(oracle_mod):
    """SURVEY 8(f) row 3: the reference headers compiled with -DUSE_REF_STATE (the macro LBM_binary.H:12 ships commented out) draw
    the noise amplitudes from the COM-shifted equilibrium profiles (:92-107, com_ref from main_run_job.cpp:229-233).  The C port's
    restatement of that branch is pinned bit for bit, with injected normals, general relaxation times and an equilibrium state
    displaced by (2, -1, 3) cells so that every component of the integer shift is non-zero."""
    if not oracle_mod.RefOracle.available(ref_state=True):
        pytest.skip("oracle/_ref/libbflbm_ref_refstate.so not built from the original project's source tree: make -C oracle ref REFERENCE=<that tree>")
    shape = (10, 12, 14)
    rng = np.random.default_rng(5)
    prm = dict(kBT=2e-5, tau_f=0.7, tau_g=0.6, alpha0=1.5, alpha1=0.0, kappa=0.1)
    f, g = oracle_mod.droplet_populations(*shape, 0.3, 0.1, 0.1, 3.0)
    P0 = oracle_mod.PortOracle(*shape)
    P0.set_params(**dict(prm, kBT=0.0), rho_lo=0.1, rho_hi=3.0)
    P0.init_from_populations(f, g)
    P0.step(5)
    hb = P0.hydrovars_bar()
    rho_eq, phi_eq = (np.roll(hb[k], (3, -1, 2), axis=(0, 1, 2)).copy() for k in (0, 1))
    # a smooth asymmetric modulation moves the centre of mass by a NON-integer amount: the shift is an integer truncation of
    # (com - com_ref), which must not sit on a rounding knife edge
    zz, yy, xx = np.meshgrid(*(np.arange(n) for n in shape[::-1]), indexing="ij")
    rho_eq *= 1.0 + 0.3 * np.cos(2 * np.pi * (xx + 0.3) / shape[0]) * np.cos(2 * np.pi * (yy - 1.1) / shape[1]) * np.sin(2 * np.pi * (zz + 0.7) / shape[2])
    R = oracle_mod.RefOracle(*shape, ref_state=True)
    assert R.uses_ref_state()
    R.set_params(**prm)
    R.set_equilibrium(rho_eq, phi_eq, rho_eq + phi_eq)
    P = oracle_mod.PortOracle(*shape)
    P.set_params(**prm, rho_lo=0.1, rho_hi=3.0)
    P.set_equilibrium(rho_eq, phi_eq, rho_eq + phi_eq)
    n = rng.standard_normal(shape[::-1] + (33,))
    R.set_normals(n)
    P.set_normals(n)
    R.init_from_populations(f, g)
    P.init_from_populations(f, g)
    assert np.array_equal(R.noise()[0], P.noise()[0]) and np.array_equal(R.hydrovars(), P.hydrovars())
    for _ in range(4):
        n = rng.standard_normal(shape[::-1] + (33,))
        R.set_normals(n)
        P.set_normals(n)
        R.step(1)
        P.step(1)
        assert np.array_equal(R.noise()[0], P.noise()[0]) and np.array_equal(R.noise()[1], P.noise()[1])
        assert np.array_equal(R.hydrovars(), P.hydrovars()) and np.array_equal(R.populations()[1], P.populations()[1])
    # and it is a different noise field from the shipped build's (current densities)
    Q = oracle_mod.PortOracle(*shape)
    Q.set_params(**prm, rho_lo=0.1, rho_hi=3.0)
    Q.set_normals(n)
    Q.init_from_populations(f, g)
    P.set_normals(n)
    P.init_from_populations(f, g)
    assert np.abs(Q.noise()[0] - P.noise()[0]).max() > 1e-3
