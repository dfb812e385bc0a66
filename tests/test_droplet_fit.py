"""Droplet (W, R) fit, SURVEY 8(f) row 4 (fittingDropletParams, LBM_hydrovs.H:160-213 + externlib.H:21-403; call site
main_run_job.cpp:358-369).  Checker: the reference's own externlib.H compiled unchanged (oracle/_ref/libbflbm_ref_fit.so,
oracle/ref_fit_wrapper.cpp) and the fixture it produced (tests/golden/droplet_fit.json, tests/golden/make_fit_golden.py).
  CPU: the host-side restatement of the closed-form flow coefficients (csrc/droplet_fit.hpp) against both;
  GPU: the device reductions of the two lattice integrals and the whole fit on a lattice, against the reference fit of the
       downloaded density field."""
import ctypes
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "droplet_fit.json")))


def _coef(lib, W, R, dt, C0):
    out = np.empty(6)
    rc = lib.bflbm_debug_fit_coefficients(W, R, 0.2, 0.2, dt, C0, out.ctypes.data)
    assert rc == 0
    return out


def test_flow_coefficients_match_the_reference_functions(bflbm, oracle_mod):
    """JRn_Rn, JWn_Rn, JRn_Wn, JWn_Wn, KWn, KRn (externlib.H:203-244, 342-366): pure host arithmetic, no GPU needed."""
    lib = bflbm.load_library()
    for row in GOLD["coefficients"]:
        got, want = _coef(lib, row["W"], row["R"], row["dt"], row["C0"]), np.array(row["values"])
        assert np.abs(got - want).max() <= 1e-13 * np.abs(want).max(), (row, got, want)
    if oracle_mod.RefFit.available():
        F = oracle_mod.RefFit()
        rng = np.random.default_rng(2)
        for _ in range(40):
            W, R = 10 ** rng.uniform(-4.2, -0.8), rng.uniform(0.12, 0.45)
            dt, C0 = 0.02 / 5 ** rng.integers(0, 4), rng.uniform(0.5, 3.0)
            got, want = _coef(lib, W, R, dt, C0), F.coefficients(W, R, 0.2, 0.2, dt, C0)
            assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max(), (W, R, dt, C0)


def test_fixture_is_the_reference_fit(oracle_mod):
    if not oracle_mod.RefFit.available():
        pytest.skip("oracle/_ref/libbflbm_ref_fit.so not built from the original project's source tree: make -C oracle ref REFERENCE=<that tree>")
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_fit_golden", os.path.join(HERE, "golden", "make_fit_golden.py"))
    G = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(G)
    W, R, u, ok, _ = oracle_mod.RefFit().fit(G.synthetic(), 0.1, 0.3)
    assert ok and W == GOLD["synthetic"]["W"] and R == GOLD["synthetic"]["R"]


@pytest.mark.gpu
def test_gpu_fit_terms_and_fit_match_the_reference(bflbm, oracle_mod):
    """The authors' droplet recipe at 32^3 relaxed for 400 steps on the GPU (kBT = 0), then fitted with the call of
    main_run_job.cpp:365 (W0 = kappa, R0 = radius, window 20, bound 0.01, 400 flow steps): the two lattice integrals of a flow
    step and the fitted (W, R) against the reference's externlib.H on the downloaded density, and against the fixture (whose
    density came from the reference headers' own 400 steps)."""
    n = 32
    prm = bflbm.Params(kBT=0.0, alpha0=1.5, kappa=0.1, rho_lo=0.1, rho_hi=3.0)
    with bflbm.Lattice(n, n, n, params=prm) as lat:
        lat.init_droplet(0.3)
        lat.step(400)
        rho = lat.hydrovars()[0]
        W, R, u, ok = lat.fit_droplet(prm.kappa, 0.3)
        gold = GOLD["relaxed"]
        assert ok and abs(W / gold["W"] - 1) < 1e-6 and abs(R / gold["R"] - 1) < 1e-8, (W, R, gold["W"], gold["R"])
        assert abs(rho.sum() / gold["rho_sum"] - 1) < 1e-12
        if oracle_mod.RefFit.available():
            F = oracle_mod.RefFit()
            mw, mr, com = F.field_terms(rho, 0.1, 0.3)
            s4 = np.empty(4)
            r0 = np.ascontiguousarray(com)
            bflbm.lattice._check(lat.lib.bflbm_droplet_fit_terms(lat.h, 0.1, 0.3, r0.ctypes.data, s4.ctypes.data))
            s, vol = np.sqrt(2 * 0.1), 1.0 / n ** 3
            assert abs(s4[0] * vol / s ** 3 / mw - 1) < 1e-12 and abs(s4[1] * vol / s / mr - 1) < 1e-12
            assert s4[2] == rho.min() and s4[3] == rho.max()
            ci = lat.center_of_mass()[0]
            assert np.allclose((ci + 0.5) / n, com, rtol=1e-13)
            Wr, Rr, ur, okr, _ = F.fit(rho, 0.1, 0.3)
            assert okr and abs(W / Wr - 1) < 1e-8 and abs(R / Rr - 1) < 1e-10 and abs(u - ur) < 1e-6, (W, Wr, R, Rr)
    with bflbm.MultiLattice(n, n, n, params=prm, ngpus=1) as M:  # the same through the multi-GPU object
        M.init_droplet(0.3)
        M.step(400)
        out, okc = np.empty(3), ctypes.c_int()
        M._mcheck(M.lib.bflbm_multi_fit_droplet(M.h, 20, 0.01, 400, 0.1, 0.3, 0.2, 0.2, 0.02, out.ctypes.data, ctypes.byref(okc)))
        assert okc.value == 1 and out[0] == W and out[1] == R
