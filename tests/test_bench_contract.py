"""bench.py's output contract on a CPU-only box: the reference arm (the reference's own LBM_timestep on the host cores)
prints ONE JSON line with the keys the driver reads; the GPU arm refuses to run without a GPU instead of falling back."""
import importlib.util
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--cpu-size", "12", "--cpu-steps", "3",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("MLUPS") and d["unit"] == "MLUPS" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "MLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_dump_outputs_are_the_state_after_warmup_plus_timed_steps(bflbm, tmp_path):
    """--dump-outputs writes the fields of the timed lattice after exactly W + K steps: the noise is keyed by the step number,
    so one step more or less gives other populations.  A 16^3 box is smaller than the sample: every cell, in order."""
    import numpy as np
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--nx", "16", "--ny", "16", "--nz", "16", "--steps", "3", "--warmup", "2",
                        "--no-e2e", "--no-cpu", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.splitlines()[-1])["steps"] == 3
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    with bflbm.Lattice(16, 16, 16, params=bflbm.Params(**bench.PARAMS)) as lat:
        lat.set_algorithm("fused")
        lat.init_mixture()
        lat.step(5)
        f, g = lat.populations()
        want = {"f": f, "g": g, "hydrovars": lat.hydrovars()}
    for name, w in want.items():
        got = np.load(out / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, w.reshape(w.shape[0], -1)), name


class _FakeLat:
    """Stands in for bflbm_b200.Lattice in bench.run_e2e: records the calls and enforces the rules of the asynchronous
    transfer calls (one staged checkpoint at a time, a frame buffer is not reused before its download was waited for)."""

    def __init__(self, err_cls, refuse_staging=False):
        self.nx, self.ny, self.nz = 4, 3, 8
        self.h, self.calls = 1, []
        self.staged, self.initialised, self.frame_in_flight, self.frames = False, False, False, 0
        self.err_cls, self.refuse = err_cls, refuse_staging

        class _Lib:
            @staticmethod
            def bflbm_get_populations(h, f, g):
                return 0

            @staticmethod
            def bflbm_get_hydrovars_bar(h, out):
                return 0
        self.lib = _Lib()

    def init_from_populations(self, f, g):
        self.calls.append("init")
        self.initialised = True

    def step(self, n):
        assert self.initialised
        self.calls.append(("step", n))

    def sync(self):
        self.calls.append("sync")

    def stage_populations(self, f, g, ghosted=False):
        if self.refuse:
            raise self.err_cls("no room for staging")
        assert not self.staged, "one checkpoint at a time"
        assert f.flags.c_contiguous and f.shape == (19, self.nz, self.ny, self.nx) and not ghosted
        self.staged = True
        self.calls.append("stage")

    def init_from_staged(self):
        assert self.staged
        self.staged, self.initialised = False, True
        self.calls.append("init_staged")

    def hydrovars_bar_async(self, out):
        assert self.initialised and not self.frame_in_flight, "download_wait before the frame buffer is reused"
        self.frame_in_flight = True
        self.frames += 1
        out[...] = float(self.frames)
        self.calls.append("frame")

    def download_wait(self):
        self.frame_in_flight = False
        self.calls.append("wait")

    def release_staging(self):
        self.calls.append("release")


def _run_fake_e2e(refuse):
    import argparse
    import importlib.util
    import types

    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class Err(Exception):
        pass

    def no_pinned(*a, **k):
        raise RuntimeError("no CUDA: cannot pin")
    fake_torch = types.SimpleNamespace(empty=no_pinned, float64=None, cuda=types.SimpleNamespace(synchronize=lambda: None))
    fake_b = types.SimpleNamespace(BflbmError=Err)
    lat = _FakeLat(Err, refuse_staging=refuse)
    a = argparse.Namespace(e2e_steps=5, e2e_intervals=3)
    cells = lat.nx * lat.ny * lat.nz
    return bench.run_e2e(a, fake_b, np, fake_torch, lat, lat, 1, cells, cells), lat


def test_e2e_leg_call_order_pipelined():
    """Host logic of the e2e leg on a fake lattice: serial interval, untimed probe, then 3 intervals in which the next
    checkpoint is staged before the steps and the previous frame is waited for before its buffer is reused."""
    e, lat = _run_fake_e2e(refuse=False)
    serial = ["init", ("step", 5), "sync"]
    probe = ["stage", "init_staged", "frame", "wait"]
    pipe = ["stage", "init_staged", "stage", ("step", 5), "frame", "init_staged", "stage", ("step", 5), "wait", "frame",
            "init_staged", ("step", 5), "wait", "frame", "wait", "sync", "release"]
    assert lat.calls == serial + probe + pipe
    assert e["intervals"] == 3 and e["steps_per_interval"] == 5 and e["pinned_host"] is False and e["frames_equal"] is False
    cells = 4 * 3 * 8
    assert e["h2d_bytes_per_step"] == 2 * 19 * 8 * cells / 5 and e["d2h_bytes_per_step"] == 9 * 8 * cells / 5
    assert e["serial_interval"]["value"] > 0 and set(e["serial_interval"]["phases_s"]) == {"upload", "steps", "download"}
    assert "pipelined" not in e


def test_e2e_leg_falls_back_to_the_serial_interval_when_staging_is_refused():
    e, lat = _run_fake_e2e(refuse=True)
    assert lat.calls == ["init", ("step", 5), "sync", "release"]
    assert e["intervals"] == 1 and e["pipelined"].startswith("unavailable: no room for staging")
    assert e["value"] > 0 and set(e["phases_s"]) == {"upload", "steps", "download"}
