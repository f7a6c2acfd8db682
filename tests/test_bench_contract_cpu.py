"""bench.py contract checks that need no GPU: the reference arm (CPU port of the reference's path) prints ONE JSON line
with the keys the driver reads, and the B200 arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, timeout=600, env=None):
    env = dict(env or os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = run("--impl", "reference", "--workload", "lift_splat", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "bev_frames_per_sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["vs_baseline"] is None
    # "reference" = the unmodified reference package (oracle/_ref or STP3_REFERENCE_ROOT); "port" only where neither exists
    assert d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["samples_per_gpu_per_step"] == 4


# A stand-in with the reference package's layout and the interfaces the reference arm calls (oracle/ref_loader.py,
# oracle/make_golden.run_reference), built from this repository's own modules and CPU port.
STAND_IN = {
    "stp3/__init__.py": "",
    "stp3/layers/__init__.py": "",
    "stp3/layers/convolutions.py": "",
    "stp3/layers/temporal.py": "",
    "stp3/utils/__init__.py": "",
    "stp3/utils/geometry.py": "from stp3_b200.utils.geometry import calculate_birds_eye_view_parameters  # noqa: F401\n",
    "stp3/utils/network.py": (
        "def pack_sequence_dim(x):\n"
        "    return x.view(x.shape[0] * x.shape[1], *x.shape[2:])\n\n\n"
        "def unpack_sequence_dim(x, b, s):\n"
        "    return x.view(b, s, *x.shape[1:])\n"),
    "stp3/models/__init__.py": "",
    "stp3/models/encoder.py": "",
    "stp3/models/decoder.py": "from stp3_b200.models.decoder import Decoder  # noqa: F401\n",
    "stp3/models/temporal_model.py": "from stp3_b200.models.temporal_model import TemporalModel  # noqa: F401\n",
    "stp3/models/stp3.py": (
        "from oracle import torch_port as TP\n"
        "from stp3_b200.utils.geometry import frustum_axes\n\n\n"
        "class STP3:\n"
        "    def create_frustum(self):\n"
        "        return TP.frustum(*frustum_axes(self.cfg.IMAGE.FINAL_DIM, self.encoder_downsample, self.cfg.LIFT.D_BOUND))\n\n"
        "    def get_geometry(self, intrinsics, extrinsics):\n"
        "        return TP.get_geometry(self.frustum, intrinsics, extrinsics)\n\n"
        "    def projection_to_birds_eye_view(self, x, geom, future_egomotion):\n"
        "        return TP.projection(x, geom, future_egomotion, self.bev_resolution, self.bev_start_position,\n"
        "                             self.bev_dimension, self.discount)\n"),
}


def test_reference_arm_uses_the_installed_reference_when_present(tmp_path):
    """A reference install present (oracle/_ref from oracle/build_ref.py, or STP3_REFERENCE_ROOT) -> the arm times
    that package's own modules."""
    for rel, text in STAND_IN.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    env = dict(os.environ, STP3_REFERENCE_ROOT=str(tmp_path))
    r = run("--impl", "reference", "--workload", "lift_splat", "--steps", "1", "--warmup", "0", env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][0])
    assert d["cpu_baseline"]["kind"] == "reference"


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    """--dump-outputs: one float32 / float64 .npy per returned tensor; beyond the byte limit, the same seeded sample
    of every array from run to run."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(0)
    out = {"a": torch.randn(2, 3, 50, 40, generator=g), "b": torch.randn(7, generator=g, dtype=torch.float64),
           "c": torch.arange(6, dtype=torch.int32), "none": None}
    bench.dump_outputs(out, tmp_path / "full")
    assert sorted(p.name for p in (tmp_path / "full").iterdir()) == ["a.npy", "b.npy", "c.npy"]
    for k, dtype in (("a", np.float32), ("b", np.float64), ("c", np.float32)):
        got = np.load(tmp_path / "full" / f"{k}.npy")
        assert got.dtype == dtype and np.array_equal(got, out[k].numpy().astype(dtype))
    limit = 16000
    for run_dir in ("s1", "s2"):
        bench.dump_outputs(out, tmp_path / run_dir, limit=limit)
    files = sorted((tmp_path / "s1").iterdir())
    assert sum(p.stat().st_size for p in files) <= limit
    a = np.load(tmp_path / "s1" / "a.npy")
    assert 0 < a.size < out["a"].numel() and np.isin(a, out["a"].numpy()).all()
    for p in files:
        assert np.array_equal(np.load(p), np.load(tmp_path / "s2" / p.name))


def test_b200_arm_has_no_cpu_fallback():
    r = run("--steps", "1", "--warmup", "3", "--no-cpu-baseline", timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_extras_watchdog_prints_the_line_it_has():
    """Once the timed regions are done the contract line exists; if the explanatory part (sustained loop, stage graphs,
    latency mode ...) never comes back, rank 0 prints that line with a note and every rank exits 0."""
    import io
    import time
    sys.path.insert(0, ROOT)
    import bench
    exits = []
    for rank in (0, 1):
        bench._LINE["line"] = {"metric": "bev_frames_per_sec", "value": 1.0}
        buf = io.StringIO()
        dog = bench.extras_watchdog(0.05, rank, exit_fn=exits.append, out=buf)
        dog.join(5)
        time.sleep(0.05)
        lines = [l for l in buf.getvalue().splitlines() if l.strip()]
        if rank == 0:
            assert len(lines) == 1
            d = json.loads(lines[0])
            assert d["value"] == 1.0 and "timed out" in d["extras"]["unavailable"]
        else:
            assert lines == []
    assert exits == [0, 0]
    # cancelled in time: nothing is printed, nobody exits
    buf = io.StringIO()
    dog = bench.extras_watchdog(0.2, 0, exit_fn=exits.append, out=buf)
    dog.cancel()
    time.sleep(0.4)
    assert buf.getvalue() == "" and exits == [0, 0]
