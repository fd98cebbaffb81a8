"""The reference arm of bench.py (the unmodified reference from oracle/_ref when built, else the oracle port,
timed on host cores) runs without a GPU and prints ONE JSON line with the keys the driver reads; the product
arm refuses to run without CUDA (no CPU fallback)."""

import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
  env = dict(os.environ, OMP_NUM_THREADS="4")
  return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env,
                        capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_the_contract_line():
  p = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-rays", "8")
  assert p.returncode == 0, p.stderr[-2000:]
  lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and d["unit"] == "rays/s" and d["higher_is_better"] is True
  assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
  from oracle import build_ref
  assert d["cpu_baseline"]["kind"] == ("reference" if build_ref.available() else "port")
  assert d["cpu_baseline"]["cores"] >= 1
  assert d["cpu_baseline"]["value"] == d["value"]
  assert d["e2e"] == {"value": d["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
  assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_falls_back_to_the_oracle_port_when_oracle_ref_is_absent(tmp_path, monkeypatch):
  """the GPU box only has what was built here; without oracle/_ref the arm times the oracle port"""
  from oracle import build_ref
  monkeypatch.setattr(build_ref, "OUT", str(tmp_path / "nothing"))
  assert not build_ref.available()
  sys.path.insert(0, ROOT)
  import bench
  kind, run = bench.make_cpu_runner()
  assert kind == "port"
  run(4)


def test_oracle_ref_is_the_unmodified_reference_when_built():
  from oracle import build_ref
  if not build_ref.available():
    if not build_ref.build():
      return  # no /root/reference here (GPU box without a prebuilt oracle/_ref)
  ref = build_ref.load()
  assert ref.rr.__file__.endswith(os.path.join("oracle", "_ref", "ibrnet", "render_ray.pyc"))
  assert callable(ref.rr.render_rays_mv) and callable(ref.ri.render_single_image_nvi)


def test_dump_outputs_writes_the_frame_as_float32_arrays(tmp_path):
  sys.path.insert(0, ROOT)
  import bench
  px = torch.randn(40, 5, generator=torch.Generator().manual_seed(0))
  bench.dump_outputs(str(tmp_path / "full"), px)
  got = {n: np.load(tmp_path / "full" / (n + ".npy")) for n in ("rgb", "depth", "mask")}
  assert all(v.dtype == np.float32 for v in got.values())
  np.testing.assert_array_equal(got["rgb"], px[:, 0:3].numpy())
  np.testing.assert_array_equal(got["depth"], px[:, 3].numpy())
  np.testing.assert_array_equal(got["mask"], px[:, 4].numpy())
  # above the size cap: the same seeded sample of rays, kept in ray order, on every call
  for d in ("a", "b"):
    bench.dump_outputs(str(tmp_path / d), px, cap_bytes=10 * 5 * 4)
  a, b = (np.load(tmp_path / d / "rgb.npy") for d in ("a", "b"))
  np.testing.assert_array_equal(a, b)
  rows = [int(np.flatnonzero((px[:, 0:3].numpy() == r).all(1))[0]) for r in a]
  assert a.shape == (10, 3) and rows == sorted(rows)


def test_steps_must_be_positive():
  p = _run("--steps", "0")
  assert p.returncode != 0 and "--steps" in p.stderr


def test_product_arm_fails_loudly_without_cuda():
  if torch.cuda.is_available():
    return  # on a GPU box the product arm is exercised by the driver itself
  p = _run("--steps", "1", "--warmup", "1")
  assert p.returncode != 0
  assert "cuda" in (p.stderr + p.stdout).lower()
