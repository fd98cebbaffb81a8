"""RaySamplerSingleImage (row a1) against outputs of the unmodified reference class
(ibrnet/sample_ray.py:19-331; fixtures tests/golden/sampler.pt from make_golden_frame.py and
sampler_17x23.pt from make_golden_checks.py)."""

import os

import numpy as np
import pytest
import torch

import scenes
from dynibar_b200 import sample_ray as sr


def _data():
  fx = torch.load(os.path.join(os.path.dirname(__file__), "golden", "sampler.pt"), weights_only=False)
  cfg = fx["cfg"]
  batch = scenes.build(cfg)[0]
  return fx, cfg, scenes.sampler_data(batch, cfg["H"], cfg["W"], cfg["seed"])


def _same(name, got, want):
  assert set(k for k, v in got.items() if torch.is_tensor(v)) == set(want.keys()), name
  for k, w in want.items():
    g = got[k]
    assert g.shape == w.shape and g.dtype == w.dtype, (name, k, g.shape, w.shape)
    if k in ("ray_d",):  # (c2w K^-1) pix: same association, different kernels -> 1 ulp
      torch.testing.assert_close(g, w, rtol=1e-6, atol=1e-6, msg=lambda m: "%s/%s: %s" % (name, k, m))
    else:
      assert torch.equal(g, w), (name, k)


def test_get_all_matches_reference_fixture():
  fx, cfg, data = _data()
  s = sr.RaySamplerSingleImage(data, "cpu")
  assert (s.H, s.W) == (cfg["H"], cfg["W"])
  _same("get_all", s.get_all(), fx["get_all"])
  s2 = sr.RaySamplerSingleImage(data, "cpu", render_stride=2)
  got = s2.get_all()
  _same("stride2", {k: got[k] for k in ("ray_o", "ray_d", "uv_grid")}, fx["get_all_stride2"])


def test_random_sample_matches_reference_fixture():
  fx, cfg, data = _data()
  s = sr.RaySamplerSingleImage(data, "cpu")
  sr.rng = np.random.RandomState(234)  # the reference's module-level stream (sample_ray.py:8)
  _same("center", s.random_sample(40, "center", 0.8), fx["random_center"])
  assert torch.equal(torch.from_numpy(np.asarray(s.sample_random_pixel(40, "center", 0.6))),
                     fx["random_center_inds"])
  r = s.random_sample(33, "uniform")
  _same("uniform", r, fx["random_uniform"])
  assert torch.equal(torch.from_numpy(np.asarray(r["selected_inds"])), fx["random_uniform_inds"])
  with pytest.raises(NotImplementedError):
    s.sample_random_pixel(4, "nope")


def test_sampler_matches_live_reference():
  """A 17x23 frame at render_stride 1 and 3 (tests/golden/sampler_17x23.pt from make_golden_checks.py)."""
  fx = torch.load(os.path.join(os.path.dirname(__file__), "golden", "sampler_17x23.pt"), weights_only=False)
  cfg = fx["cfg"]
  assert cfg == dict(scenes.GOLDEN_CONFIGS["mv_small"], H=17, W=23, rays=None, seed=91)
  batch = scenes.build(cfg)[0]
  data = scenes.sampler_data(batch, cfg["H"], cfg["W"], cfg["seed"])
  for stride in (1, 3):
    a = sr.RaySamplerSingleImage(data, "cpu", render_stride=stride).get_all()
    b = fx[stride]
    for k, w in b.items():
      if torch.is_tensor(w):
        torch.testing.assert_close(a[k], w, rtol=1e-6, atol=1e-6)
      else:
        assert a[k] is None and w is None, k
