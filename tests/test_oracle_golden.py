"""Pin the CPU oracle (oracle/dynibar_oracle.py) against the reference.

Against committed golden fixtures: outputs of the unmodified reference
(tests/golden/make_golden.py, make_golden_checks.py).
"""

import pytest
import torch

import scenes
from oracle import dynibar_oracle as orc
from util import assert_close_frac

TOL = dict(rtol=2e-4, atol=2e-5)


def _cmp(name, got, want, rtol=2e-4, atol=2e-5):
  if want.dtype == torch.bool:
    assert torch.equal(got, want), name
    return
  torch.testing.assert_close(got, want, rtol=rtol, atol=atol, msg=lambda m: name + ": " + m)


def _checksum(batch, feats):
  acc = 0.0
  for k in sorted(batch):
    if torch.is_tensor(batch[k]):
      acc += float(batch[k].double().abs().sum())
  for f in feats:
    for x in f:
      if x is not None:
        acc += float(x.double().abs().sum())
  return acc


@pytest.mark.parametrize("name", list(scenes.GOLDEN_CONFIGS))
def test_oracle_matches_golden(name, golden):
  fx = golden(name)
  cfg = fx["cfg"]
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  assert abs(_checksum(batch, [feat_c, feat_f]) - fx["checksum"]) < 1e-6 * fx["checksum"], \
      "seeded inputs drifted from the ones the fixture was generated with"
  with torch.no_grad():
    if cfg["mono"]:
      train = cfg.get("anchor_offset") is not None
      ret = orc.render_rays_mono(frame, t, offs, batch, model, feat_c, None,
                                 cfg["N_samples"], args, inv_uniform=cfg["inv_uniform"],
                                 det=True, is_train=train, num_vv=cfg["num_vv"],
                                 return_aux=True)
      keys = ("outputs_coarse_ref", "outputs_coarse_ref_dy", "outputs_coarse_st")
      if train:  # cross-time branch, render_ray.py:1099-1270
        keys += ("outputs_coarse_anchor", "outputs_coarse_anchor_dy")
      aux = ret["_aux"]
    else:
      ret = orc.render_rays_mv(frame, t, offs, batch, model, None, feat_c, feat_f,
                               cfg["N_samples"], args, inv_uniform=cfg["inv_uniform"],
                               N_importance=cfg["N_importance"], det=True,
                               is_train=False, return_aux=True)
      keys = ("outputs_coarse_ref", "outputs_fine_ref", "outputs_fine_ref_dy")
      aux = ret["_aux_coarse"]
  for k in keys:
    assert list(ret[k].keys()) == list(fx[k].keys()), k
    for kk in fx[k]:
      _cmp("%s/%s" % (k, kk), ret[k][kk], fx[k][kk])
  st = fx["stages"]
  _cmp("coeff", aux["coeff"], st["coeff"])
  _cmp("seq", aux["seq"], st["seq"])
  _cmp("rgb_feat_dy", aux["rgb_feat_dy"], st["rgb_feat_dy"])
  _cmp("rgb_feat_st", aux["rgb_feat_st"], st["rgb_feat_st"])
  _cmp("ray_diff_st", aux["ray_diff_st"], st["ray_diff_st"])
  _cmp("mask_dy", aux["mask_dy"], st["mask_dy"])
  _cmp("mask_st", aux["mask_st"], st["mask_st"])
  # raw is compared where the point has >= 1 valid view (SURVEY App. B 5.ii)
  for br in ("dy", "st"):
    valid = (st["mask_" + br].sum(2) > 0).expand(-1, -1, 4)
    _cmp("raw_" + br, aux["raw_" + br][valid], st["raw_" + br][valid])


@pytest.mark.parametrize("name", list(scenes.OCC_MODE_CONFIGS))
def test_oracle_occlusion_weight_modes_match_golden(name, golden):
  """occ_weights_mode 1 / 2 of the cross-time branch (render_ray.py:1243-1252)."""
  fx = golden("occ_modes")[name]
  cfg = fx["cfg"]
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  assert abs(_checksum(batch, [feat_c, feat_f]) - fx["checksum"]) < 1e-6 * fx["checksum"]
  with torch.no_grad():
    ret = orc.render_rays_mono(frame, t, offs, batch, model, feat_c, None, cfg["N_samples"], args,
                               inv_uniform=cfg["inv_uniform"], det=True, is_train=True, num_vv=cfg["num_vv"])
  for k in ("outputs_coarse_anchor", "outputs_coarse_anchor_dy"):
    for kk, want in fx[k].items():
      _cmp("%s/%s" % (k, kk), ret[k][kk], want)


def test_oracle_random_sampling_matches_golden(golden):
  """det=False: the oracle takes the reference's random draws as inputs."""
  fx = golden("mv_small")
  cfg = fx["cfg"]
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  R = batch["ray_o"].shape[0]
  torch.manual_seed(cfg["seed"] + 1000)
  jitter = torch.rand(R, cfg["N_samples"])
  u = torch.rand(R, cfg["N_importance"])
  with torch.no_grad():
    ret = orc.render_rays_mv(frame, t, offs, batch, model, None, feat_c, feat_f,
                             cfg["N_samples"], args, inv_uniform=cfg["inv_uniform"],
                             N_importance=cfg["N_importance"], det=False,
                             is_train=False, jitter=jitter, u=u)
  # one fine sample of one ray projects within rounding of an image border and
  # flips its mask between the two fp32 evaluation orders -> allow 1 ray in 40
  for kk, want in fx["rand_outputs_fine_ref"].items():
    assert_close_frac(kk, ret["outputs_fine_ref"][kk], want, max_bad_frac=0.03)


def test_sample_pdf_edge_cases():
  # all-zero weights -> uniform pdf; single spike; u hitting cdf entries exactly
  bins = torch.linspace(0, 1, 9)[None].repeat(3, 1)
  w = torch.zeros(3, 8)
  w[1, 3] = 5.0
  w[2] = torch.arange(8).float()
  s = orc.sample_pdf(bins, w, 16)
  assert s.shape == (3, 16)
  assert torch.all(s[:, 1:] >= s[:, :-1] - 1e-6)
  assert torch.all((s >= 0) & (s <= 1))
  torch.testing.assert_close(s[0], torch.linspace(0, 1, 16), atol=1e-5, rtol=0)


def test_oracle_matches_live_reference(golden):
  """A scene none of the other fixtures uses (seed 77, 7 + 4 views), against the reference's render_rays_mv
  (tests/golden/mv_seed77.pt from make_golden_checks.py)."""
  fx = golden("mv_seed77")
  cfg = fx["cfg"]
  assert cfg == dict(scenes.GOLDEN_CONFIGS["mv_small"], seed=77, rays=16, V_dy=7, V_st=4)
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  assert abs(_checksum(batch, [feat_c, feat_f]) - fx["checksum"]) < 1e-6 * fx["checksum"]
  with torch.no_grad():
    got = orc.render_rays_mv(frame, t, offs, batch, model, None, feat_c, feat_f,
                             cfg["N_samples"], args, inv_uniform=True,
                             N_importance=cfg["N_importance"], det=True, is_train=False)
  for k in ("outputs_coarse_ref", "outputs_fine_ref", "outputs_fine_ref_dy"):
    assert list(got[k].keys()) == list(fx[k].keys()), k
    for kk in fx[k]:
      _cmp("%s/%s" % (k, kk), got[k][kk], fx[k][kk])


def test_oracle_encoder_matches_reference_fixture(golden):
  """oracle.encoder_forward (feature_network.py:302-311) against outputs of the unmodified reference ResNet
  (tests/golden/encoder.pt); it is the autograd reference of the encoder's backward kernels."""
  from dynibar_b200 import feature_network as fn
  fx = golden("encoder")
  torch.manual_seed(fx["seed"])
  m = fn.ResNet()
  with torch.no_grad():  # same initialisation as tests/test_encoder_gpu.py::_model
    for name, p in m.named_parameters():
      if name.endswith("bn1.weight") or name.endswith("bn2.weight") or name.endswith("downsample.1.weight"):
        p.uniform_(0.5, 1.5)
      elif name.endswith(".bias"):
        p.uniform_(-0.3, 0.3)
  g = torch.Generator().manual_seed(fx["seed"] + 1)
  x = torch.rand(*fx["shape"], generator=g)
  with torch.no_grad():
    c, f = orc.encoder_forward(m, x)
  torch.testing.assert_close(c, fx["coarse"], rtol=2e-4, atol=2e-4)
  torch.testing.assert_close(f, fx["fine"], rtol=2e-4, atol=2e-4)
