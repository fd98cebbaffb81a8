"""GPU parity: every C-ABI entry point and the two orchestrators against the
CPU oracle and the committed golden fixtures (DYN_PREC_FP32 mode)."""

import pytest
import torch

import scenes
from dynibar_b200 import synthetic
from oracle import dynibar_oracle as orc
from util import assert_close_frac

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture
def rr():
  """every test of this module runs in the fp32 parity mode (the library default is bf16)"""
  from dynibar_b200 import render_ray
  with render_ray.precision_scope("fp32"):
    yield render_ray


def _dev(x):
  return synthetic.to_device(x, DEV)


def _cmp_ray_diff(name, got, want):
  """ray_diff = [normalize(a - b), a.b] for unit vectors a, b (projection.py:85-100).
  The direction part is ill-conditioned when a ~= b (fp32 cancellation in a - b
  is amplified by 1/|a-b|), so its tolerance scales with 1/|a-b| = 1/sqrt(2-2 a.b);
  the dot product is compared tightly."""
  got, want = got.cpu(), want.cpu()
  assert_close_frac(name + ".dot", got[..., 3], want[..., 3], rtol=1e-5, atol=2e-6)
  nrm = torch.sqrt(torch.clamp(2 - 2 * want[..., 3:4].double(), min=1e-12)).float()
  err = (got[..., :3] - want[..., :3]).abs()
  assert (err <= 1e-5 + 5e-6 / nrm).all(), "%s.dir: max err %.3e" % (name, err.max().item())


@pytest.mark.parametrize("inv_uniform", [True, False])
@pytest.mark.parametrize("det", [True, False])
def test_sample_along_camera_ray(rr, inv_uniform, det):
  torch.manual_seed(0)
  R, S = 37, 64
  o, d = torch.randn(R, 3), torch.randn(R, 3)
  dr = torch.tensor([[0.7, 41.0]])
  jit = None if det else torch.rand(R, S)
  want = orc.sample_along_ray(o, d, dr, S, inv_uniform, jit)
  got = rr.sample_along_camera_ray(_dev(o), _dev(d), _dev(dr), S, inv_uniform, det,
                                   None if det else _dev(jit))
  for g, w, n in zip(got, want, ("pts", "z", "s")):
    assert_close_frac(n, g, w, rtol=1e-6, atol=1e-6)
  assert torch.equal(got[1].cpu(), want[1]), "z_vals must be bit-exact"


@pytest.mark.parametrize("name", list(scenes.GOLDEN_CONFIGS))
def test_stages_against_golden(rr, golden, name):
  """motion coefficients, displaced points, projector outputs, net outputs on
  the reference's own stage-boundary tensors."""
  from dynibar_b200.projection import Projector
  fx = golden(name)
  cfg, st = fx["cfg"], fx["stages"]
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  b, fc, m = _dev(batch), _dev(feat_c), synthetic.model_to(model, DEV)
  tt = float(t[0].float())
  pts = _dev(st["pts"])
  coeff = rr.motion_coefficients(m.motion_mlp, pts, tt)
  assert_close_frac("coeff", coeff, st["coeff"], rtol=1e-4, atol=1e-6)
  seq = rr.displaced_points(pts, _dev(st["coeff"]), m.trajectory_basis, frame[0], offs[0],
                            cfg["num_vv"])
  assert_close_frac("seq", seq, st["seq"], rtol=1e-6, atol=1e-6)
  P = Projector(DEV)
  f, rd, mk = P.compute_with_motions(pts, _dev(st["seq"]), b["camera"], b["src_rgbs"],
                                     b["src_cameras"], fc[0])
  assert_close_frac("mask_dy", mk, st["mask_dy"], max_bad_frac=1e-3)
  assert_close_frac("rgb_feat_dy", f, st["rgb_feat_dy"], rtol=1e-4, atol=2e-5, max_bad_frac=1e-3)
  _cmp_ray_diff("ray_diff_dy", rd, st["ray_diff_dy"])
  # the public compute_angle (projection.py:61-101), called the way compute_with_motions calls it
  # (static point expanded over the views) and with the un-expanded point
  seq_d = _dev(st["seq"])
  for xyz_st in (pts[None].expand(seq_d.shape[0], -1, -1, -1), pts[None]):
    ang = P.compute_angle(xyz_st, seq_d, b["camera"][0], b["src_cameras"][0])
    assert ang.shape == seq_d.shape[:-1] + (4,)
    _cmp_ray_diff("compute_angle", ang.permute(1, 2, 0, 3), st["ray_diff_dy"])
  V_st = b["static_src_rgbs"].shape[1]
  f, rd, mk = P.compute_with_motions(pts, pts[None].repeat(V_st, 1, 1, 1), b["camera"],
                                     b["static_src_rgbs"], b["static_src_cameras"], fc[2])
  assert_close_frac("mask_st", mk, st["mask_st"], max_bad_frac=1e-3)
  assert_close_frac("rgb_feat_st", f, st["rgb_feat_st"], rtol=1e-4, atol=2e-5, max_bad_frac=1e-3)
  _cmp_ray_diff("ray_diff_st", rd, st["ray_diff_st"])
  assert_close_frac("ref_plucker", rr.compute_ref_plucker_coordinate(b["ray_o"], b["ray_d"]),
                    st["ref_plucker"], rtol=1e-5, atol=1e-6)
  assert_close_frac("src_plucker", rr.compute_src_plucker_coordinate(pts, b["static_src_cameras"]),
                    st["src_plucker"], rtol=1e-5, atol=1e-6)
  # networks on the reference's inputs; compare where >= 1 view is valid
  ray_dir = torch.nn.functional.normalize(b["ray_d"], dim=-1)
  raw_dy = m.net_coarse_dy(pts, _dev(st["rgb_feat_dy"]), ray_dir, None, None, _dev(st["mask_dy"]),
                           torch.tensor([tt]))
  raw_st = m.net_coarse_st(pts, _dev(st["ref_plucker"]), _dev(st["src_plucker"]),
                           _dev(st["rgb_feat_st"]), ray_dir, _dev(st["ray_diff_st"]),
                           _dev(st["mask_st"]))
  for br, raw in (("dy", raw_dy), ("st", raw_st)):
    valid = (st["mask_" + br].sum(2) > 0).expand(-1, -1, 4)
    # (a few samples sit on the mask_rgb / in-bounds discontinuities: their blending softmax
    #  differs in the 3rd digit; everything else must meet the tolerance)
    assert_close_frac("raw_" + br, raw.cpu()[valid], st["raw_" + br][valid], rtol=2e-4, atol=2e-5,
                      max_bad_frac=5e-3)
    inval = ~valid[..., 3]
    assert (raw.cpu()[..., 3][inval] == -1e9).all()


def test_motion_mlp_forward_module_call(rr):
  model, _ = synthetic.make_model(16, 16, seed=3)
  x = torch.randn(5, 7, 4)
  want = orc.motion_mlp(orc._sd(model.motion_mlp), x)
  got = synthetic.model_to(model, DEV).motion_mlp(x.to(DEV))
  assert_close_frac("motion", got, want, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("S", [16, 64, 128, 100])
def test_composite_dicts(rr, S):
  from dynibar_b200 import autograd as ag
  torch.manual_seed(S)
  R, Va, Vb = 53, 7, 5
  raw_a, raw_b = torch.randn(R, S, 4), torch.randn(R, S, 4)
  raw_a[..., 3] = raw_a[..., 3] * 3 - 2
  raw_b[..., 3] = raw_b[..., 3] * 3 - 2
  raw_a[3, :, 3] = -1e9  # a ray with no valid dynamic sample
  raw_b[4, 5:, 3] = 30.0  # saturating density (softplus threshold branch)
  z = torch.sort(torch.rand(R, S) * 20 + 1, -1)[0]
  ma = (torch.rand(R, S, Va) > 0.4).float()
  mb = (torch.rand(R, S, Vb) > 0.6).float()
  ma[7] = 0
  want = orc.composite(raw_a, raw_b, z, ma.sum(2) > 1, mb.sum(2) > 1)
  got = ag.composite(_dev(raw_a), _dev(raw_b), _dev(z), _dev(ma), _dev(mb), 1, 1)
  assert list(got.keys()) == list(want.keys())
  for k in want:
    assert_close_frac(k, got[k], want[k], rtol=1e-5, atol=1e-6)
  want = orc.composite_vanilla(raw_a, z, ma.sum(2) > 0)
  got = ag.composite_vanilla(_dev(raw_a), _dev(z), _dev(ma), 0)
  assert list(got.keys()) == list(want.keys())
  for k in want:
    assert_close_frac(k, got[k], want[k], rtol=1e-5, atol=1e-6)
  # reference-signature wrappers ([R,S] bool masks)
  got = rr.raw2outputs(_dev(raw_a), _dev(raw_b), _dev(z), _dev(ma.sum(2) > 1), _dev(mb.sum(2) > 1))
  want = orc.composite(raw_a, raw_b, z, ma.sum(2) > 1, mb.sum(2) > 1)
  for k in want:
    assert_close_frac(k, got[k], want[k], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("inv_uniform", [True, False])
@pytest.mark.parametrize("det", [True, False])
def test_resample(rr, inv_uniform, det):
  torch.manual_seed(5)
  R, S, Ni = 61, 64, 64
  z = orc.sample_along_ray(torch.zeros(R, 3), torch.ones(R, 3), torch.tensor([[1.0, 30.0]]), S,
                           inv_uniform)[1]
  w = torch.rand(R, S) ** 4
  w[0] = 0           # uniform pdf
  w[1] = 0; w[1, 20] = 1.0  # single spike
  u = None if det else torch.rand(R, Ni)
  want = orc.resample_depths(z, w.clone(), Ni, inv_uniform, u)
  got = rr.resample_depths(_dev(z), _dev(w), Ni, inv_uniform, det, None if det else _dev(u))
  assert torch.all(got[:, 1:] >= got[:, :-1]), "fine depths must be sorted"
  assert_close_frac("z_fine", got, want, rtol=2e-5, atol=1e-6, max_bad_frac=2e-3)


def _run_both(rr, cfg, mono, det=True, seed_draws=None):
  from dynibar_b200.projection import Projector
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  b, fc, ff = _dev(batch), _dev(feat_c), _dev(feat_f)
  m = synthetic.model_to(model, DEV)
  if mono:
    got = rr.render_rays_mono(frame, t, offs, b, m, fc, Projector(DEV), cfg["N_samples"], args,
                              inv_uniform=cfg["inv_uniform"], det=True,
                              is_train=cfg.get("anchor_offset") is not None, num_vv=cfg["num_vv"])
  else:
    kw = {}
    if not det:
      kw = dict(jitter=_dev(seed_draws[0]), u=_dev(seed_draws[1]))
    got = rr.render_rays_mv(frame, t, offs, b, m, Projector(DEV), fc, ff, cfg["N_samples"], args,
                            inv_uniform=cfg["inv_uniform"], N_importance=cfg["N_importance"],
                            det=det, is_train=False, **kw)
  return got


@pytest.mark.parametrize("name", list(scenes.GOLDEN_CONFIGS))
def test_render_rays_against_golden(rr, golden, name):
  fx = golden(name)
  cfg = fx["cfg"]
  got = _run_both(rr, cfg, cfg["mono"])
  keys = (("outputs_coarse_ref", "outputs_coarse_ref_dy", "outputs_coarse_st") if cfg["mono"]
          else ("outputs_coarse_ref", "outputs_fine_ref", "outputs_fine_ref_dy"))
  if cfg.get("anchor_offset") is not None:  # cross-time branch (row a16)
    keys += ("outputs_coarse_anchor", "outputs_coarse_anchor_dy")
  for k in keys:
    assert list(got[k].keys()) == list(fx[k].keys()), k
    for kk, want in fx[k].items():
      assert got[k][kk].shape == want.shape and got[k][kk].dtype == want.dtype, (k, kk)
      assert_close_frac("%s/%s" % (k, kk), got[k][kk], want, rtol=5e-4, atol=5e-5,
                        max_bad_frac=0.03 if cfg.get("stress") else 1e-3)
  assert got["outputs_coarse"] is None and got["outputs_fine"] is None
  if not cfg["mono"]:
    assert got["outputs_fine_anchor"] is None and got["outputs_fine_anchor_dy"] is None
    rgb = got["outputs_fine_ref"]["rgb"].cpu()
    assert orc.psnr(rgb, fx["outputs_fine_ref"]["rgb"]) > 60.0


def test_render_rays_mv_random_sampling_against_golden(rr, golden):
  fx = golden("mv_small")
  cfg = fx["cfg"]
  R = cfg["rays"]
  torch.manual_seed(cfg["seed"] + 1000)
  draws = (torch.rand(R, cfg["N_samples"]), torch.rand(R, cfg["N_importance"]))
  got = _run_both(rr, cfg, False, det=False, seed_draws=draws)
  for kk, want in fx["rand_outputs_fine_ref"].items():
    assert_close_frac(kk, got["outputs_fine_ref"][kk], want, rtol=5e-4, atol=5e-5,
                      max_bad_frac=0.03)


def test_full_size_properties(rr):
  """BASELINE config-2 shape on one chunk (8192 rays would take the fp32 path a
  while; 1024 rays of the real 512x288 / 64+64 / 8+8 configuration): rays are
  independent, so (i) a permutation of the rays permutes the outputs, (ii)
  splitting the chunk gives identical results, (iii) weights are a
  sub-probability distribution and fine depths are sorted."""
  from dynibar_b200.projection import Projector
  cfg = dict(mono=False, H=288, W=512, V_dy=8, V_st=8, rays=1024, N_samples=64, N_importance=64,
             num_vv=0, inv_uniform=True, anti_alias_pooling=1, mask_rgb=0, seed=21, stress=False)
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  b, fc, ff = _dev(batch), _dev(feat_c), _dev(feat_f)
  m = synthetic.model_to(model, DEV)

  def run(bb):
    return rr.render_rays_mv(frame, t, offs, bb, m, Projector(DEV), fc, ff, 64, args,
                             inv_uniform=True, N_importance=64, det=True, is_train=False)

  full = run(b)["outputs_fine_ref"]
  perm = torch.randperm(1024, device=DEV)
  bp = dict(b)
  for k in ("ray_o", "ray_d", "uv_grid"):
    bp[k] = b[k][perm].contiguous()
  permuted = run(bp)["outputs_fine_ref"]
  for k in ("rgb", "depth", "weights", "z_vals"):
    assert torch.equal(permuted[k], full[k][perm]), k
  half = dict(b)
  for k in ("ray_o", "ray_d", "uv_grid"):
    half[k] = b[k][:300].contiguous()
  part = run(half)["outputs_fine_ref"]
  for k in ("rgb", "depth", "weights"):
    assert torch.equal(part[k], full[k][:300]), k
  w = full["weights"]
  assert (w >= 0).all() and (w.sum(1) <= 1 + 1e-4).all()
  z = full["z_vals"]
  assert (z[:, 1:] >= z[:, :-1]).all() and z.shape == (1024, 128)
  assert torch.isfinite(full["rgb"]).all() and full["mask"].dtype == torch.bool


def test_render_single_image_driver(rr, golden):
  """Frame driver (render_image.py:9-217): same structure as the reference's (CPU tensors
  reshaped to [H,W,...], rgb zeroed where mask == 0) and identical to one un-chunked call."""
  from dynibar_b200.projection import Projector
  from dynibar_b200.render_image import render_single_image_nvi
  cfg = dict(scenes.GOLDEN_CONFIGS["mv_small"], rays=None, H=12, W=16)
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(cfg)
  b, fc, ff = _dev(batch), _dev(feat_c), _dev(feat_f)
  m = synthetic.model_to(model, DEV)
  sampler = type("S", (), {"H": 12, "W": 16})()
  ret = render_single_image_nvi(frame, t, offs, sampler, b, m, Projector(DEV), 50, cfg["N_samples"], args,
                                inv_uniform=True, N_importance=cfg["N_importance"], det=True,
                                coarse_featmaps=fc, fine_featmaps=ff, is_train=False)
  assert list(ret.keys()) == ["outputs_fine_anchor", "outputs_fine_ref", "outputs_coarse_ref", "outputs_fine"]
  one = rr.render_rays_mv(frame, t, offs, b, m, Projector(DEV), fc, ff, cfg["N_samples"], args,
                          inv_uniform=True, N_importance=cfg["N_importance"], det=True, is_train=False)
  f = ret["outputs_fine_ref"]
  assert not f["rgb"].is_cuda and f["rgb"].shape == (12, 16, 3) and f["depth"].shape == (12, 16)
  assert f["weights"].shape == (12, 16, 32) and f["render_flows"].shape == (7, 12, 16, 2)
  want = one["outputs_fine_ref"]["rgb"].cpu().masked_fill(~one["outputs_fine_ref"]["mask"].cpu()[:, None], 0.0)
  assert torch.equal(f["rgb"].reshape(-1, 3), want)
  assert torch.equal(f["depth"].reshape(-1), one["outputs_fine_ref"]["depth"].cpu())
