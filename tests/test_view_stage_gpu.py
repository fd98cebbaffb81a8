"""The fused per-view kernel (csrc/view_twin3.cu: projection, gather, per-view MLP chain and pooling on
tcgen05, then the point stages and blending head) against the fp32 staged path on the same inputs, at view
counts that fill 8 and 16 view slots, ragged tails and stressed masks.  Differences come from the bf16 operands
of the tensor cores and the fp32 summation order inside them (tolerances of
test_tensorcore_gpu.py::test_fused_view_stage_matches_staged)."""

import pytest
import torch

from dynibar_b200 import _lib, synthetic
from util import assert_close_frac

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _inputs(V_dy, V_st, rays, S, seed, stress=False, mask_rgb=0):
  from dynibar_b200 import render_ray as rr
  batch, feat_c, feat_f, frame, t, offs = synthetic.make_scene(H=72, W=96, V_dy=V_dy, V_st=V_st, rays=rays,
                                                               seed=seed, stress=stress)
  args = synthetic.make_args(1, mask_rgb)
  model, args = synthetic.make_model(S, 0, args=args, seed=seed, mono=True)
  d = lambda x: synthetic.to_device(x, DEV)
  b, fc = d(batch), d(feat_c)
  m = synthetic.model_to(model, DEV)
  pts, z, s = rr.sample_along_camera_ray(b["ray_o"], b["ray_d"], b["depth_range"], S, True, True)
  g = torch.Generator(device=DEV).manual_seed(seed)
  seq = pts[None] + 0.02 * torch.randn(V_dy, rays, S, 3, device=DEV, generator=g)
  return b, fc, m, pts, seq, float(t[0].float())


def _run_fused(b, fc, m, pts, seq, tt):
  from dynibar_b200 import render_ray as rr
  ray_dir = torch.nn.functional.normalize(b["ray_d"], dim=-1)
  raw_st, m_st = rr.net_static_fused(m.net_coarse_st, pts, b["ray_o"], b["ray_d"], b["camera"],
                                     b["static_src_rgbs"], b["static_src_cameras"],
                                     rr.featmaps_channels_last(fc[2]))
  raw_dy, m_dy = rr.net_dynamic_fused(m.net_coarse_dy, pts, seq, ray_dir, b["camera"], b["src_rgbs"],
                                      b["src_cameras"], rr.featmaps_channels_last(fc[0]), tt)
  torch.cuda.synchronize()
  return raw_st, m_st, raw_dy, m_dy


def _run_staged(b, fc, m, pts, seq, tt):
  """The fp32 staged evaluation of render_ray._render_pass (gather, then one kernel per layer)."""
  from dynibar_b200 import render_ray as rr
  from dynibar_b200.projection import project_gather
  with rr.precision_scope("fp32"):
    ref_plucker = rr.compute_ref_plucker_coordinate(b["ray_o"], b["ray_d"])
    f_dy, _, m_dy = project_gather(pts, seq, b["camera"], b["src_rgbs"], b["src_cameras"], fc[0])
    f_st, rd_st, m_st = project_gather(pts, None, b["camera"], b["static_src_rgbs"], b["static_src_cameras"],
                                       fc[2])
    raw_dy = rr.net_dynamic_forward(m.net_coarse_dy, pts, f_dy, ref_plucker[:, :3], m_dy, tt)
    raw_st = rr.net_static_forward(m.net_coarse_st, pts, ref_plucker,
                                   rr.compute_src_plucker_coordinate(pts, b["static_src_cameras"]),
                                   f_st, rd_st, m_st)
  torch.cuda.synchronize()
  return raw_st, m_st, raw_dy, m_dy


@pytest.mark.parametrize("V_dy,V_st,rays,S,stress,mask_rgb", [
    (8, 8, 300, 64, False, 0),     # the benchmark's view counts, several 256-row iterations, ragged tail
    (7, 11, 130, 32, True, 1),     # eval_nvidia.py:92-119 view counts: 8 and 16 view slots, masks stressed
    (10, 15, 70, 64, False, 1),    # BASELINE config 4
    (3, 2, 33, 16, True, 0),       # tiny: a single partially filled tile
    (16, 16, 40, 32, False, 0),    # full 16-slot groups
])
def test_view_stage_matches_staged(V_dy, V_st, rays, S, stress, mask_rgb):
  inp = _inputs(V_dy, V_st, rays, S, seed=V_dy * 100 + V_st, stress=stress, mask_rgb=mask_rgb)
  f_st, fm_st, f_dy, fm_dy = _run_fused(*inp)
  s_st, sm_st, s_dy, sm_dy = _run_staged(*inp)
  assert_close_frac("mask_st", fm_st, sm_st, max_bad_frac=1e-3)
  assert_close_frac("mask_dy", fm_dy, sm_dy, max_bad_frac=1e-3)
  for br, got, want, mask in (("st", f_st, s_st, sm_st), ("dy", f_dy, s_dy, sm_dy)):
    assert torch.isfinite(got[..., :3]).all()
    valid = (mask.sum(2) > 0)[..., 0]
    assert (got[..., 3][~valid] == -1e9).all()
    assert_close_frac("rgb_" + br, got[..., :3][valid], want[..., :3][valid], rtol=0, atol=1e-2,
                      max_bad_frac=5e-3)
    assert_close_frac("sigma_" + br, got[..., 3][valid], want[..., 3][valid], rtol=0, atol=2e-2,
                      max_bad_frac=5e-3)


def test_view_stage_is_deterministic_and_chunk_invariant():
  """rows are independent: evaluating a prefix of the rays gives bit-identical results (different
  grid size, different tile pairing), and repeated launches are bit-identical."""
  b, fc, m, pts, seq, tt = _inputs(8, 8, 520, 32, seed=5)
  full = _run_fused(b, fc, m, pts, seq, tt)
  again = _run_fused(b, fc, m, pts, seq, tt)
  for x, y in zip(full, again):
    assert torch.equal(x, y)
  n = 200
  bs = dict(b)
  for k in ("ray_o", "ray_d", "uv_grid"):
    bs[k] = b[k][:n].contiguous()
  part = _run_fused(bs, fc, m, pts[:n].contiguous(), seq[:, :n].contiguous(), tt)
  for x, y in zip(full, part):
    assert torch.equal(x[:n], y)


@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_removed_view_kernel_variants_fail_loudly(kernel):
  """The ids of the removed comparison variants make the fused per-view call fail (instead of timing the
  library's kernel under their name); -1 restores it."""
  inp = _inputs(3, 2, 33, 16, seed=7)
  try:
    _lib.lib.dyn_debug_set_view_kernel(kernel)
    with pytest.raises(RuntimeError, match="was removed"):
      _run_fused(*inp)
  finally:
    _lib.lib.dyn_debug_set_view_kernel(-1)
  raw_st, _, raw_dy, _ = _run_fused(*inp)
  assert torch.isfinite(raw_st).all() and torch.isfinite(raw_dy).all()
