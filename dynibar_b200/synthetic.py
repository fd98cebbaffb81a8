"""Seeded synthetic scenes for tests and bench (no files, no network).

Construction follows SURVEY.md 8(d): a pinhole target camera at the origin,
source cameras translated along x, uniform-random source images, Gaussian
feature maps, DCT trajectory basis, default-init networks with a non-zero
`coeff_linear` (otherwise motion is identically 0, mlp_network.py:602-603) and
a negative density bias (otherwise every ray saturates at its first sample).
No tensor dimension other than xyz equals 3 (reference `torch.cross` hazard,
render_ray.py:375,392).
"""

from types import SimpleNamespace

import numpy as np
import torch

from dynibar_b200 import mlp_network as nets


def init_dct_basis(num_basis, num_frames):
  """DCT-II trajectory basis [T,K] (ibrnet/model.py:18-30), vectorised."""
  t = torch.arange(num_frames, dtype=torch.float64)[:, None]
  k = torch.arange(1, num_basis + 1, dtype=torch.float64)[None, :]
  b = np.sqrt(2.0 / num_frames) * torch.cos(np.pi / (2.0 * num_frames) * (2 * t + 1) * k)
  return b.float()


def camera_vector(H, W, K, c2w):
  """34-float camera: [h, w, K(4x4 row-major), c2w(4x4 row-major)]
  (eval_nvidia.py:81-83; parsed at sample_ray.py:11-16, projection.py:38-41)."""
  return torch.cat([torch.tensor([float(H), float(W)]), K.reshape(-1), c2w.reshape(-1)])


def make_args(anti_alias_pooling=1, mask_rgb=0, occ_weights_mode=0):
  return SimpleNamespace(anti_alias_pooling=anti_alias_pooling, mask_rgb=mask_rgb,
                         input_dir=True, input_xyz=False,
                         occ_weights_mode=occ_weights_mode, num_basis=6)


def make_cameras(H, W, V_dy, V_st, focal_scale=0.78, stress=False):
  """`stress=True` pushes one dynamic camera far sideways (mostly out of
  bounds) and moves the last static camera forward to z=+4 (near samples are
  behind it) so fixtures exercise the in-front / in-bounds masks and points
  with zero valid views."""
  f = focal_scale * W
  K = torch.eye(4)
  K[0, 0] = f
  K[1, 1] = f
  K[0, 2] = W / 2.0
  K[1, 2] = H / 2.0
  tgt = camera_vector(H, W, K, torch.eye(4))[None]

  def rig(V, spacing):
    cams = []
    for i in range(V):
      c2w = torch.eye(4)
      c2w[0, 3] = spacing * (i - V / 2.0)
      # small generic y/z offsets: with a pure-x rig the first/last pixel rows
      # project EXACTLY onto the source image border and the in-bounds test
      # becomes a coin flip under fp32 rounding
      c2w[1, 3] = 0.013 * (i - V / 2.0) + 0.007
      c2w[2, 3] = 0.011 * ((i * 7) % 5 - 2) + 0.003
      cams.append(c2w)
    return cams

  dy, st = rig(V_dy, 0.05), rig(V_st, 0.08)
  if stress:
    dy[0][0, 3] = -1.5
    st[-1][2, 3] = 4.0
    st[0][0, 3] = 2.5
  pack = lambda cs: torch.stack([camera_vector(H, W, K, c) for c in cs])[None]
  return K, tgt, pack(dy), pack(st)


def time_offsets(V_dy, num_vv=0):
  """`V_dy - num_vv` temporal offsets: a sorted symmetric subset of [-3..3]
  (7 views = eval_nvidia.py:92-94), extended with 0-offset duplicates."""
  order = [-1, 1, -2, 2, -3, 3, 0]
  n = V_dy - num_vv
  return sorted(order[:min(n, 7)]) + [0] * max(0, n - 7)


def make_scene(H=288, W=512, V_dy=8, V_st=8, C=32, num_frames=24, frame_idx=10,
               num_vv=0, seed=0, near=1.0, far=30.0, rays=None, stress=False, anchor_offset=None):
  """Returns (ray_batch, featmaps_coarse, featmaps_fine, frame/time tuples).
  `rays`: None -> all H*W pixel rays; int n -> first n rays of a seeded
  permutation (keeps fixtures small)."""
  g = torch.Generator().manual_seed(seed)
  K, tgt, cams_dy, cams_st = make_cameras(H, W, V_dy, V_st, stress=stress)
  from dynibar_b200.sample_ray import pixel_rays
  ray_o, ray_d, uv = pixel_rays(H, W, K, torch.eye(4))
  if rays is not None:
    sel = torch.randperm(H * W, generator=g)[:rays]
    ray_o, ray_d, uv = ray_o[sel], ray_d[sel], uv[sel]
  h4, w4 = H // 4, W // 4
  batch = {
      "ray_o": ray_o, "ray_d": ray_d, "uv_grid": uv,
      "depth_range": torch.tensor([[near, far]]),
      "camera": tgt,
      "src_rgbs": torch.rand(1, V_dy, H, W, 3, generator=g),
      "src_cameras": cams_dy,
      "static_src_rgbs": torch.rand(1, V_st, H, W, 3, generator=g),
      "static_src_cameras": cams_st,
  }
  def fm():
    return (torch.randn(V_dy, C, h4, w4, generator=g), None,
            torch.randn(V_st, C, h4, w4, generator=g))
  feat_c, feat_f = fm(), fm()
  frame = (frame_idx, None)
  t = (torch.tensor([frame_idx / num_frames], dtype=torch.float64), None)
  offs = (time_offsets(V_dy, num_vv), None)
  if anchor_offset is not None:
    # cross-time (training) inputs: a second set of dynamic source views around the
    # anchor frame (train.py:264-281 builds featmaps[1] from `anchor_src_rgbs`)
    _, _, cams_an, _ = make_cameras(H, W, V_dy, V_st, stress=False)
    cams_an = cams_an.clone()
    cams_an[0, :, 18 + 3] += 0.021  # shift the anchor rig a little in x
    batch["anchor_src_rgbs"] = torch.rand(1, V_dy, H, W, 3, generator=g)
    batch["anchor_src_cameras"] = cams_an
    batch["anchor_camera"] = tgt
    feat_c = (feat_c[0], torch.randn(V_dy, C, h4, w4, generator=g), feat_c[2])
    a_idx = frame_idx + anchor_offset
    frame = (frame_idx, a_idx)
    t = (t[0], torch.tensor([a_idx / num_frames], dtype=torch.float64))
    offs = (offs[0], time_offsets(V_dy, num_vv))
  return batch, feat_c, feat_f, frame, t, offs


def make_supervision(batch, n_flow=6, seed=0):
  """`batch` plus seeded per-ray supervision in the layout RaySamplerSingleImage.random_sample returns
  (sample_ray.py:262-331): rgb [R,3] in [0,1), disp [R], binary motion_mask / static_mask [R], flows [n_flow,R,2]
  and binary masks [n_flow,R,1], on the device of batch['ray_o']."""
  R = batch["ray_o"].shape[0]
  g = torch.Generator().manual_seed(seed)
  sup = {
      "rgb": torch.rand(R, 3, generator=g),
      "disp": torch.rand(R, generator=g) * 0.9 + 0.05,
      "motion_mask": (torch.rand(R, generator=g) > 0.5).float(),
      "static_mask": (torch.rand(R, generator=g) > 0.6).float(),
      "flows": torch.randn(n_flow, R, 2, generator=g) * 2.0,
      "masks": (torch.rand(n_flow, R, 1, generator=g) > 0.3).float(),
  }
  out = dict(batch)
  out.update(to_device(sup, batch["ray_o"].device))
  return out


def make_model(N_samples=64, N_importance=64, num_frames=24, args=None, seed=0,
               mono=False, sigma_bias=-4.0, coeff_std=1e-2):
  """Duck-typed model namespace with the attributes render_rays_* read
  (render_ray.py:683-698, :749, :766, :852-855)."""
  args = args or make_args()
  torch.manual_seed(seed)
  m = SimpleNamespace()
  shift = 5.0 if mono else 0.0  # ibrnet/model.py:307
  m.net_coarse_dy = nets.DynibarDynamic(args, 32, N_samples, shift=shift)
  m.net_coarse_st = nets.DynibarStatic(args, 32, N_samples)
  m.motion_mlp = nets.MotionMLP(num_basis=6)
  m.trajectory_basis = init_dct_basis(6, num_frames)
  mods = [m.net_coarse_dy, m.net_coarse_st, m.motion_mlp]
  if not mono:
    m.net_fine_dy = nets.DynibarDynamic(args, 32, N_samples + N_importance)
    m.net_fine_st = nets.DynibarStatic(args, 32, N_samples + N_importance)
    m.motion_mlp_fine = nets.MotionMLP(num_basis=6)
    m.trajectory_basis_fine = init_dct_basis(6, num_frames)
    mods += [m.net_fine_dy, m.net_fine_st, m.motion_mlp_fine]
  with torch.no_grad():
    for mod in mods:
      if isinstance(mod, nets.MotionMLP):
        mod.coeff_linear.weight.normal_(0.0, coeff_std)
      else:
        bias = sigma_bias + (shift if isinstance(mod, nets.DynibarDynamic) else 0.0)
        mod.out_geometry_fc[2].bias.fill_(bias)
      mod.requires_grad_(False)
  return m, args


def to_device(obj, device):
  if torch.is_tensor(obj):
    return obj.to(device)
  if isinstance(obj, dict):
    return {k: to_device(v, device) for k, v in obj.items()}
  if isinstance(obj, (tuple, list)):
    return type(obj)(to_device(v, device) for v in obj)
  return obj


def model_to(model, device):
  for k, v in vars(model).items():
    if isinstance(v, torch.nn.Module) or torch.is_tensor(v):
      setattr(model, k, v.to(device))
  return model
