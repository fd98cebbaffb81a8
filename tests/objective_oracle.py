"""Torch restatement of the DynIBaR training objective -- the reference the tests hold dynibar_b200.criterion to.

Follows the reference line by line (file:line under google/dynibar @ 5412b55): the criteria of ibrnet/criterion.py,
utils.img2charbonier, the loss composition of train.py:300-458, the static-bootstrap loss of train.py:187-196 and
eff_distloss_native of torch_efficient_distloss (prefix-sum form).  Plain torch ops, so torch autograd gives the
gradients; it runs on CPU or CUDA tensors in the dtype of the predictions (fp64 for the precision checks).  The
masks the reference casts with `.float()` are cast to that dtype instead.  tests/golden/criterion.pt pins the
criterion functions to the unmodified reference.
"""

import torch

EPSILON = 0.001           # ibrnet/criterion.py:19
TINY_NUMBER = 1e-6        # utils.py:12
LOSS_DEFAULTS = dict(w_disp=5e-2, w_flow=5e-3, w_cycle=0.1, cycle_factor=0.1, anneal_cycle=False, w_reg=0.05,
                     w_skew_entropy=1e-3, w_distortion=1e-3, decay_rate=10.0, init_decay_epoch=150)  # config.py


def img2charbonier(x, y, mask=None, eps=0.001):
  """utils.py:32-39."""
  if mask is None:
    return torch.mean(torch.sqrt((x - y) ** 2 + eps ** 2))
  return torch.sum(torch.sqrt((x - y) ** 2 + eps ** 2) * mask.unsqueeze(-1)) / (
      torch.sum(mask) * x.shape[-1] + TINY_NUMBER)


def criterion(outputs, ray_batch, motion_mask=None):
  """Criterion.forward, criterion.py:25-38."""
  pred_rgb = outputs["rgb"]
  pred_mask = outputs["mask"].to(pred_rgb.dtype)
  if motion_mask is not None:
    pred_mask = pred_mask * motion_mask.to(pred_rgb.dtype)
  return img2charbonier(pred_rgb, ray_batch["rgb"], pred_mask, EPSILON)


def compute_temporal_rgb_loss(outputs, ray_batch, motion_mask=None):
  """criterion.py:42-56."""
  pred_rgb = outputs["rgb"]
  gt_rgb = ray_batch["rgb"]
  occ_weight_map = outputs["occ_weight_map"]
  pred_mask = outputs["mask"].to(pred_rgb.dtype)
  if motion_mask is not None:
    pred_mask = pred_mask * motion_mask
  final_w = pred_mask * occ_weight_map
  final_w = final_w.unsqueeze(-1).repeat(1, 3)
  return torch.sum(final_w * torch.sqrt((pred_rgb - gt_rgb) ** 2 + EPSILON ** 2)) / (torch.sum(final_w) + 1e-8)


def compute_rgb_loss(pred_rgb, ray_batch, pred_mask):
  """criterion.py:58-62."""
  return img2charbonier(pred_rgb, ray_batch["rgb"], pred_mask, EPSILON)


def compute_flow_loss(render_flow, gt_flow, gt_mask):
  """criterion.py:83-85."""
  gt_mask_rep = gt_mask.repeat(1, 1, 2)
  return torch.sum(torch.abs(render_flow - gt_flow) * gt_mask_rep) / (torch.sum(gt_mask_rep) + 1e-8)


def eff_distloss_native(w, m, interval):
  """torch_efficient_distloss.eff_distloss_native: (1/3) mean sum delta w^2 + 2 mean sum_i (w_i m_i W_{i-1} -
  w_i WM_{i-1}), W / WM inclusive cumulative sums of w / w m."""
  loss_uni = (1 / 3) * (interval * w.pow(2)).sum(dim=-1).mean()
  wm = w * m
  w_cumsum = w.cumsum(dim=-1)
  wm_cumsum = wm.cumsum(dim=-1)
  loss_bi_0 = wm[..., 1:] * w_cumsum[..., :-1]
  loss_bi_1 = w[..., 1:] * wm_cumsum[..., :-1]
  loss_bi = 2 * (loss_bi_0 - loss_bi_1).sum(dim=-1).mean()
  return loss_bi + loss_uni


def eff_distloss_pairwise(w, m, interval):
  """mip-NeRF 360 definition: mean over rays of sum_ij w_i w_j |m_i - m_j| + (1/3) sum_i w_i^2 delta_i."""
  pair = (w[..., :, None] * w[..., None, :] * (m[..., :, None] - m[..., None, :]).abs()).sum((-1, -2))
  return (pair + (1 / 3) * (w.pow(2) * interval).sum(-1)).mean()


def _arg(args, k):
  return getattr(args, k, LOSS_DEFAULTS[k])


def objective(ret, ray_batch, args, epoch):
  """The loss of one training step, train.py:300-458 -> (loss, terms)."""
  ref, ref_dy = ret["outputs_coarse_ref"], ret["outputs_coarse_ref_dy"]
  anc, anc_dy = ret["outputs_coarse_anchor"], ret["outputs_coarse_anchor_dy"]
  dt = ref["rgb"].dtype
  decay_rate = _arg(args, "decay_rate")
  init_decay_epoch = _arg(args, "init_decay_epoch")
  divisor = epoch // init_decay_epoch                                                      # :302
  motion_mask = ray_batch["motion_mask"].to(dt)

  rgb_loss = criterion(ref, ray_batch)                                                    # :304
  rgb_loss = rgb_loss + compute_temporal_rgb_loss(anc, ray_batch)                          # :305-307
  if epoch < init_decay_epoch:                                                             # :309-316
    dynamic_mask = ref["mask"].to(dt) * motion_mask
    rgb_loss = rgb_loss + compute_rgb_loss(ref["rgb_dy"], ray_batch, dynamic_mask)
  dynamic_rgb_decay_rate = 10.0                                                            # :318-329
  rgb_loss = rgb_loss + criterion(ref_dy, ray_batch, motion_mask=motion_mask) / (dynamic_rgb_decay_rate ** divisor)
  rgb_loss = rgb_loss + compute_temporal_rgb_loss(anc_dy, ray_batch, motion_mask=motion_mask) / (
      dynamic_rgb_decay_rate ** divisor)

  w_disp = _arg(args, "w_disp") / (decay_rate ** divisor)                                  # :330-343
  pred_disp = 1.0 / torch.clamp(ref["depth"], min=1e-2)
  gt_disp = ray_batch["disp"]
  pred_mask = ref["mask"].to(dt)
  disp_loss = w_disp * torch.sum(torch.abs(pred_disp - gt_disp) * pred_mask) / (torch.sum(pred_mask) + 1e-8)

  w_flow = _arg(args, "w_flow") / (decay_rate ** divisor)                                  # :344-352
  flow_mask = pred_mask[None, :, None] * ray_batch["masks"].to(dt)
  flow_loss = w_flow * compute_flow_loss(ref["render_flows"], ray_batch["flows"], flow_mask)

  if _arg(args, "anneal_cycle"):                                                           # :353-371
    w_cycle = min(0.5, _arg(args, "w_cycle") + divisor * _arg(args, "cycle_factor"))
  else:
    w_cycle = _arg(args, "w_cycle")
  pts_traj_anchor, pts_traj_ref = anc["pts_traj_anchor"], anc["pts_traj_ref"]
  occ_weights = anc["occ_weights"][None, ..., None].repeat(pts_traj_anchor.shape[0], 1, 1, pts_traj_anchor.shape[-1])
  cycle_loss = w_cycle * torch.sum(torch.abs(pts_traj_ref - pts_traj_anchor) * occ_weights) / (
      torch.sum(occ_weights) + 1e-8)

  w_reg = _arg(args, "w_reg")                                                              # :373-397
  sf = anc["sf_seq"]
  reg_loss = w_reg * torch.mean(torch.abs(sf))
  reg_loss = reg_loss + w_reg * 0.5 * torch.mean(torch.pow(sf[:-1] - sf[1:], 2))
  reg_loss = reg_loss + w_reg * torch.mean(torch.abs(sf[:, :, 1:, :] - sf[:, :, :-1, :]))

  render_weights_dy = torch.sum(ref["weights_dy"], dim=-1)                                 # :399-413
  render_weights_st = torch.sum(ref["weights_st"], dim=-1)
  weights_ratio = render_weights_dy / torch.clamp(render_weights_dy + render_weights_st, min=1e-9)
  entropy_loss = -(weights_ratio * torch.log(weights_ratio + 1e-9)
                   + (1.0 - weights_ratio) * torch.log(1.0 - weights_ratio + 1e-9))
  entropy_loss = _arg(args, "w_skew_entropy") * torch.mean(entropy_loss)

  s_vals = ref["s_vals"]                                                                   # :415-423
  mid_dist = (s_vals[:, 1:] + s_vals[:, :-1]) * 0.5
  interval = s_vals[:, 1:] - s_vals[:, :-1]
  distortion_loss = _arg(args, "w_distortion") * eff_distloss_native(ref["weights"][:, :-1], mid_dist, interval)

  static_static_mask = 1.0 - ray_batch["static_mask"].to(dt)                               # :425-435
  static_static_mask = static_static_mask * ref["mask"].to(dt)
  static_static_mask = static_static_mask * (1.0 - weights_ratio).detach()
  static_loss = compute_rgb_loss(ref["rgb_static"], ray_batch, static_static_mask)
  if divisor > 4:                                                                          # :437-445
    static_sfm_mask_2 = static_static_mask * (weights_ratio < 0.1).to(dt)
    static_loss = static_loss + 0.1 * torch.sum(torch.abs(render_weights_dy * static_sfm_mask_2.detach())) / (
        torch.sum(static_sfm_mask_2 + 1e-8))

  loss = rgb_loss + cycle_loss + flow_loss + disp_loss + reg_loss + entropy_loss + distortion_loss + static_loss
  terms = dict(rgb_loss=rgb_loss, flow_loss=flow_loss, disp_loss=disp_loss, distortion_loss=distortion_loss,
               entropy_loss=entropy_loss, static_loss=static_loss, cycle_loss=cycle_loss, reg_loss=reg_loss)
  return loss, terms


def static_bootstrap_loss(ret, ray_batch):
  """train.py:187-196."""
  dt = ret["outputs_coarse_st"]["rgb"].dtype
  static_static_mask = 1.0 - ray_batch["static_mask"].to(dt)
  static_static_mask = static_static_mask * ret["outputs_coarse_ref"]["mask"].to(dt)
  return compute_rgb_loss(ret["outputs_coarse_st"]["rgb"], ray_batch, static_static_mask)
