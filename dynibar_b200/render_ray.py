"""Per-ray renderer: drop-in for ibrnet/render_ray.py on the CUDA library.

Public surface (same names / signatures / returned dict keys as the
reference): `render_rays_mv` (render_ray.py:600), `render_rays_mono` (:870),
`sample_along_camera_ray` (:67), `raw2outputs` (:214), `raw2outputs_vanilla`
(:134), `compute_optical_flow` (:333), `compute_ref_plucker_coordinate` (:372),
`compute_src_plucker_coordinate` (:380), `z_to_s` (:399).

All math runs in `csrc/` kernels through the C ABI (include/dynibar_b200.h);
this file only allocates tensors and sequences calls.  `_render_pass` (one pass
at the reference time) and `_cross_time` (the anchor branch) state that sequence
once.  `render_rays_mono` is differentiable (training, SURVEY 8(f) f2): when
gradients are enabled and the model's parameters or the feature maps require
grad it runs the same sequence with `train=True`, and the stages whose kernels
differ use the autograd Functions of dynibar_b200/autograd.py over the backward
kernels.  `render_rays_mv` is the evaluation path (the reference calls it under
no_grad) and refuses inputs that require grad.
"""

from collections import OrderedDict
import contextlib
import ctypes as C
import os
import threading
import weakref

import torch

from dynibar_b200 import _lib
from dynibar_b200 import autograd as ag
from dynibar_b200 import weights as _weights
from dynibar_b200._lib import lib, ptr, f32c, check, stream, dev_of, Args
from dynibar_b200.projection import project_gather

# GEMM precision of the network kernels: "bf16" = tcgen05 (bf16 operands / fp32 accumulate and statistics; the
# production mode and the default), "fp32" = SIMT everywhere (parity mode).  Three ways to choose, innermost wins:
# the `precision=` argument of render_rays_mv / render_rays_mono (per call), `precision_scope(name)` (per
# thread, a context manager), `set_precision(name)` / the DYNIBAR_B200_PRECISION environment variable (process
# default).
_PREC = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16}
PRECISION = _PREC[os.environ.get("DYNIBAR_B200_PRECISION", "bf16")]
_tls = threading.local()


def set_precision(name):
  """Process-wide default ("fp32" | "bf16")."""
  global PRECISION
  PRECISION = _PREC[name]


@contextlib.contextmanager
def precision_scope(name):
  """Precision of every library call made by this thread inside the block (None = leave unchanged)."""
  if name is None:
    yield
    return
  prev = getattr(_tls, "override", None)
  _tls.override = _PREC[name]
  try:
    yield
  finally:
    _tls.override = prev


def _prec():
  o = getattr(_tls, "override", None)
  return PRECISION if o is None else o


def _no_grad_only(*tensors):
  if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
    raise NotImplementedError(
        "dynibar_b200 kernels are forward-only (training backward = SURVEY 8(f) f2); "
        "call under torch.no_grad() with detached inputs")


def _wants_grad(model, *featmaps):
  """True when gradients are enabled and a parameter of the model or a feature map requires grad."""
  if not torch.is_grad_enabled():
    return False
  mods = [m for m in vars(model).values() if isinstance(m, torch.nn.Module)]
  live = any(p.requires_grad for m in mods for p in m.parameters())
  return live or any(torch.is_tensor(f) and f.requires_grad for fm in featmaps if fm is not None
                     for f in fm if f is not None)


def _refuse_training(model, *featmaps):
  """render_rays_mv runs under no_grad (evaluation path; forward-only fused kernels): a training loop that
  called it would get detached outputs and fail late (or silently).  Fail loudly instead."""
  if _wants_grad(model, *featmaps):
    raise NotImplementedError(
        "dynibar_b200.render_rays_mv is the evaluation path (forward-only fused kernels): parameters or "
        "feature maps require grad; call under torch.no_grad() or freeze them (training = render_rays_mono)")


def _scalar(x):
  return float(x.reshape(-1)[0]) if torch.is_tensor(x) else float(x)


# ---------------------------------------------------------------------------
# a2
# ---------------------------------------------------------------------------
def sample_along_camera_ray(ray_o, ray_d, depth_range, N_samples, inv_uniform=False, det=False,
                            jitter=None):
  """render_ray.py:67-131.  `jitter` ([R,N_samples] U[0,1)) lets a caller
  supply the random draws; with det=False and jitter=None they are drawn with
  torch.rand like the reference (:119)."""
  R = ray_o.shape[0]
  dev = dev_of(ray_o)
  near, far = _scalar(depth_range[0, 0]), _scalar(depth_range[0, 1])
  assert near > 0 and far > 0 and far > near
  if not det and jitter is None:
    jitter = torch.rand(R, N_samples, device=dev)
  if det:
    jitter = None
  pts = torch.empty(R, N_samples, 3, device=dev)
  z = torch.empty(R, N_samples, device=dev)
  s = torch.empty(R, N_samples, device=dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_sample_rays(A(ray_o), A(ray_d), near, far, R, N_samples,
                              int(bool(inv_uniform)),
                              A(jitter),
                              ptr(pts), ptr(z), ptr(s), stream()))
  return pts, z, s


def z_to_s(z_vals, near_depth_value, far_depth_value):
  """render_ray.py:399-404 (elementwise; kept in torch, it is not on the hot
  path -- the kernels emit s_vals directly)."""
  return ((1.0 / z_vals) - (1.0 / near_depth_value)) / (1.0 / far_depth_value - 1.0 / near_depth_value)


def points_from_depths(ray_o, ray_d, z_vals, depth_range):
  R, S = z_vals.shape
  dev = dev_of(z_vals)
  near, far = _scalar(depth_range[0, 0]), _scalar(depth_range[0, 1])
  pts = torch.empty(R, S, 3, device=dev)
  s = torch.empty(R, S, device=dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_points_from_depths(A(ray_o), A(ray_d), A(z_vals), near,
                                     far, R, S, ptr(pts), ptr(s), stream()))
  return pts, s


# ---------------------------------------------------------------------------
# a3
# ---------------------------------------------------------------------------
def motion_mlp_forward(module, xyzt):
  """MotionMLP.forward on [...,4] rows (mlp_network.py:605-618)."""
  _no_grad_only(xyzt)
  dev = dev_of(xyzt)
  net = _weights.packed_of(module, dev)
  x = f32c(xyzt).reshape(-1, 4)
  N = x.shape[0]
  out = torch.empty(N, 3 * net.num_basis, device=dev)
  nbytes = lib.dyn_motion_workspace_bytes(N, 1)
  ws = _lib.workspace.get(nbytes, dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_motion_mlp(net.handle, ptr(x), N, ptr(out), ws.data_ptr(), nbytes, _prec(),
                             stream()))
  return _sf_mag_div(module, out).reshape(xyzt.shape[:-1] + (out.shape[-1],))


def motion_coefficients(module, pts, t):
  """coeffs [R,S,3*nb], last round(0.1*S) samples zeroed (render_ray.py:459-472)."""
  dev = dev_of(pts)
  net = _weights.packed_of(module, dev)
  R, S = pts.shape[:2]
  out = torch.empty(R, S, 3 * net.num_basis, device=dev)
  nbytes = lib.dyn_motion_workspace_bytes(R, S)
  ws = _lib.workspace.get(nbytes, dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_motion_coeffs(net.handle, A(pts), float(t), R, S, ptr(out),
                                ws.data_ptr(), nbytes, _prec(), stream()))
  return _sf_mag_div(module, out)


def _sf_mag_div(module, out):
  """MotionMLP.forward divides its output by the module's sf_mag_div (mlp_network.py:617)."""
  div = float(getattr(_weights.de_parallel(module), "sf_mag_div", 1.0))
  return out / div if div != 1.0 else out


def displaced_points(pts, coeff, basis, frame_idx, offsets, num_vv=0):
  """pts_3d_seq [len(offsets)+num_vv, R, S, 3] (render_ray.py:479-497, :988-991)."""
  dev = dev_of(pts)
  R, S = pts.shape[:2]
  n_off = len(offsets)
  T, nb = basis.shape
  seq = torch.empty(n_off + num_vv, R, S, 3, device=dev)
  offs = (C.c_int * max(n_off, 1))(*[int(o) for o in offsets])
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_traj_displace(A(pts), A(coeff), A.host(basis), T, nb,
                                int(frame_idx), offs, n_off, int(num_vv), R, S, ptr(seq), stream()))
  return seq


def traj_deltas(coeff, basis, frames_a, frames_b):
  """traj(frames_a[v]) - traj(frames_b[v]) -> [n,R,S,3] (scene-flow sequence,
  render_ray.py:1101-1105)."""
  dev = dev_of(coeff)
  R, S = coeff.shape[:2]
  n = len(frames_a)
  T, nb = basis.shape
  out = torch.empty(n, R, S, 3, device=dev)
  fa = (C.c_int * n)(*[int(f) for f in frames_a])
  fb = (C.c_int * n)(*[int(f) for f in frames_b])
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_traj_delta(A(coeff), A.host(basis), T, nb, fa, fb, n, R, S, ptr(out), stream()))
  return out


def occlusion_weights(w_ref, w_anchor):
  """occ_weights, occ_weight_map (render_ray.py:1224-1257)."""
  dev = dev_of(w_ref)
  R, S = w_ref.shape
  occ = torch.empty(R, S, device=dev)
  occ_map = torch.empty(R, device=dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_occlusion_weights(A(w_ref), A(w_anchor), R, S, ptr(occ), ptr(occ_map), stream()))
  return occ, occ_map


# ---------------------------------------------------------------------------
# a7
# ---------------------------------------------------------------------------
def compute_ref_plucker_coordinate(ray_o, ray_d):
  R = ray_o.shape[0]
  out = torch.empty(R, 6, device=dev_of(ray_o))
  A = Args()
  with torch.cuda.device(ray_o.device):
    check(lib.dyn_plucker_ref(A(ray_o), A(ray_d), R, ptr(out), stream()))
  return out


def compute_src_plucker_coordinate(pts, src_cameras):
  """pts [R,S,3], src_cameras [1,V,34] -> [R,S,V,6] (render_ray.py:380-396)."""
  R, S = pts.shape[:2]
  V = src_cameras.shape[1]
  out = torch.empty(R, S, V, 6, device=dev_of(pts))
  A = Args()
  with torch.cuda.device(pts.device):
    check(lib.dyn_plucker_src(A(pts), A.host(src_cameras), V, R, S, ptr(out), stream()))
  return out


# ---------------------------------------------------------------------------
# a8-a11
# ---------------------------------------------------------------------------
def net_dynamic_forward(module, pts, rgb_feat, ray_dir, mask, time):
  """DynibarDynamic.forward (mlp_network.py:236-316).  `time` is the
  reference's [R,S,1] tensor (constant) or a scalar."""
  _no_grad_only(pts, rgb_feat)
  dev = dev_of(pts)
  net = _weights.packed_of(module, dev)
  R, S, V = rgb_feat.shape[:3]
  raw = torch.empty(R, S, 4, device=dev)
  nbytes = lib.dyn_net_workspace_bytes(_lib.NET_DYNAMIC, R, S, V)
  ws = _lib.workspace.get(nbytes, dev)
  t = _scalar(time.float() if torch.is_tensor(time) else time)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_net_dynamic(net.handle, A(pts), A(rgb_feat), A(ray_dir),
                              A(mask), t, R, S, V, ptr(raw), ws.data_ptr(), nbytes,
                              _prec(), stream()))
  return raw


def net_static_forward(module, pts, ref_rays, src_rays, rgb_feat, ray_diff, mask):
  """DynibarStatic.forward (mlp_network.py:423-527)."""
  _no_grad_only(pts, rgb_feat)
  dev = dev_of(pts)
  net = _weights.packed_of(module, dev)
  R, S, V = rgb_feat.shape[:3]
  raw = torch.empty(R, S, 4, device=dev)
  nbytes = lib.dyn_net_workspace_bytes(_lib.NET_STATIC, R, S, V)
  ws = _lib.workspace.get(nbytes, dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_net_static(net.handle, A(pts), A(ref_rays), A(src_rays),
                             A(rgb_feat), A(ray_diff), A(mask), R, S, V,
                             ptr(raw), ws.data_ptr(), nbytes, _prec(), stream()))
  return raw


# ---------------------------------------------------------------------------
# fused a4-a11 (DYN_PREC_BF16): gather + per-view MLP chain in one tcgen05 kernel
# ---------------------------------------------------------------------------
class _FrameCache(object):
  """Packed per-frame copies of the source views, keyed by the IDENTITY of the source tensor (a weak
  reference plus its version counter), so the 18 chunks x 2 passes of one frame pack each map once
  while a new frame -- new tensor objects, or the same ones modified in place -- is packed again."""

  def __init__(self, capacity=16):
    self.entries = OrderedDict()
    self.capacity = capacity

  def get(self, tag, src, make):
    key = (tag, id(src))
    e = self.entries.get(key)
    if e is not None and e[0]() is src and e[1] == src._version:
      return e[2]
    packed = make(src)
    self.entries[key] = (weakref.ref(src), src._version, packed)
    self.entries.move_to_end(key)
    while len(self.entries) > self.capacity:
      self.entries.popitem(last=False)
    return packed


_frame_cache = _FrameCache()


def new_frame():
  """Drop the packed per-frame copies (a frame driver may call this when the source views change in place
  without their tensors' version counters noticing, e.g. after a collective wrote into them)."""
  _frame_cache.entries.clear()


def _pack_featmaps(featmaps):
  V, Cc, h, w = featmaps.shape
  dev = dev_of(featmaps)
  out = torch.empty(V, h, w, Cc, dtype=torch.bfloat16, device=dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_featmaps_channels_last(A(featmaps), ptr(out, torch.bfloat16), V, Cc, h, w, stream()))
  return out


def _pack_rgba(src_rgbs):
  _, V, H, W, _ = src_rgbs.shape
  dev = dev_of(src_rgbs)
  out = torch.empty(V, H, W, 4, device=dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_rgbs_rgba(A(src_rgbs), ptr(out), V, H, W, stream()))
  return out


def featmaps_channels_last(featmaps):
  """[V,C,h,w] fp32 -> channels-last bf16 [V,h,w,C] on the device (one bilinear tap of all 32 channels
  = 64 contiguous bytes); packed once per frame."""
  return _frame_cache.get("feat", featmaps, _pack_featmaps)


def source_rgba(src_rgbs):
  """[1,V,H,W,3] fp32 -> [V,H,W,4] fp32 (one tap = one aligned 16-byte load); packed once per frame."""
  return _frame_cache.get("rgba", src_rgbs, _pack_rgba)


def net_static_fused(module, pts, ray_o, ray_d, query_cam, src_rgbs, src_cams, feat_cl):
  """Projector.compute_with_motions + DynibarStatic.forward fused
  (projection.py:103-176 + mlp_network.py:423-527) -> raw [R,S,4], mask [R,S,V,1]."""
  dev = dev_of(pts)
  net = _weights.packed_of(module, dev)
  R, S = pts.shape[:2]
  V = src_cams.shape[1]
  _, _, H, W, _ = src_rgbs.shape
  _, h, w, Cc = feat_cl.shape
  raw = torch.empty(R, S, 4, device=dev)
  mask = torch.empty(R, S, V, 1, device=dev)
  nbytes = lib.dyn_net_fused_workspace_bytes(_lib.NET_STATIC, R, S, V)
  ws = _lib.workspace.get(nbytes, dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_net_static_fused(net.handle, A(pts), A(ray_o), A(ray_d), A.host(query_cam),
                                   ptr(source_rgba(src_rgbs)), A.host(src_cams),
                                   ptr(feat_cl, torch.bfloat16), R, S, V, H, W, Cc, h, w, ptr(raw),
                                   ptr(mask), ws.data_ptr(), nbytes, stream()))
  return raw, mask


def net_dynamic_fused(module, pts, pts_seq, ray_dir, query_cam, src_rgbs, src_cams, feat_cl, time):
  """Projector.compute_with_motions + DynibarDynamic.forward fused
  (projection.py:103-176 + mlp_network.py:236-316) -> raw [R,S,4], mask [R,S,V,1]."""
  dev = dev_of(pts)
  net = _weights.packed_of(module, dev)
  R, S = pts.shape[:2]
  V = src_cams.shape[1]
  _, _, H, W, _ = src_rgbs.shape
  _, h, w, Cc = feat_cl.shape
  raw = torch.empty(R, S, 4, device=dev)
  mask = torch.empty(R, S, V, 1, device=dev)
  nbytes = lib.dyn_net_fused_workspace_bytes(_lib.NET_DYNAMIC, R, S, V)
  ws = _lib.workspace.get(nbytes, dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_net_dynamic_fused(net.handle, A(pts), A(pts_seq), A(ray_dir), A.host(query_cam),
                                    ptr(source_rgba(src_rgbs)), A.host(src_cams),
                                    ptr(feat_cl, torch.bfloat16), float(time), R, S, V, H, W,
                                    Cc, h, w, ptr(raw), ptr(mask), ws.data_ptr(), nbytes, stream()))
  return raw, mask


# ---------------------------------------------------------------------------
# a12
# ---------------------------------------------------------------------------
def raw2outputs(raw_dy, raw_static, z_vals, mask_dy, mask_static, raw_noise_std=0.0):
  """render_ray.py:214-330; mask_* are the per-sample [R,S] validity masks."""
  return ag.composite(raw_dy, raw_static, z_vals, mask_dy.float()[..., None], mask_static.float()[..., None], 0, 0)


def raw2outputs_vanilla(raw, z_vals, mask):
  """render_ray.py:134-211."""
  return ag.composite_vanilla(raw, z_vals, mask.float()[..., None], 0)


# ---------------------------------------------------------------------------
# a13
# ---------------------------------------------------------------------------
def resample_depths(z_vals, weights, N_importance, inv_uniform, det=True, u=None):
  """sample_pdf on the interior weights + concat + sort
  (render_ray.py:790-819) -> [R, S+N_importance] ascending depths."""
  R, S = z_vals.shape
  dev = dev_of(z_vals)
  if not det and u is None:
    u = torch.rand(R, N_importance, device=dev)
  if det:
    u = None
  out = torch.empty(R, S + N_importance, device=dev)
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_resample(A(z_vals), A(weights),
                           A(u), R, S, N_importance,
                           int(bool(inv_uniform)), ptr(out), stream()))
  return out


# ---------------------------------------------------------------------------
# a14
# ---------------------------------------------------------------------------
def _flow_sceneflow(weights, pts_seq, src_cameras, uv, coeff, basis, frame_idx, sf_k, n_flow):
  R, S = weights.shape
  dev = dev_of(weights)
  flows = torch.empty(n_flow, R, 2, device=dev)
  exp_sf = torch.empty(R, 3, device=dev) if coeff is not None else None
  T, nb = (basis.shape if basis is not None else (0, 1))
  A = Args()
  with torch.cuda.device(dev):
    check(lib.dyn_flow_sceneflow(
        A(weights), A(pts_seq), A.host(src_cameras), A(uv),
        A(coeff),
        A.host(basis), T, nb, int(frame_idx), int(sf_k),
        int(n_flow), R, S, ptr(flows), ptr(exp_sf) if exp_sf is not None else None, stream()))
  return flows, exp_sf


def compute_optical_flow(outputs_coarse, raw_pts_3d_seq, src_cameras, uv_grid):
  """render_ray.py:333-358 -> [V,R,2]."""
  V = raw_pts_3d_seq.shape[0]
  flows, _ = _flow_sceneflow(outputs_coarse["weights"], raw_pts_3d_seq, src_cameras[:, :V],
                             uv_grid, None, None, 0, 0, V)
  return flows


# ---------------------------------------------------------------------------
# a15 orchestrators
# ---------------------------------------------------------------------------

_HOST_KEYS = ("camera", "src_cameras", "static_src_cameras", "anchor_src_cameras", "depth_range")


def _with_host_copies(ray_batch, model, basis_names):
  """One device->host read of the tiny per-frame arrays (cameras, depth range,
  trajectory basis) per render call instead of one per kernel launch."""
  rb = dict(ray_batch)
  for k in _HOST_KEYS:
    v = ray_batch.get(k)
    if torch.is_tensor(v) and v.is_cuda:
      rb[k] = v.detach().float().cpu()
  basis = {}
  for name in basis_names:
    b = getattr(model, name, None)
    basis[name] = b.detach().float().cpu() if torch.is_tensor(b) else b
  return rb, basis


# The stages of the sequence whose kernels differ between evaluation and training (`train`): the forward-only
# kernels, or the autograd Functions of dynibar_b200/autograd.py over the forward/backward kernels.
def _coefficients(train, motion, pts, t):
  """Motion coefficients [R,S,3*nb] at time t with the last round(0.1*S) samples zeroed (render_ray.py:957-958,
  :1126-1127)."""
  if not train:
    return motion_coefficients(motion, pts, t)
  R, S = pts.shape[:2]
  keep = torch.ones(1, S, 1, device=pts.device)
  keep[:, -int(round(S * 0.1)):] = 0.0  # the reference's x[:, -n:]: n == 0 (S <= 5) zeroes every sample
  xyzt = torch.cat([pts, torch.full((R, S, 1), t, device=pts.device)], dim=-1)
  return ag.motion_mlp(motion, xyzt) * keep


def _basis_rows(basis, pairs, dev):
  """D[i] = basis[a_i] - basis[b_i] ((None, None): a zero row) on the device; the host basis [T, nb] is indexed like
  the reference's (negative indices wrap)."""
  zero = torch.zeros_like(basis[0])
  return torch.stack([basis[a] - basis[b] if a is not None else zero for a, b in pairs]).to(dev)


def _displace(train, pts, coeff, basis, frame_idx, offsets, num_vv=0):
  """pts + traj(frame_idx + o) - traj(frame_idx) per offset, then num_vv copies of pts -> [n+num_vv,R,S,3]."""
  if not train:
    return displaced_points(pts, coeff, basis, frame_idx, offsets, num_vv)
  pairs = [(frame_idx + o, frame_idx) for o in offsets] + [(None, None)] * num_vv
  return ag.traj_combine(coeff, _basis_rows(basis, pairs, pts.device), pts)


def _deltas(train, coeff, basis, frames_a, frames_b):
  """traj(frames_a[i]) - traj(frames_b[i]) -> [n,R,S,3]."""
  if not train:
    return traj_deltas(coeff, basis, frames_a, frames_b)
  return ag.traj_combine(coeff, _basis_rows(basis, list(zip(frames_a, frames_b)), coeff.device))


def _fused(train, *cameras):
  """Evaluation in bf16 mode with at most 16 views per branch runs gather + per-view MLP chain + pooling as one
  tcgen05 kernel per branch: the [R,S,V,35] gather output and the per-view activations never reach HBM.  Otherwise
  the gather, then the networks' layers."""
  return not train and _prec() == _lib.PREC_BF16 and all(c.shape[1] <= 16 for c in cameras)


def _dynamic_branch(train, fused, net, pts, pts_net, seq, ray_dir, cam, rgbs, cams, feat, t):
  """DynibarDynamic on the views `cams` seen from the displaced points `seq` -> raw [R,S,4], mask [R,S,V,1].  As in
  the reference the gather takes the reference-time points `pts` and the network `pts_net` (:1178-1196)."""
  if fused:
    return net_dynamic_fused(net, pts_net, seq, ray_dir, cam, rgbs, cams, featmaps_channels_last(feat), t)
  gather, net_fn = (ag.project_gather, ag.net_dynamic) if train else (project_gather, net_dynamic_forward)
  f, _, m = gather(pts, seq, cam, rgbs, cams, feat)
  return net_fn(net, pts_net, f, ray_dir, m, t), m


def _render_pass(ray_batch, feat_dy, feat_st, pts, z, s, t, frame_idx, offsets, num_vv, net_dy, net_st, motion,
                 basis, flow_views, sf_k, train=False, want_extras=True, want_vanilla_st=False):
  """One coarse-or-fine evaluation at the reference time (render_ray.py:455-597 == :672-782 == :951-1096)
  -> the composited dicts (joint, dynamic, static or None) and what the cross-time branch reuses."""
  cam, ray_o, ray_d = ray_batch["camera"], ray_batch["ray_o"], ray_batch["ray_d"]
  cams_dy, cams_st = ray_batch["src_cameras"], ray_batch["static_src_cameras"]
  ref_plucker = compute_ref_plucker_coordinate(ray_o, ray_d)  # [d_hat, o x d_hat]
  ray_dir = ref_plucker[:, :3]  # == F.normalize(ray_d) (render_ray.py:455)
  coeff = _coefficients(train, motion, pts, t)
  seq = _displace(train, pts, coeff, basis, frame_idx, offsets, num_vv)
  fused = _fused(train, cams_dy, cams_st)
  raw_dy, m_dy = _dynamic_branch(train, fused, net_dy, pts, pts, seq, ray_dir, cam, ray_batch["src_rgbs"], cams_dy,
                                 feat_dy, t)
  if fused:
    raw_st, m_st = net_static_fused(net_st, pts, ray_o, ray_d, cam, ray_batch["static_src_rgbs"], cams_st,
                                    featmaps_channels_last(feat_st))
  else:
    gather, net_fn = (ag.project_gather, ag.net_static) if train else (project_gather, net_static_forward)
    f_st, rd_st, m_st = gather(pts, None, cam, ray_batch["static_src_rgbs"], cams_st, feat_st)
    raw_st = net_fn(net_st, pts, ref_plucker, compute_src_plucker_coordinate(pts, cams_st), f_st, rd_st, m_st)
  # a sample counts when MORE THAN ONE view sees it (render_ray.py:524-529)
  out = ag.composite(raw_dy, raw_st, z, m_dy, m_st, 1, 1)
  out_dy = ag.composite_vanilla(raw_dy, z, m_dy, 1)
  out_st = ag.composite_vanilla(raw_st, z, m_st, 1) if want_vanilla_st else None
  if want_extras:
    nflow = seq.shape[0] if flow_views is None else flow_views
    uv = ray_batch["uv_grid"]
    if train:  # exp_sf is detached in the reference (:1086-1096)
      flows = ag.optical_flow(out["weights"], seq[:nflow], cams_dy[:, :nflow], uv)
      _, exp_sf = _flow_sceneflow(out["weights"], seq, cams_dy, uv, coeff, basis, frame_idx, sf_k, 1)
    else:
      flows, exp_sf = _flow_sceneflow(out["weights"], seq, cams_dy, uv, coeff, basis, frame_idx, sf_k, nflow)
    out["render_flows"] = flows
    out["s_vals"] = s
    out["exp_sf"] = exp_sf
  return out, out_dy, out_st, dict(coeff=coeff, raw_st=raw_st, m_st=m_st, ray_dir=ray_dir)


def render_rays_mv(frame_idx, time_embedding, time_offset, ray_batch, model, projector,
                   coarse_featmaps, fine_featmaps, N_samples, args, inv_uniform=False,
                   N_importance=0, raw_noise_std=0.0, det=False, white_bkgd=False, is_train=True,
                   jitter=None, u=None, precision=None):
  """Coarse + fine rendering for the Nvidia multi-view benchmark
  (render_ray.py:600-867).  Extra keyword-only inputs `jitter` / `u` carry the
  random draws of :119 / :34 when det=False (drawn with torch.rand if None).
  Returns the reference's dict: outputs_coarse_ref, outputs_fine_ref,
  outputs_fine_ref_dy, outputs_fine_anchor(None), outputs_fine_anchor_dy(None)."""
  assert N_importance > 0  # render_ray.py:787
  _refuse_training(model, coarse_featmaps, fine_featmaps)
  with torch.no_grad(), precision_scope(precision):
    t = _scalar(time_embedding[0].float())
    offs = [int(o) for o in time_offset[0]]
    fidx = int(frame_idx[0])
    ret = {"outputs_coarse": None, "outputs_fine": None}
    ray_batch, hb = _with_host_copies(ray_batch, model, ("trajectory_basis", "trajectory_basis_fine"))
    pts, z, _ = sample_along_camera_ray(ray_batch["ray_o"], ray_batch["ray_d"],
                                        ray_batch["depth_range"], N_samples, inv_uniform, det, jitter)
    out_c = _render_pass(ray_batch, coarse_featmaps[0], coarse_featmaps[2], pts, z, None, t, fidx, offs, 0,
                         model.net_coarse_dy, model.net_coarse_st, model.motion_mlp, hb["trajectory_basis"], None,
                         2, want_extras=False)[0]
    ret["outputs_coarse_ref"] = out_c
    zf = resample_depths(z, out_c["weights"], N_importance, inv_uniform, det, u)
    pts_f, s = points_from_depths(ray_batch["ray_o"], ray_batch["ray_d"], zf,
                                  ray_batch["depth_range"])
    out_f, out_f_dy = _render_pass(ray_batch, fine_featmaps[0], fine_featmaps[2], pts_f, zf, s, t, fidx, offs, 0,
                                   model.net_fine_dy, model.net_fine_st, model.motion_mlp_fine,
                                   hb["trajectory_basis_fine"], None, 2)[:2]
    ret["outputs_fine_ref"] = out_f
    ret["outputs_fine_ref_dy"] = out_f_dy
    ret["outputs_fine_anchor"] = None
    ret["outputs_fine_anchor_dy"] = None
  return ret


def render_rays_mono(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps, projector,
                     N_samples, args, inv_uniform=False, N_importance=0, raw_noise_std=0.0,
                     det=False, white_bkgd=False, is_train=True, num_vv=2, jitter=None, precision=None):
  """Coarse-only rendering for monocular video (render_ray.py:870-1277), including the
  cross-time branch (:1099-1270) when is_train=True.  With gradients enabled and parameters / feature
  maps that require grad it is differentiable (training, see _render_mono); otherwise the forward-only kernels
  (fused tcgen05 path in bf16 mode) run under no_grad."""
  with precision_scope(precision):
    if _wants_grad(model, featmaps):
      return _render_mono_train_chunked(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps,
                                        N_samples, args, inv_uniform, det, is_train, num_vv, jitter)
    with torch.no_grad():
      return _render_mono(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps, N_samples, args,
                          inv_uniform, det, is_train, num_vv, jitter, False)


def _render_mono(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps, N_samples, args, inv_uniform,
                 det, is_train, num_vv, jitter, train):
  """render_rays_mono on one batch of rays.  `train`: the stages that gradients pass through are
  `torch.autograd.Function`s over the forward/backward kernels (dynibar_b200/autograd.py), so gradients reach the
  parameters of motion_mlp / net_coarse_dy / net_coarse_st and the feature maps.  Training precision (the
  library-wide setting / `precision=`): "bf16" runs the products of the three networks, forward and backward, on
  tcgen05 (bf16 operands, fp32 accumulation, fp32 master weights and gradients); "fp32" = SIMT products."""
  t = _scalar(time_embedding[0].float())
  ray_batch, hb = _with_host_copies(ray_batch, model, ("trajectory_basis",))
  basis = hb["trajectory_basis"]
  fidx = int(frame_idx[0])
  pts, z, s = sample_along_camera_ray(ray_batch["ray_o"], ray_batch["ray_d"], ray_batch["depth_range"], N_samples,
                                      inv_uniform, det, jitter)
  out, out_dy, out_st, aux = _render_pass(ray_batch, featmaps[0], featmaps[2], pts, z, s, t, fidx,
                                          [int(o) for o in time_offset[0]], num_vv, model.net_coarse_dy,
                                          model.net_coarse_st, model.motion_mlp, basis, 6, 1, train=train,
                                          want_vanilla_st=True)
  ret = {"outputs_coarse": None, "outputs_fine": None, "outputs_coarse_ref": out,
         "outputs_coarse_ref_dy": out_dy, "outputs_coarse_st": out_st}
  if is_train:
    ret.update(_cross_time(ray_batch, featmaps[1], pts, z, aux, fidx, int(frame_idx[1]),
                           _scalar(time_embedding[1].float()), [int(o) for o in time_offset[1]], num_vv, model,
                           basis, args.occ_weights_mode, out, out_dy, train))
  return ret


def _cross_time(ray_batch, feat_anchor, pts, z, aux, ref_idx, anc_idx, t_anc, anchor_offsets, num_vv,
                model, basis, occ_mode, out_ref, out_ref_dy, train):
  """Cross-time rendering for temporal consistency (render_ray.py:1099-1270)."""
  coeff = aux["coeff"]
  sf_seq = _deltas(train, coeff, basis, [ref_idx + o for o in (-2, -1, 0, 1, 2, 3)],
                   [ref_idx + o - 1 for o in (-2, -1, 0, 1, 2, 3)])
  pts_anchor = _displace(train, pts, coeff, basis, ref_idx, [anc_idx - ref_idx])[0]  # :1109-1112
  coeff_a = _coefficients(train, model.motion_mlp, pts_anchor, t_anc)                 # :1126-1127
  seq_a = _displace(train, pts_anchor, coeff_a, basis, anc_idx, anchor_offsets, num_vv)  # :1149-1176
  kept = [(i, anc_idx + o - ref_idx) for i, o in enumerate(anchor_offsets)
          if -3 <= anc_idx + o - ref_idx <= 3]
  pts_traj_anchor = seq_a[[i for i, _ in kept]]
  pts_traj_ref = _displace(train, pts, coeff, basis, ref_idx, [ro for _, ro in kept])
  cams_a = ray_batch["anchor_src_cameras"]
  raw_a, m_a = _dynamic_branch(train, _fused(train, cams_a), model.net_coarse_dy, pts, pts_anchor, seq_a,
                               aux["ray_dir"], ray_batch["camera"], ray_batch["anchor_src_rgbs"], cams_a,
                               feat_anchor, t_anc)
  # anchor samples count when ANY view sees them (render_ray.py:1198-1200)
  out_a = ag.composite(raw_a, aux["raw_st"], z, m_a, aux["m_st"], 0, 1)
  out_a_dy = ag.composite_vanilla(raw_a, z, m_a, 0)
  if occ_mode == 0:
    key = "weights_dy" if abs(ref_idx - anc_idx) > 1 else "weights"
  elif occ_mode == 1:
    key = "weights_dy"
  elif occ_mode == 2:
    key = "weights"
  else:
    raise NotImplementedError
  # detached in the reference (:1222, :1254)
  out_a["occ_weights"], out_a["occ_weight_map"] = occlusion_weights(out_ref[key], out_a[key])
  out_a["pts_traj_ref"] = pts_traj_ref
  out_a["pts_traj_anchor"] = pts_traj_anchor
  out_a["sf_seq"] = sf_seq
  out_a_dy["occ_weights"], out_a_dy["occ_weight_map"] = occlusion_weights(out_ref_dy["weights"],
                                                                         out_a_dy["weights"])
  return {"outputs_coarse_anchor": out_a, "outputs_coarse_anchor_dy": out_a_dy}


# (point, view) rows one training call of a network may hold (csrc/nets_f32.cu: net_rows_per_chunk; the training
# forward keeps every activation of ONE internal chunk); larger ray batches are rendered in slices
TRAIN_ROWS_LIMIT = 4194304
_RAY_AXIS1 = ("render_flows", "pts_traj_ref", "pts_traj_anchor", "sf_seq")  # [n, R, ...]; every other key is [R, ...]


def _render_mono_train_chunked(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps, N_samples, args,
                               inv_uniform, det, is_train, num_vv, jitter):
  """Slices the rays so that no network call exceeds TRAIN_ROWS_LIMIT rows, renders each slice with
  `_render_mono(..., train=True)` and concatenates the per-slice output dicts along their ray axis (autograd sees
  one graph; gradients accumulate over the slices)."""
  R = ray_batch["ray_o"].shape[0]
  vmax = max(ray_batch[k].shape[1] for k in ("src_cameras", "static_src_cameras", "anchor_src_cameras")
             if k in ray_batch and (is_train or k != "anchor_src_cameras"))
  per = max(1, TRAIN_ROWS_LIMIT // (N_samples * vmax))
  if R <= per:
    return _render_mono(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps, N_samples, args,
                        inv_uniform, det, is_train, num_vv, jitter, True)
  parts = []
  for lo in range(0, R, per):
    hi = min(R, lo + per)
    rb = dict(ray_batch)
    for k in ("ray_o", "ray_d", "uv_grid"):
      rb[k] = ray_batch[k][lo:hi]
    parts.append(_render_mono(frame_idx, time_embedding, time_offset, rb, model, featmaps, N_samples, args,
                              inv_uniform, det, is_train, num_vv, None if jitter is None else jitter[lo:hi], True))
  ret = {}
  for name, first in parts[0].items():
    if first is None:
      ret[name] = None
      continue
    ret[name] = OrderedDict((k, torch.cat([p[name][k] for p in parts], 1 if k in _RAY_AXIS1 else 0))
                            for k in first)
  return ret
