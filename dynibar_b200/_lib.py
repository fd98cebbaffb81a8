"""ctypes binding of the C-ABI library (include/dynibar_b200.h).

The CUDA library is the product; there is NO fallback.  Importing this module
without a built `csrc/libdynibar_b200.so` raises ImportError telling the user
to run `python __graft_entry__.py` (which calls build()).
"""

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libdynibar_b200.so")

if not os.path.exists(LIB_PATH):
  raise ImportError(
      "dynibar_b200: %s is missing. Build it with `python __graft_entry__.py` "
      "(nvcc, sm_100a). There is no CPU/PyTorch fallback for the hot path." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

PREC_FP32, PREC_BF16 = 0, 1
NET_DYNAMIC, NET_STATIC, NET_MOTION = 0, 1, 2

_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t

# struct dyn_objective_in / dyn_objective_grad (pointer fields, in header order)
OBJ_IN_FIELDS = ("rgb", "rgb_dy", "rgb_static", "depth", "mask", "weights", "weights_dy", "weights_st", "s_vals",
                 "render_flows", "ref_dy_rgb", "ref_dy_mask", "a_rgb", "a_mask", "a_occ_map", "occ_weights",
                 "pts_traj_ref", "pts_traj_anchor", "sf_seq", "a_dy_rgb", "a_dy_mask", "a_dy_occ_map", "st_rgb",
                 "gt_rgb", "disp", "motion_mask", "static_mask", "flows", "flow_masks", "dist_mid", "dist_interval")
OBJ_GRAD_FIELDS = ("rgb", "rgb_dy", "rgb_static", "depth", "weights", "weights_dy", "weights_st", "render_flows",
                   "ref_dy_rgb", "a_rgb", "pts_traj_ref", "pts_traj_anchor", "sf_seq", "a_dy_rgb", "st_rgb")


class ObjectiveIn(C.Structure):
  _fields_ = [(n, _i) for n in ("R", "S", "K", "T", "F")] + [(n, _vp) for n in OBJ_IN_FIELDS]


class ObjectiveGrad(C.Structure):
  _fields_ = [(n, _vp) for n in OBJ_GRAD_FIELDS]


OBJ_NSUMS, OBJ_NTERMS, OBJ_NCOEF = 32, 8, 7
(OBJ_RGB, OBJ_TEMPORAL, OBJ_DYREGION, OBJ_DYNAMIC, OBJ_DISP, OBJ_FLOW, OBJ_CYCLE, OBJ_REG, OBJ_ENTROPY,
 OBJ_DISTORTION, OBJ_STATIC, OBJ_STATIC_EXTRA, OBJ_BOOTSTRAP) = (1 << i for i in range(13))

# name -> (restype, argtypes); mirrors include/dynibar_b200.h one to one
SIGNATURES = {
    "dyn_version": (_i, []),
    "dyn_last_error": (C.c_char_p, []),
    "dyn_device_sm_count": (_i, []),
    "dyn_launch_count": (C.c_ulonglong, [_i]),
    "dyn_profile_enable": (None, [_i]),
    "dyn_profile_read": (_i, [_i, C.POINTER(C.c_float), C.POINTER(_i)]),
    "dyn_net_param_count": (_sz, [_i]),
    "dyn_net_packed_bytes": (_sz, [_i]),
    "dyn_net_create": (_i, [_i, _vp, _sz, _vp, _i, _f, _i, _i, _vp, C.POINTER(_vp)]),
    "dyn_net_layer_images_bytes": (_sz, [_i]),
    "dyn_net_create_ex": (_i, [_i, _vp, _sz, _vp, _i, _i, _f, _i, _i, _vp, C.POINTER(_vp)]),
    "dyn_net_destroy": (None, [_vp]),
    "dyn_sample_rays": (_i, [_vp, _vp, _f, _f, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "dyn_points_from_depths": (_i, [_vp, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp]),
    "dyn_motion_workspace_bytes": (_sz, [_i, _i]),
    "dyn_motion_coeffs": (_i, [_vp, _vp, _f, _i, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_motion_mlp": (_i, [_vp, _vp, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_traj_displace": (_i, [_vp, _vp, _vp, _i, _i, _i, C.POINTER(_i), _i, _i, _i, _i, _vp, _vp]),
    "dyn_traj_delta": (_i, [_vp, _vp, _i, _i, C.POINTER(_i), C.POINTER(_i), _i, _i, _i, _vp, _vp]),
    "dyn_occlusion_weights": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "dyn_project_gather": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i,
                                _vp, _vp, _vp, _vp, _vp]),
    "dyn_compute_projections": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "dyn_compute_angle": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "dyn_plucker_ref": (_i, [_vp, _vp, _i, _vp, _vp]),
    "dyn_plucker_src": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "dyn_net_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "dyn_net_dynamic": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_net_static": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_net_fused_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "dyn_featmaps_channels_last": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "dyn_rgbs_rgba": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "dyn_net_static_fused": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i,
                                  _i, _vp, _vp, _vp, _sz, _vp]),
    "dyn_net_dynamic_fused": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _i, _i,
                                   _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "dyn_composite": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "dyn_composite_vanilla": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "dyn_resample": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "dyn_debug_set_view_timestamps": (None, [_vp]),
    "dyn_debug_set_view_kernel": (None, [_i]),
    "dyn_debug_point_chain": (_i, [_vp] * 5 + [_i, _i] + [_vp] * 9),
    "dyn_debug_pack_layer": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _f, _i, _vp, _sz, _vp, _vp]),
    "dyn_debug_tile_image_off": (_sz, [C.c_longlong, _i, _i]),
    "dyn_linear_tc_packed_bytes": (_sz, [_i, _i]),
    "dyn_linear_tc": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _sz, _vp]),
    "dyn_motion_train_workspace_bytes": (_sz, [_i]),
    "dyn_motion_mlp_train_forward": (_i, [_vp, _vp, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_motion_mlp_backward": (_i, [_vp, _vp, _vp, _i, _vp, _sz, _vp, _vp, _i, _vp]),
    "dyn_composite_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "dyn_project_gather_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "dyn_net_train_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "dyn_net_backward_scratch_bytes": (_sz, [_i, _i, _i, _i]),
    "dyn_net_dynamic_train_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_net_dynamic_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _i, _vp]),
    "dyn_net_static_train_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _i, _vp]),
    "dyn_net_static_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp, _sz, _vp, _vp, _i, _vp]),
    "dyn_composite_vanilla_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "dyn_traj_combine": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "dyn_traj_combine_backward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "dyn_flow_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "dyn_debug_tc_grad_w": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _vp, _i, _vp]),
    "dyn_debug_tc_grad_in": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _i, _vp, _sz, _vp]),
    "dyn_debug_tc_grad_in_scratch_bytes": (_sz, []),
    "dyn_encoder_param_count": (_sz, []),
    "dyn_encoder_workspace_bytes": (_sz, [_i, _i, _i]),
    "dyn_encoder_forward": (_i, [_vp, _sz, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "dyn_encoder_train_workspace_bytes": (_sz, [_i, _i, _i]),
    "dyn_encoder_backward_scratch_bytes": (_sz, [_i, _i, _i]),
    "dyn_encoder_train_forward": (_i, [_vp, _sz, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "dyn_encoder_backward": (_i, [_vp, _sz, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _i, _vp]),
    "dyn_flow_sceneflow": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i,
                                _vp, _vp, _vp]),
    "dyn_objective_workspace_bytes": (_sz, [_i]),
    "dyn_objective_sums": (_i, [C.POINTER(ObjectiveIn), _i, _vp, _vp, _sz, _vp]),
    "dyn_objective_finalize": (_i, [_vp, _i, C.POINTER(C.c_double), _vp, _vp, _vp, _vp]),
    "dyn_objective_backward": (_i, [C.POINTER(ObjectiveIn), _i, _vp, _vp, _vp, C.POINTER(ObjectiveGrad), _vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
  _fn = getattr(lib, _name)  # AttributeError here == header/library mismatch
  _fn.restype = _res
  _fn.argtypes = _args


def check(rc):
  if rc != 0:
    raise RuntimeError("dynibar_b200: %s (code %d)" % (lib.dyn_last_error().decode(), rc))


def ptr(t, dtype=torch.float32, allow_none=False):
  """Device pointer of a contiguous CUDA tensor (or None -> NULL)."""
  if t is None:
    if allow_none:
      return None
    raise ValueError("dynibar_b200: required tensor is None")
  if not t.is_cuda:
    raise RuntimeError("dynibar_b200 runs on CUDA tensors only (no CPU fallback); got a %s tensor"
                       % t.device)
  if t.dtype != dtype:
    raise TypeError("expected %s, got %s" % (dtype, t.dtype))
  if not t.is_contiguous():
    raise ValueError("tensor must be contiguous")
  return t.data_ptr()


def dev_of(t):
  """Device of a tensor that must live on a GPU (fail loudly otherwise)."""
  if not t.is_cuda:
    raise RuntimeError("dynibar_b200 runs on CUDA tensors only (no CPU fallback); got a %s tensor"
                       % t.device)
  return t.device


def f32c(t):
  """contiguous fp32 view/copy on the tensor's own device."""
  return t.detach().to(torch.float32).contiguous()


class Args(object):
  """Marshals tensors for ONE library call and keeps every temporary
  (contiguous / fp32 copies) alive until the caller drops this object, i.e.
  until after the kernels have been enqueued.  Without this a temporary's
  storage is returned to the caching allocator as soon as `ptr()` returns and
  the next temporary overwrites it before the kernel reads it."""

  def __init__(self):
    self.keep = []

  def host(self, t):
    """Small per-frame arrays (cameras, basis): a HOST fp32 pointer is accepted by
    the library and avoids a device read-back + stream sync inside the call."""
    if t is None:
      return None
    c = t.detach().to(torch.float32).contiguous()
    if c.is_cuda:
      c = c.cpu()
    self.keep.append(c)
    return c.data_ptr()

  def __call__(self, t, dtype=torch.float32):
    if t is None:
      return None
    c = t.detach()
    if dtype == torch.float32:
      c = c.to(torch.float32)
    c = c.contiguous()
    self.keep.append(c)
    return ptr(c, dtype)


def stream():
  return torch.cuda.current_stream().cuda_stream


class Workspace(object):
  """Grow-only per-device scratch buffer handed to the library."""

  def __init__(self):
    self._bufs = {}

  def get(self, nbytes, device, slot=0):
    key = (str(device), slot)
    buf = self._bufs.get(key)
    if buf is None or buf.numel() < nbytes:
      buf = None
      self._bufs[key] = None
      buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
      self._bufs[key] = buf
    return buf


workspace = Workspace()
