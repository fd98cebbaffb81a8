"""Training objective of DynIBaR on the GPU (csrc/objective.cu).

  * `dynibar_objective(ret, ray_batch, args, epoch)`  the loss of one training step, train.py:300-458, with the
                        criteria of ibrnet/criterion.py and utils.img2charbonier: rgb, temporal, dynamic-region and
                        dynamic-branch Charbonnier terms, disparity, flow, cycle, scene-flow regularisers, weight
                        entropy, distortion and the static terms.  Returns (loss, terms): 0-d device tensors, named
                        like the values train.py logs (train.py:458-465) plus `cycle_loss` and `reg_loss`.
  * `static_bootstrap_loss(ret, ray_batch)`  the loss of the static bootstrap epochs, train.py:187-196.
  * `eff_distloss_native(w, m, interval)`  drop-in for `torch_efficient_distloss.eff_distloss_native`.
  * `objective_sums(...)`  the fp64 sums the objective is made of (numerators, denominators, counts).

Each call is one `torch.autograd.Function` over three kernels: the sums (one warp per ray, fixed-order fp64
reductions: bit-identical between runs), the finalize step and the analytic backward.  Nothing synchronises with
the host.  Inputs are CUDA fp32 tensors; masks may also be bool.

Sharded training (rays split over ranks, `distributed.shard_ray_batch`): the mask-normalised terms need the sums
of the whole batch.  Pass `group=` to all-reduce the local sums vector before the finalize step, or `totals=` to
hand in a global sums vector computed elsewhere.  Every rank then reports the full-batch loss and its gradients
are its rays' share of the full-batch gradient, so `distributed.allreduce_gradients(params, average=False)` gives
the full-batch gradient.
"""

import ctypes as C

import torch

from dynibar_b200 import _lib
from dynibar_b200._lib import lib, check, stream

# config.py defaults of the fields the objective reads
LOSS_DEFAULTS = dict(w_disp=5e-2, w_flow=5e-3, w_cycle=0.1, cycle_factor=0.1, anneal_cycle=False, w_reg=0.05,
                     w_skew_entropy=1e-3, w_distortion=1e-3, decay_rate=10.0, init_decay_epoch=150)
TERM_NAMES = ("rgb_loss", "flow_loss", "disp_loss", "distortion_loss", "entropy_loss", "static_loss", "cycle_loss",
              "reg_loss")

_REF, _REF_DY, _ANC, _ANC_DY, _ST = ("outputs_coarse_ref", "outputs_coarse_ref_dy", "outputs_coarse_anchor",
                                     "outputs_coarse_anchor_dy", "outputs_coarse_st")
_BATCH = "ray_batch"
# struct field -> (where, key, shape); shape letters: R rays, S samples, K trajectory views, T sf_seq steps,
# F flow views, digits fixed; a trailing 1 may be left out.  Fields marked mask accept bool.
_SOURCES = {
    "rgb": (_REF, "rgb", "R3"), "rgb_dy": (_REF, "rgb_dy", "R3"), "rgb_static": (_REF, "rgb_static", "R3"),
    "depth": (_REF, "depth", "R"), "mask": (_REF, "mask", "R"), "weights": (_REF, "weights", "RS"),
    "weights_dy": (_REF, "weights_dy", "RS"), "weights_st": (_REF, "weights_st", "RS"),
    "s_vals": (_REF, "s_vals", "RS"), "render_flows": (_REF, "render_flows", "FR2"),
    "ref_dy_rgb": (_REF_DY, "rgb", "R3"), "ref_dy_mask": (_REF_DY, "mask", "R"),
    "a_rgb": (_ANC, "rgb", "R3"), "a_mask": (_ANC, "mask", "R"), "a_occ_map": (_ANC, "occ_weight_map", "R"),
    "occ_weights": (_ANC, "occ_weights", "RS"), "pts_traj_ref": (_ANC, "pts_traj_ref", "KRS3"),
    "pts_traj_anchor": (_ANC, "pts_traj_anchor", "KRS3"), "sf_seq": (_ANC, "sf_seq", "TRS3"),
    "a_dy_rgb": (_ANC_DY, "rgb", "R3"), "a_dy_mask": (_ANC_DY, "mask", "R"),
    "a_dy_occ_map": (_ANC_DY, "occ_weight_map", "R"),
    "st_rgb": (_ST, "rgb", "R3"),
    "gt_rgb": (_BATCH, "rgb", "R3"), "disp": (_BATCH, "disp", "R"), "motion_mask": (_BATCH, "motion_mask", "R"),
    "static_mask": (_BATCH, "static_mask", "R"), "flows": (_BATCH, "flows", "FR2"),
    "flow_masks": (_BATCH, "masks", "FR1"),
}
_MASKS = {"mask", "ref_dy_mask", "a_mask", "a_dy_mask", "motion_mask", "static_mask", "flow_masks"}
_OBJECTIVE_FIELDS = tuple(f for f in _SOURCES if f != "st_rgb")
_BOOTSTRAP_FIELDS = ("st_rgb", "mask", "gt_rgb", "static_mask")
_GRAD_FIELDS = set(_lib.OBJ_GRAD_FIELDS)


def schedule(args, epoch):
  """(term bits, coefficients) of train.py:302-445 at `epoch`; `args` fields missing -> config.py defaults."""
  a = lambda k: getattr(args, k, LOSS_DEFAULTS[k])
  init = int(a("init_decay_epoch"))
  divisor = int(epoch) // init
  terms = (_lib.OBJ_RGB | _lib.OBJ_TEMPORAL | _lib.OBJ_DYNAMIC | _lib.OBJ_DISP | _lib.OBJ_FLOW | _lib.OBJ_CYCLE |
           _lib.OBJ_REG | _lib.OBJ_ENTROPY | _lib.OBJ_DISTORTION | _lib.OBJ_STATIC)
  if epoch < init:
    terms |= _lib.OBJ_DYREGION
  if divisor > 4:
    terms |= _lib.OBJ_STATIC_EXTRA
  decay = float(a("decay_rate")) ** divisor
  if a("anneal_cycle"):
    w_cycle = min(0.5, a("w_cycle") + divisor * a("cycle_factor"))
  else:
    w_cycle = a("w_cycle")
  coef = (1.0 / 10.0 ** divisor, a("w_disp") / decay, a("w_flow") / decay, w_cycle, a("w_reg"),
          a("w_skew_entropy"), a("w_distortion"))
  return terms, tuple(float(c) for c in coef)


def _prepare(fn, named, dims):
  """named: field -> (label, tensor).  Checks device / dtype / shape (naming the argument) and returns the
  contiguous fp32 tensors and the dims {R, S, K, T, F}."""
  dev = None
  for f, (label, t, shape) in named.items():
    where = "%s: %s" % (fn, label)
    if not torch.is_tensor(t):
      raise RuntimeError("%s is missing (got %s)" % (where, type(t).__name__))
    if not t.is_cuda:
      raise RuntimeError("%s is a %s tensor: dynibar_b200 runs on CUDA tensors only (no CPU fallback)"
                         % (where, t.device))
    if t.dtype != torch.float32 and not (f in _MASKS and t.dtype == torch.bool):
      raise RuntimeError("%s has dtype %s, expected torch.float32%s" % (where, t.dtype,
                                                                       " or torch.bool" if f in _MASKS else ""))
    want = list(shape)
    got = list(t.shape)
    if len(got) == len(want) - 1 and want[-1] == "1":
      got.append(1)
    ok = len(got) == len(want)
    if ok:
      for sym, n in zip(want, got):
        if sym.isdigit():
          ok = ok and n == int(sym)
        elif sym in dims:
          ok = ok and n == dims[sym]
        else:
          dims[sym] = n
    if not ok:
      raise RuntimeError("%s has shape %s, expected [%s] with %s" % (
          where, tuple(t.shape), ", ".join(want), ", ".join("%s=%d" % kv for kv in sorted(dims.items()))))
    if dev is not None and t.device != dev:
      raise RuntimeError("%s is on %s, the inputs before it on %s" % (where, t.device, dev))
    dev = t.device
  # converted only once every argument has been checked: a rejected call launches nothing
  return {f: t.detach().float().contiguous() for f, (_, t, _) in named.items()}


def _struct(prep, dims):
  s = _lib.ObjectiveIn(R=dims.get("R", 0), S=dims.get("S", 0), K=dims.get("K", 0), T=dims.get("T", 0),
                       F=dims.get("F", 0))
  for f, t in prep.items():
    setattr(s, f, t.data_ptr())
  return s


def _sums(ins, terms, dev):
  nbytes = int(lib.dyn_objective_workspace_bytes(ins.R))
  ws = _lib.workspace.get(nbytes, dev, slot=4)
  sums = torch.empty(_lib.OBJ_NSUMS, dtype=torch.float64, device=dev)
  check(lib.dyn_objective_sums(C.byref(ins), terms, sums.data_ptr(), ws.data_ptr(), ws.numel(), stream()))
  return sums


class _Objective(torch.autograd.Function):
  """Inputs: (spec, *tensors) with spec = (fn, fields, labels, terms, coef, totals, group); tensors in the order
  of `fields`.  Outputs: loss (0-d) and the DYN_OBJ_NTERMS term values."""

  @staticmethod
  def forward(ctx, spec, *tensors):
    fn, fields, labels, terms, coef, totals, group = spec
    dims = {}
    prep = _prepare(fn, {f: (labels[i], t, _shape(f)) for i, (f, t) in enumerate(zip(fields, tensors))}, dims)
    dev = tensors[0].device
    ins = _struct(prep, dims)
    with torch.cuda.device(dev):
      if totals is None:
        sums = _sums(ins, terms, dev)
        if group is not None:
          import torch.distributed as dist
          dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
      else:
        sums = totals
      loss = torch.empty((), device=dev)
      vals = torch.empty(_lib.OBJ_NTERMS, device=dev)
      scales = torch.empty(_lib.OBJ_NSUMS, dtype=torch.float64, device=dev)
      check(lib.dyn_objective_finalize(sums.data_ptr(), terms, (C.c_double * _lib.OBJ_NCOEF)(*coef), loss.data_ptr(),
                                       vals.data_ptr(), scales.data_ptr(), stream()))
    ctx.set_materialize_grads(False)
    ctx.keep = (fields, terms, prep, dims, scales, [t.shape for t in tensors])
    return loss, vals

  @staticmethod
  def backward(ctx, g_loss, g_vals):
    fields, terms, prep, dims, scales, shapes = ctx.keep
    grads = [None] * len(fields)
    want = [i for i, f in enumerate(fields) if f in _GRAD_FIELDS and ctx.needs_input_grad[1 + i]]
    if not want or (g_loss is None and g_vals is None):
      return (None,) + tuple(grads)
    dev = scales.device
    gs = _lib.ObjectiveGrad()
    for i in want:
      grads[i] = torch.empty(shapes[i], device=dev)
      setattr(gs, fields[i], grads[i].data_ptr())
    gl = g_loss.detach().float().contiguous() if g_loss is not None else None
    gv = g_vals.detach().float().contiguous() if g_vals is not None else None
    ins = _struct(prep, dims)
    with torch.cuda.device(dev):
      check(lib.dyn_objective_backward(C.byref(ins), terms, scales.data_ptr(),
                                       gl.data_ptr() if gl is not None else None,
                                       gv.data_ptr() if gv is not None else None, C.byref(gs), stream()))
    return (None,) + tuple(grads)


def _shape(field):
  if field in _SOURCES:
    return _SOURCES[field][2]
  return {"dist_mid": "RS", "dist_interval": "RS"}[field]


def _lookup(fn, ret, ray_batch, fields):
  tensors, labels = [], []
  for f in fields:
    where, key, _ = _SOURCES[f]
    src = ray_batch if where == _BATCH else (ret.get(where) if isinstance(ret, dict) else None)
    if src is None:
      raise RuntimeError("%s: %s is missing (an output of render_rays_mono(is_train=True) expected)" % (fn, where))
    tensors.append(src.get(key))
    labels.append("%s['%s']" % (where, key))
  return tensors, labels


def _run(fn, ret, ray_batch, fields, terms, coef, totals=None, group=None):
  tensors, labels = _lookup(fn, ret, ray_batch, fields)
  if totals is not None:
    if not (torch.is_tensor(totals) and totals.is_cuda and totals.dtype == torch.float64
            and tuple(totals.shape) == (_lib.OBJ_NSUMS,)):
      raise RuntimeError("%s: totals must be a CUDA float64 tensor of shape [%d] (objective_sums)"
                         % (fn, _lib.OBJ_NSUMS))
    totals = totals.contiguous()
  return _Objective.apply((fn, tuple(fields), tuple(labels), terms, coef, totals, group), *tensors)


def dynibar_objective(ret, ray_batch, args, epoch, *, totals=None, group=None):
  """The loss of train.py:300-458 for `ret = render_rays_mono(..., is_train=True)` and the supervision keys of
  `ray_batch` (rgb, disp, motion_mask, static_mask, flows, masks).  Returns (loss, terms): 0-d device tensors;
  nothing is copied to the host.  `totals`: the global sums vector (sum of `objective_sums` over the shards) to
  normalise with instead of this batch's own; `group`: a process group whose ranks' sums are all-reduced first."""
  if totals is not None and group is not None:
    raise RuntimeError("dynibar_objective: pass totals or group, not both")
  terms, coef = schedule(args, epoch)
  loss, vals = _run("dynibar_objective", ret, ray_batch, _OBJECTIVE_FIELDS, terms, coef, totals, group)
  return loss, {n: vals[i] for i, n in enumerate(TERM_NAMES)}


def objective_sums(ret, ray_batch, args, epoch):
  """The DYN_OBJ_NSUMS fp64 sums of this batch (no gradient).  Sums of ray shards add up to the sums of the
  whole batch: pass their total as `dynibar_objective(..., totals=)`."""
  terms, _ = schedule(args, epoch)
  tensors, labels = _lookup("objective_sums", ret, ray_batch, _OBJECTIVE_FIELDS)
  dims = {}
  prep = _prepare("objective_sums", {f: (lb, t, _shape(f)) for f, lb, t in zip(_OBJECTIVE_FIELDS, labels, tensors)},
                  dims)
  dev = tensors[0].device
  with torch.cuda.device(dev):
    return _sums(_struct(prep, dims), terms, dev)


def static_bootstrap_loss(ret, ray_batch):
  """train.py:187-196: Charbonnier of outputs_coarse_st['rgb'] under (1 - static_mask) * outputs_coarse_ref['mask']."""
  loss, _ = _run("static_bootstrap_loss", ret, ray_batch, _BOOTSTRAP_FIELDS, _lib.OBJ_BOOTSTRAP,
                 (0.0,) * _lib.OBJ_NCOEF)
  return loss


def eff_distloss_native(w, m, interval):
  """Distortion loss of mip-NeRF 360 in the prefix-sum form of torch_efficient_distloss: w, m (ascending
  midpoints), interval [..., N]; mean over the leading elements.  Differentiable in w (m, interval carry no
  gradient, as train.py uses it)."""
  for name, t in (("w", w), ("m", m), ("interval", interval)):
    if not torch.is_tensor(t) or t.dim() < 1:
      raise RuntimeError("eff_distloss_native: %s must be a tensor with at least one dimension" % name)
  if m.shape != w.shape or interval.shape != w.shape:
    raise RuntimeError("eff_distloss_native: w %s, m %s and interval %s must have the same shape"
                       % (tuple(w.shape), tuple(m.shape), tuple(interval.shape)))
  n = w.shape[-1]
  fields = ("weights", "dist_mid", "dist_interval")
  loss, _ = _Objective.apply(("eff_distloss_native", fields, ("w", "m", "interval"), _lib.OBJ_DISTORTION,
                              (0.0,) * (_lib.OBJ_NCOEF - 1) + (1.0,), None, None),
                             w.reshape(-1, n), m.reshape(-1, n), interval.reshape(-1, n))
  return loss
