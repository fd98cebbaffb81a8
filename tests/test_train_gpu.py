"""Training backward (row f2) against torch autograd through the oracle's restatement of the same reference
functions: DynibarDynamic.forward / DynibarStatic.forward (mlp_network.py:236-316, :423-527), the small
differentiable pieces (raw2outputs_vanilla, compute_traj_pts, compute_optical_flow) and the whole
`render_rays_mono(is_train=True)` training forward + backward (render_ray.py:870-1277).

Bar, precision "fp32": forward values rtol 2e-4; gradients 1e-3 relative in the L2 norm per tensor (fp32 kernels
with a different summation order than ATen; ELU is C1, so there are no kink flips except the MotionMLP's ReLUs, see
test_backward_gpu.py).  Precision "bf16" (products on tcgen05 with bf16 operands, everything else fp32): forward
2e-2, gradients 5e-2 (matrices) / 1e-1 (vectors) against the same fp32 oracle."""

import pytest
import torch
import torch.nn.functional as F

import scenes
from dynibar_b200 import synthetic
from oracle import dynibar_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


class _W(dict):
  """state_dict of leaf tensors for the oracle (which reads `shift` off the module it is handed)."""
  shift = 0.0


def _leaves(module, shift=0.0):
  w = _W({k: v.detach().clone().requires_grad_(True) for k, v in module.state_dict().items()})
  w.shift = shift
  return w


def _close(name, got, ref, tol=1e-3, floor=1e-6):
  """`floor`: gradients that are zero in exact arithmetic (the bias of the blending logit: a softmax is invariant
  to a common shift) come out as rounding noise of either sign on both sides."""
  d = got.detach().cpu().double() - ref.detach().double()
  rn = ref.detach().double().norm().item()
  assert d.norm().item() <= tol * rn + floor, (name, d.norm().item(), rn)
  assert d.abs().max().item() <= 10 * tol * ref.detach().abs().max().item() + floor, (name, d.abs().max().item())


def _net_inputs(R, S, V, seed):
  g = torch.Generator().manual_seed(seed)
  pts = torch.randn(R, S, 3, generator=g) * 2
  feat = torch.randn(R, S, V, 35, generator=g)
  feat[..., :3] = torch.rand(R, S, V, 3, generator=g)
  mask = (torch.rand(R, S, V, 1, generator=g) > 0.3).float()
  mask[0, 0] = 0.0          # a point no view sees
  mask[0, 1] = 0.0
  mask[0, 1, 0] = 1.0       # a point with exactly one valid view (masked query row of the ray transformer)
  ray_dir = F.normalize(torch.randn(R, 3, generator=g), dim=-1)
  return g, pts, feat, mask, ray_dir


def _tol(prec, dim):
  if prec == "fp32":
    return 1e-3
  return 5e-2 if dim > 1 else 1e-1


@pytest.mark.parametrize("R,S,V,prec", [(6, 16, 5, "fp32"), (3, 40, 8, "fp32"), (40, 16, 8, "bf16")])
def test_net_dynamic_backward_matches_oracle_autograd(R, S, V, prec):
  from dynibar_b200 import autograd as ag, mlp_network as nets
  torch.manual_seed(R * S + V)
  args = synthetic.make_args(1, 0)
  mod = nets.DynibarDynamic(args, 32, S, shift=5.0)
  with torch.no_grad():
    mod.out_geometry_fc[2].bias.fill_(1.0)
  g, pts, feat, mask, ray_dir = _net_inputs(R, S, V, 7 + V)
  t = torch.tensor([0.4])
  gen = torch.randn(R, S, 4, generator=g)
  # ---- oracle + torch autograd (CPU, fp32)
  w = _leaves(mod, 5.0)
  po, fo = pts.clone().requires_grad_(True), feat.clone().requires_grad_(True)
  want = orc.net_dynamic(w, po, fo, ray_dir, mask, t, 5.0)
  live = (mask.sum(2) >= 1).float()  # sigma is -1e9 where no view sees the point
  (want * gen * torch.cat([live.expand(-1, -1, 3), live], -1)).sum().backward()
  # ---- library
  mod = mod.to(DEV).requires_grad_(True)
  pd, fd = pts.to(DEV).requires_grad_(True), feat.to(DEV).requires_grad_(True)
  got = ag.net_dynamic(mod, pd, fd, ray_dir.to(DEV), mask.to(DEV), t, precision=prec)
  ft = dict(rtol=2e-4, atol=2e-5) if prec == "fp32" else dict(rtol=2e-2, atol=5e-3)
  torch.testing.assert_close(got.detach().cpu(), want.detach(), **ft)
  (got * (gen * torch.cat([live.expand(-1, -1, 3), live], -1)).to(DEV)).sum().backward()
  for k, p in mod.named_parameters():
    _close(k, p.grad, w[k].grad, _tol(prec, p.dim()))
  _close("rgb_feat", fd.grad, fo.grad, _tol(prec, 2))
  _close("pts", pd.grad, po.grad, _tol(prec, 2))


@pytest.mark.parametrize("R,S,V,aa,mrgb,prec", [(6, 16, 5, 1, 0, "fp32"), (3, 24, 8, 0, 1, "fp32"),
                                                   (4, 16, 11, 1, 1, "fp32"), (40, 16, 8, 1, 0, "bf16")])
def test_net_static_backward_matches_oracle_autograd(R, S, V, aa, mrgb, prec):
  from dynibar_b200 import autograd as ag, mlp_network as nets
  torch.manual_seed(R * S + V)
  args = synthetic.make_args(aa, mrgb)
  mod = nets.DynibarStatic(args, 32, S)
  with torch.no_grad():
    mod.out_geometry_fc[2].bias.fill_(0.5)
  g, pts, feat, mask, ray_dir = _net_inputs(R, S, V, 11 + V)
  if mrgb:
    feat[1, 2, 1, :3] = 0.0  # a dark source colour: masked out by mask_rgb
  ref_rays = torch.randn(R, 6, generator=g)
  src_rays = torch.randn(R, S, V, 6, generator=g)
  ray_diff = torch.cat([F.normalize(torch.randn(R, S, V, 3, generator=g), dim=-1),
                        torch.rand(R, S, V, 1, generator=g) * 0.3 + 0.7], -1)
  gen = torch.randn(R, S, 4, generator=g)
  w = _leaves(mod)
  fo = feat.clone().requires_grad_(True)
  want = orc.net_static(w, pts, ref_rays, src_rays, fo, ray_diff, mask, anti_alias_pooling=bool(aa),
                        mask_rgb=bool(mrgb))
  meff = mask * (feat[..., :3].sum(-1, keepdim=True) > 1e-3).float() if mrgb else mask
  live = (meff.sum(2) >= 1).float()
  scale = torch.cat([torch.ones(R, S, 3), live], -1)
  (want * gen * scale).sum().backward()
  mod = mod.to(DEV).requires_grad_(True)
  fd = feat.to(DEV).requires_grad_(True)
  d = lambda x: x.to(DEV)
  got = ag.net_static(mod, d(pts), d(ref_rays), d(src_rays), fd, d(ray_diff), d(mask), precision=prec)
  ft = dict(rtol=2e-4, atol=2e-5) if prec == "fp32" else dict(rtol=2e-2, atol=5e-3)
  torch.testing.assert_close(got.detach().cpu(), want.detach(), **ft)
  (got * d(gen * scale)).sum().backward()
  for k, p in mod.named_parameters():
    # `s` (anti-alias pooling): a small sum of large cancelling terms, (e - min e) / (sum + 1e-8): 1e-2 in fp32; with
    # bf16 products the 0.5 % noise of d(pooling weights) is amplified by 1 / (sum + 1e-8) past the signal
    # (profiles/r02_train.md), so only finiteness is checked there
    if k == "s":
      if prec == "fp32":
        _close(k, p.grad, w[k].grad, 1e-2)
      else:
        assert torch.isfinite(p.grad).all()
      continue
    _close(k, p.grad, w[k].grad, _tol(prec, p.dim()))
  _close("rgb_feat", fd.grad, fo.grad, _tol(prec, 2))


def test_small_pieces_match_oracle_autograd():
  """raw2outputs_vanilla, compute_traj_pts combinations, compute_optical_flow."""
  from dynibar_b200 import autograd as ag
  g = torch.Generator().manual_seed(5)
  R, S, V, nb = 9, 40, 7, 6
  # ---- vanilla compositing
  raw = torch.randn(R, S, 4, generator=g)
  raw[..., :3].sigmoid_()
  raw[..., 3] -= 2.0
  z = torch.sort(torch.rand(R, S, generator=g) * 20 + 1, dim=1).values
  m = (torch.rand(R, S, V, 1, generator=g) > 0.2).float()
  keys = ("rgb", "depth", "weights", "alpha")
  a = raw.clone().requires_grad_(True)
  want = orc.composite_vanilla(a, z, m.sum(2)[..., 0] > 1)
  gens = {k: torch.randn(want[k].shape, generator=g) for k in keys}
  sum((want[k] * gens[k]).sum() for k in keys).backward()
  ad = raw.to(DEV).requires_grad_(True)
  got = ag.composite_vanilla(ad, z.to(DEV), m.to(DEV), 1)
  for k in keys:
    torch.testing.assert_close(got[k].detach().cpu(), want[k].detach(), rtol=1e-4, atol=1e-5)
  assert torch.equal(got["mask"].cpu(), want["mask"])
  sum((got[k] * gens[k].to(DEV)).sum() for k in keys).backward()
  torch.testing.assert_close(ad.grad.cpu(), a.grad, rtol=2e-4, atol=2e-5)
  # ---- trajectory combination
  coeff = torch.randn(R, S, 3 * nb, generator=g)
  base = torch.randn(R, S, 3, generator=g)
  basis = synthetic.init_dct_basis(nb, 24)
  D = torch.stack([basis[12] - basis[10], basis[7] - basis[10], torch.zeros(nb)])
  co, bo = coeff.clone().requires_grad_(True), base.clone().requires_grad_(True)
  want_t = torch.stack([bo + orc.traj_offset(co, basis[12]) - orc.traj_offset(co, basis[10]),
                        bo + orc.traj_offset(co, basis[7]) - orc.traj_offset(co, basis[10]), bo])
  gt = torch.randn(want_t.shape, generator=g)
  (want_t * gt).sum().backward()
  cd, bd = coeff.to(DEV).requires_grad_(True), base.to(DEV).requires_grad_(True)
  got_t = ag.traj_combine(cd, D.to(DEV), bd)
  torch.testing.assert_close(got_t.detach().cpu(), want_t.detach(), rtol=1e-5, atol=1e-5)
  (got_t * gt.to(DEV)).sum().backward()
  torch.testing.assert_close(cd.grad.cpu(), co.grad, rtol=1e-4, atol=1e-5)
  torch.testing.assert_close(bd.grad.cpu(), bo.grad, rtol=1e-4, atol=1e-5)
  # ---- optical flow
  cfg = scenes.GOLDEN_CONFIGS["mono_train"]
  batch = scenes.build(cfg)[0]
  Rr = batch["ray_o"].shape[0]
  wts = torch.softmax(torch.randn(Rr, S, generator=g), 1) * 0.9
  seq = torch.randn(6, Rr, S, 3, generator=g) * 0.3 + torch.tensor([0.0, 0.0, 6.0])
  wo, so = wts.clone().requires_grad_(True), seq.clone().requires_grad_(True)
  want_f = orc.optical_flow(wo, so, batch["src_cameras"][:, :6], batch["uv_grid"])
  gf = torch.randn(want_f.shape, generator=g)
  (want_f * gf).sum().backward()
  wd, sd = wts.to(DEV).requires_grad_(True), seq.to(DEV).requires_grad_(True)
  got_f = ag.optical_flow(wd, sd, batch["src_cameras"][:, :6], batch["uv_grid"].to(DEV))
  torch.testing.assert_close(got_f.detach().cpu(), want_f.detach(), rtol=1e-4, atol=1e-3)
  (got_f * gf.to(DEV)).sum().backward()
  _close("flow d weights", wd.grad, wo.grad, 2e-4)
  _close("flow d pts", sd.grad, so.grad, 2e-4)


_TRAIN_KEYS = {
    "outputs_coarse_ref": ("rgb", "rgb_static", "rgb_dy", "depth", "weights", "weights_dy", "weights_st", "alpha",
                           "alpha_dy", "render_flows"),
    "outputs_coarse_ref_dy": ("rgb", "depth", "weights"),
    "outputs_coarse_st": ("rgb", "depth", "weights"),
    "outputs_coarse_anchor": ("rgb", "rgb_static", "rgb_dy", "depth", "weights", "weights_dy", "pts_traj_ref",
                              "pts_traj_anchor", "sf_seq"),
    "outputs_coarse_anchor_dy": ("rgb", "depth", "weights"),
}


# S4: with 4 samples per ray round(0.1 * 4) = 0, and the reference's x[:, -0:] zeroes the motion coefficients of every
# sample.  Without anti-alias pooling: with it, torch's own fp32 autograd of this 4-sample rig is 0.7 % away from its
# fp64 autograd for the static net's attention weights, above the bar below; without it, under 0.1 % for every tensor.
@pytest.mark.parametrize("name,prec,over", [("mono_train", "fp32", {}), ("mono_train_near", "fp32", {}),
                                            ("mono_train", "bf16", {}),
                                            ("mono_train", "fp32", dict(N_samples=4, anti_alias_pooling=0))],
                         ids=["mono_train-fp32", "mono_train_near-fp32", "mono_train-bf16", "mono_train-fp32-S4"])
def test_render_rays_mono_training_step_matches_oracle_autograd(name, prec, over):
  """The whole differentiable path: loss = sum of randomly weighted differentiable outputs of
  render_rays_mono(is_train=True); d loss / d (every parameter of motion_mlp, net_coarse_dy, net_coarse_st and the
  three feature maps) against torch autograd through the oracle."""
  from dynibar_b200 import render_ray as rr
  from dynibar_b200.projection import Projector
  cfg = dict(scenes.GOLDEN_CONFIGS[name], **over)
  motion_off = int(round(0.1 * cfg["N_samples"])) == 0  # every sample's motion coefficients are zeroed
  if prec == "bf16":
    cfg["rays"] = 96  # >= 2048 (point, view) rows per product: the tensor-core kernels take over
  batch, feat_c, _, frame, t, offs, model, args = scenes.build(cfg)
  with torch.no_grad():  # larger motion than the bench initialisation so that its gradients are well above rounding
    model.motion_mlp.coeff_linear.weight.normal_(0.0, 0.05)
  g = torch.Generator().manual_seed(99)
  # ---- oracle (CPU): leaf copies of everything trainable
  shift = model.net_coarse_dy.shift
  om = type(model)(**vars(model))
  om.net_coarse_dy = _leaves(model.net_coarse_dy, shift)
  om.net_coarse_st = _leaves(model.net_coarse_st)
  om.motion_mlp = _leaves(model.motion_mlp)
  fo = tuple(f.clone().requires_grad_(True) for f in feat_c)
  want = orc.render_rays_mono(frame, t, offs, batch, om, fo, None, cfg["N_samples"], args,
                              inv_uniform=cfg["inv_uniform"], det=True, is_train=True, num_vv=cfg["num_vv"])
  gens = {(o, k): torch.randn(want[o][k].shape, generator=g) for o, ks in _TRAIN_KEYS.items() for k in ks}
  sum((want[o][k] * v).sum() for (o, k), v in gens.items()).backward()
  # ---- library (GPU)
  dev = torch.device(DEV)
  m_dev = synthetic.model_to(model, dev)
  for mod in (m_dev.net_coarse_dy, m_dev.net_coarse_st, m_dev.motion_mlp):
    mod.requires_grad_(True)
  fd = tuple(f.to(dev).requires_grad_(True) for f in feat_c)
  got = rr.render_rays_mono(frame, t, offs, synthetic.to_device(batch, dev), m_dev, fd, Projector(dev),
                            cfg["N_samples"], args, inv_uniform=cfg["inv_uniform"], det=True, is_train=True,
                            num_vv=cfg["num_vv"], precision=prec)
  ft = dict(rtol=1e-3, atol=2e-4) if prec == "fp32" else dict(rtol=3e-2, atol=2e-2)
  for (o, k), v in gens.items():
    assert got[o][k].requires_grad, (o, k)
    if prec == "bf16" and k == "render_flows":
      continue  # pixels: a bf16-sized change of the weights moves the expected point by a fraction of a pixel
    torch.testing.assert_close(got[o][k].detach().cpu(), want[o][k].detach(),
                               msg=lambda s: "%s/%s: %s" % (o, k, s), **ft)
  for o in ("outputs_coarse_anchor", "outputs_coarse_anchor_dy"):  # detached in the reference (:1222, :1254)
    assert not got[o]["occ_weights"].requires_grad and not got[o]["occ_weight_map"].requires_grad
    torch.testing.assert_close(got[o]["occ_weights"].cpu(), want[o]["occ_weights"].detach(), **ft)
  assert not got["outputs_coarse_ref"]["exp_sf"].requires_grad
  sum((got[o][k] * v.to(dev)).sum() for (o, k), v in gens.items()).backward()
  for mname, w in (("net_coarse_dy", om.net_coarse_dy), ("net_coarse_st", om.net_coarse_st),
                   ("motion_mlp", om.motion_mlp)):
    for k, p in getattr(m_dev, mname).named_parameters():
      assert p.grad is not None, (mname, k)
      if mname == "motion_mlp" and motion_off:
        assert not p.grad.any(), (mname, k)
      if mname == "net_coarse_st" and k == "s":
        # ill-conditioned in fp32 on this rig (far samples: cos ~ 1 for every view, so the pooling weights are
        # (e - min e) / (sum + 1e-8) with sum ~ 1e-6): torch's own fp32 autograd differs from its fp64 autograd by
        # 300 % here (profiles/r02_train.md); the well-conditioned case is test_net_static_backward_*
        assert torch.isfinite(p.grad).all()
        continue
      # bar: 5e-3 for weight matrices -- torch's own fp32 autograd is 1.5e-3 away from its fp64 autograd on this rig
      # (profiles/r02_train.md) -- and 2e-2 for bias / LayerNorm vectors: column sums over all rows whose terms cancel
      # to ~1e-3 of their magnitude (e.g. the blending head: sum_v d logit_v = 0 per point), so the summation order
      # shows; a wrong or missing term is an O(1) error
      if prec == "fp32":
        _close("%s.%s" % (mname, k), p.grad, w[k].grad, 5e-3 if p.dim() > 1 else 2e-2)
      elif mname == "motion_mlp" and k.startswith("pts_linears"):
        # ReLU network with bf16 products: pre-activations within bf16 rounding of 0 (~0.3 % of the units per layer)
        # take the other side of the kink, each flip is an O(1) change of that unit's gradient -> sqrt(0.003) ~ 5 %
        # in L2 at the last hidden layer, growing to ~11 % at the first (measured: profiles/r02_train.md); the smooth
        # (ELU) aggregation nets stay at 0.2 - 0.5 %
        _close("%s.%s" % (mname, k), p.grad, w[k].grad, 2e-1, floor=1e-5)
      else:  # bf16 operands: 2^-9 per element, averaged over the reductions and chained through ~10 layers
        _close("%s.%s" % (mname, k), p.grad, w[k].grad, 5e-2 if p.dim() > 1 else 1.5e-1, floor=1e-5)
  for i in range(3):
    _close("featmaps[%d]" % i, fd[i].grad, fo[i].grad, 5e-3 if prec == "fp32" else 5e-2)


@pytest.mark.parametrize("rows,out,width,ldx_pad,scaled", [(5000, 128, 128, 0, False), (9000, 129, 70, 0, True),
                                                          (4100, 256, 256, 0, False), (3000, 35, 66, 3, True),
                                                          (20000, 64, 128, 1, False)])
def test_tensorcore_training_products(rows, out, width, ldx_pad, scaled):
  """csrc/train_tc.cu: dW += dZ^T X (MN-major UMMA operands, reduction over the rows) and dIn = dZ W on tcgen05
  against fp64 products of the bf16-rounded operands (what the tensor cores multiply), fp32 accumulation."""
  from dynibar_b200._lib import lib, ptr, check, stream
  g = torch.Generator().manual_seed(rows + out)
  dz = torch.randn(rows, out, generator=g)
  ldx = width + ldx_pad
  xfull = torch.randn(rows, ldx, generator=g)
  sc = torch.rand(rows, generator=g) + 0.5 if scaled else None
  r16 = lambda t: t.to(torch.bfloat16).double()
  xs = xfull[:, :width] * sc[:, None] if scaled else xfull[:, :width]
  want_w = r16(dz).t() @ r16(xs)
  dzd, xd = dz.to(DEV), xfull.to(DEV)
  dW = torch.zeros(out, width + 2, device=DEV)  # leading dimension larger than the width
  with torch.cuda.device(DEV):
    check(lib.dyn_debug_tc_grad_w(ptr(dzd), out, out, rows, ptr(xd), ldx, width,
                                  ptr(sc.to(DEV)) if scaled else None, ptr(dW), width + 2, stream()))
  got_w = dW[:, :width].cpu().double()
  assert (dW[:, width:] == 0).all()
  err = (got_w - want_w).norm() / want_w.norm()
  assert err < 2e-5, ("grad_w", err.item())
  # dIn = dZ W[:, :width] with W [out, ldw]
  if width >= 16 and out >= 16:
    ldw = width + 5
    W = torch.randn(out, ldw, generator=g) * 0.1
    want_in = r16(dz) @ r16(W[:, :width])
    nb = int(lib.dyn_debug_tc_grad_in_scratch_bytes())
    scratch = torch.empty(nb, dtype=torch.uint8, device=DEV)
    din = torch.full((rows, width + 1), 7.0, device=DEV)
    with torch.cuda.device(DEV):
      check(lib.dyn_debug_tc_grad_in(ptr(dzd), out, out, rows, ptr(W.to(DEV)), ldw, width, ptr(din), width + 1,
                                     scratch.data_ptr(), nb, stream()))
    assert (din[:, width] == 7.0).all()
    err = (din[:, :width].cpu().double() - want_in).norm() / want_in.norm()
    assert err < 2e-5, ("grad_in", err.item())


def test_training_ray_slices_match_one_call(monkeypatch):
  """Ray batches whose (point, view) rows exceed one internal chunk are rendered in slices: same outputs, same
  gradients (accumulated over the slices by autograd) as the single call."""
  from dynibar_b200 import render_ray as rr
  from dynibar_b200.projection import Projector
  cfg = dict(scenes.GOLDEN_CONFIGS["mono_train"])
  batch, feat_c, _, frame, t, offs, model, args = scenes.build(cfg)
  dev = torch.device(DEV)
  m_dev = synthetic.model_to(model, dev)
  mods = (m_dev.net_coarse_dy, m_dev.net_coarse_st, m_dev.motion_mlp)
  for mod in mods:
    mod.requires_grad_(True)
  b = synthetic.to_device(batch, dev)
  g = torch.Generator().manual_seed(4)
  results = []
  for limit in (rr.TRAIN_ROWS_LIMIT, 7 * cfg["N_samples"] * 8):  # the second forces slices of 7 rays
    monkeypatch.setattr(rr, "TRAIN_ROWS_LIMIT", limit)
    for mod in mods:
      mod.zero_grad(set_to_none=True)
    fd = tuple(f.to(dev).requires_grad_(True) for f in feat_c)
    got = rr.render_rays_mono(frame, t, offs, b, m_dev, fd, Projector(dev), cfg["N_samples"], args,
                              inv_uniform=True, det=True, is_train=True, num_vv=cfg["num_vv"], precision="fp32")
    if not results:
      gens = {(o, k): torch.randn(got[o][k].shape, generator=g).to(dev) for o, ks in _TRAIN_KEYS.items() for k in ks}
    sum((got[o][k] * v).sum() for (o, k), v in gens.items()).backward()
    # (`s`: ill-conditioned sum, see above -- its value depends on the summation order)
    results.append((got, [p.grad.clone() for mod in mods for k, p in mod.named_parameters() if k != "s"],
                    [f.grad.clone() for f in fd]))
  (a, ga, fa), (bb, gb, fb) = results
  for o, ks in _TRAIN_KEYS.items():
    for k in ks:
      torch.testing.assert_close(bb[o][k], a[o][k], rtol=1e-5, atol=1e-6, msg=lambda s: "%s/%s: %s" % (o, k, s))
  assert torch.equal(bb["outputs_coarse_ref"]["mask"], a["outputs_coarse_ref"]["mask"])
  for x, y in zip(gb + fb, ga + fa):
    assert (x - y).norm().item() <= 2e-3 * y.norm().item() + 1e-6
