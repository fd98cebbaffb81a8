"""dynibar_b200.criterion (csrc/objective.cu) against torch autograd through the restatement of the reference
objective (tests/objective_oracle.py, train.py:300-458, :187-196) evaluated in fp64.

Bars: loss and terms rtol 1e-5; gradients 1e-5 relative in the L2 norm per tensor and max-abs within 10x that
(`_close` of test_train_gpu.py).  The kernels evaluate every per-ray quantity in fp64 and round only the outputs to
fp32, so the remaining difference is that rounding."""

import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import objective_oracle as oo
import scenes
from dynibar_b200 import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
_KEYS1 = ("render_flows", "pts_traj_ref", "pts_traj_anchor", "sf_seq")  # ray axis 1; every other key: axis 0
_DIFF = {"outputs_coarse_ref": ("rgb", "rgb_dy", "rgb_static", "depth", "weights", "weights_dy", "weights_st",
                                "render_flows"),
         "outputs_coarse_ref_dy": ("rgb",),
         "outputs_coarse_anchor": ("rgb", "pts_traj_ref", "pts_traj_anchor", "sf_seq"),
         "outputs_coarse_anchor_dy": ("rgb",),
         "outputs_coarse_st": ("rgb",)}
SCHEDULES = {  # name -> (epoch, anneal_cycle) with init_decay_epoch = 10
    "warmup": (3, False), "divisor1": (14, False), "divisor1_anneal": (17, True), "divisor5": (55, True)}


def _args(anneal):
  return SimpleNamespace(w_disp=5e-2, w_flow=5e-3, w_cycle=0.1, cycle_factor=0.1, anneal_cycle=anneal, w_reg=0.05,
                         w_skew_entropy=1e-3, w_distortion=1e-3, decay_rate=10.0, init_decay_epoch=10)


def make_ret(R, S, K, seed, device=DEV):
  """Seeded stand-in for render_rays_mono(is_train=True) outputs (the keys and shapes the objective reads) and
  the supervision of make_supervision."""
  g = torch.Generator().manual_seed(seed)
  u = lambda *s: torch.rand(*s, generator=g)
  n = lambda *s: torch.randn(*s, generator=g)
  msk = lambda p: u(R) < p
  wdy = u(R, S) / S
  wdy[::3] *= 0.01  # rays with a dynamic / total weight ratio below 0.1 (train.py:438)
  ret = {
      "outputs_coarse_ref": {"rgb": u(R, 3), "rgb_dy": u(R, 3), "rgb_static": u(R, 3), "depth": u(R) * 8 + 0.2,
                             "mask": msk(0.8), "weights": u(R, S) / S, "weights_dy": wdy, "weights_st": u(R, S) / S,
                             "s_vals": torch.sort(u(R, S), dim=1).values, "render_flows": n(6, R, 2) * 2},
      "outputs_coarse_ref_dy": {"rgb": u(R, 3), "mask": msk(0.7)},
      "outputs_coarse_anchor": {"rgb": u(R, 3), "mask": msk(0.8), "occ_weight_map": u(R), "occ_weights": u(R, S),
                                "pts_traj_ref": n(K, R, S, 3), "pts_traj_anchor": n(K, R, S, 3),
                                "sf_seq": n(6, R, S, 3) * 0.1},
      "outputs_coarse_anchor_dy": {"rgb": u(R, 3), "mask": msk(0.7), "occ_weight_map": u(R)},
      "outputs_coarse_st": {"rgb": u(R, 3)},
  }
  batch = synthetic.make_supervision({"ray_o": torch.zeros(R, 3)}, n_flow=6, seed=seed + 1)
  return synthetic.to_device(ret, device), synthetic.to_device(batch, device)


def leaves(ret, dtype=torch.float32):
  """Copy of `ret` whose differentiable entries are leaf tensors of `dtype` (masks stay bool)."""
  out = {}
  for o, d in ret.items():
    out[o] = {}
    for k, v in d.items():
      if v.dtype == torch.bool:
        out[o][k] = v
      elif k in _DIFF[o]:
        out[o][k] = v.detach().to(dtype).clone().requires_grad_(True)
      else:
        out[o][k] = v.detach().to(dtype)
  return out


def grads(ret):
  return {(o, k): ret[o][k].grad for o, ks in _DIFF.items() for k in ks}


def _close(name, got, ref, tol=1e-5, floor=1e-12):
  assert got is not None and ref is not None, name
  d = got.detach().double() - ref.detach().double()
  rn = ref.detach().double().norm().item()
  assert d.norm().item() <= tol * rn + floor, (name, d.norm().item(), rn)
  assert d.abs().max().item() <= 10 * tol * ref.detach().double().abs().max().item() + floor, (name,
                                                                                             d.abs().max().item())


def _scalar_close(name, got, want, rtol=1e-5, atol=1e-12):
  g, w = float(got), float(want)
  assert abs(g - w) <= rtol * abs(w) + atol, (name, g, w)


def _run_both(ret, batch, args, epoch, oracle_dtype=torch.float64):
  from dynibar_b200 import criterion as cr
  lg = leaves(ret)
  loss, terms = cr.dynibar_objective(lg, batch, args, epoch)
  loss.backward()
  lw = leaves(ret, oracle_dtype)
  bw = {k: (v.to(oracle_dtype) if v.is_floating_point() else v) for k, v in batch.items()}
  want, wterms = oo.objective(lw, bw, args, epoch)
  want.backward()
  return (loss, terms, grads(lg)), (want, wterms, grads(lw))


def _check(got, want, skip_grads=()):
  (loss, terms, gg), (wl, wt, gw) = got, want
  _scalar_close("loss", loss, wl)
  assert sorted(terms) == sorted(wt)
  for k in wt:
    _scalar_close(k, terms[k], wt[k])
  for key in gw:
    if key in skip_grads:
      continue
    if gw[key] is None:  # an input the reference's loss does not read at this epoch: zero gradient (or none)
      assert gg[key] is None or not gg[key].any(), key
      continue
    _close("d loss / d %s[%s]" % key, gg[key], gw[key])


@pytest.mark.parametrize("schedule", sorted(SCHEDULES))
@pytest.mark.parametrize("K", [1, 6])
@pytest.mark.parametrize("S", [2, 33, 64, 128])
@pytest.mark.parametrize("R", [1, 1000, 3072])
def test_objective_matches_fp64_autograd(R, S, K, schedule):
  epoch, anneal = SCHEDULES[schedule]
  ret, batch = make_ret(R, S, K, seed=R + 7 * S + K)
  _check(*_run_both(ret, batch, _args(anneal), epoch))


def test_objective_edge_cases():
  """All masks zero (only the epsilon denominators remain); depths below the clamp and exactly on it; weight ratios
  exactly 0 and 1 and a ray without weight; exact ties (abs'(0) = 0) in the trajectories, sf_seq and flows."""
  R, S, K = 300, 40, 6
  ret, batch = make_ret(R, S, K, seed=5)
  # ---- all masks zero
  z = {o: dict(d) for o, d in ret.items()}
  for o in ("outputs_coarse_ref", "outputs_coarse_ref_dy", "outputs_coarse_anchor", "outputs_coarse_anchor_dy"):
    z[o]["mask"] = torch.zeros_like(z[o]["mask"])
  z["outputs_coarse_anchor"]["occ_weights"] = torch.zeros(R, S, device=DEV)
  zb = dict(batch, motion_mask=torch.zeros(R, device=DEV), static_mask=torch.zeros(R, device=DEV),
            masks=torch.zeros(6, R, 1, device=DEV))
  for sched in ("warmup", "divisor5"):
    epoch, anneal = SCHEDULES[sched]
    _check(*_run_both(z, zb, _args(anneal), epoch))
  # ---- thresholds and ties
  e = {o: {k: v.clone() for k, v in d.items()} for o, d in ret.items()}
  ref, anc = e["outputs_coarse_ref"], e["outputs_coarse_anchor"]
  ref["depth"][:20] = torch.rand(20, device=DEV) * 0.009
  ref["depth"][20:25] = torch.tensor(1e-2, dtype=torch.float32)  # exactly on the fp32 clamp
  ref["mask"][:25] = True
  ref["weights_dy"][30:40] = 0.0   # ratio 0
  ref["weights_st"][40:50] = 0.0   # ratio 1
  ref["weights_dy"][50:55] = 0.0   # no weight at all: clamp(0, 1e-9)
  ref["weights_st"][50:55] = 0.0
  anc["pts_traj_anchor"][:, :100] = anc["pts_traj_ref"][:, :100]
  anc["sf_seq"][:, :50, :10] = 0.0                       # |sf| at 0 and equal temporal / spatial neighbours
  anc["sf_seq"][2, 60:80] = anc["sf_seq"][3, 60:80]
  ref["render_flows"][:, 100:150] = batch["flows"][:, 100:150]
  for sched in ("warmup", "divisor1", "divisor5"):
    epoch, anneal = SCHEDULES[sched]
    depth_key = ("outputs_coarse_ref", "depth")
    got, want = _run_both(e, batch, _args(anneal), epoch)
    _check(got, want, skip_grads=(depth_key,))
    # the depth gradient at the clamp: the fp32 tensor sits on the threshold, so compare with the oracle in fp32
    _, want32 = _run_both(e, batch, _args(anneal), epoch, oracle_dtype=torch.float32)
    _close("d loss / d depth (fp32 oracle)", got[2][depth_key], want32[2][depth_key])
    _scalar_close("disp_loss (fp32 oracle)", got[1]["disp_loss"], want32[1]["disp_loss"])
    assert (got[2][depth_key][20:25] != 0).any() and (got[2][depth_key][:20] == 0).all()


def test_objective_is_deterministic():
  from dynibar_b200 import criterion as cr
  ret, batch = make_ret(3072, 64, 6, seed=9)
  runs = []
  for _ in range(3):
    lg = leaves(ret)
    loss, terms = cr.dynibar_objective(lg, batch, _args(True), 55)
    loss.backward()
    runs.append([loss.detach().clone()] + [terms[k].detach().clone() for k in sorted(terms)]
                + [v.clone() for v in grads(lg).values() if v is not None])
  for other in runs[1:]:
    for a, b in zip(runs[0], other):
      assert torch.equal(a, b)


def test_objective_launches_and_no_host_sync():
  from dynibar_b200 import criterion as cr
  from dynibar_b200._lib import lib
  ret, batch = make_ret(1024, 64, 6, seed=3)
  lg = leaves(ret)
  cr.dynibar_objective(leaves(ret), batch, _args(False), 3)[0].backward()  # warm-up (workspace, modules)
  torch.cuda.synchronize()
  n0 = lib.dyn_launch_count(0)
  torch.cuda.set_sync_debug_mode("error")
  try:
    loss, terms = cr.dynibar_objective(lg, batch, _args(False), 3)
    loss.backward()
    n_both = lib.dyn_launch_count(0) - n0
    boot = cr.static_bootstrap_loss(lg, batch)
    boot.backward()
    w = ret["outputs_coarse_ref"]["weights"].clone().requires_grad_(True)
    s = ret["outputs_coarse_ref"]["s_vals"]
    cr.eff_distloss_native(w, s, s).backward()
  finally:
    torch.cuda.set_sync_debug_mode("default")
  assert n_both <= 3, n_both
  assert lib.dyn_launch_count(0) - n0 <= 9
  torch.cuda.synchronize()


def test_static_bootstrap_and_distloss_match_oracle():
  from dynibar_b200 import criterion as cr
  ret, batch = make_ret(1000, 33, 1, seed=12)
  lg, lw = leaves(ret), leaves(ret, torch.float64)
  got = cr.static_bootstrap_loss(lg, batch)
  want = oo.static_bootstrap_loss(lw, {k: v.double() for k, v in batch.items()})
  _scalar_close("static bootstrap", got, want)
  got.backward()
  want.backward()
  _close("d bootstrap / d st.rgb", lg["outputs_coarse_st"]["rgb"].grad, lw["outputs_coarse_st"]["rgb"].grad)
  # eff_distloss_native with leading dims and S = 2
  for shape in ((4, 5, 2), (1000, 63)):
    g = torch.Generator().manual_seed(shape[-1])
    w = torch.rand(*shape, generator=g).to(DEV)
    s = torch.sort(torch.rand(*shape[:-1], shape[-1] + 1, generator=g), -1).values.to(DEV)
    m, iv = (s[..., 1:] + s[..., :-1]) * 0.5, s[..., 1:] - s[..., :-1]
    wg, ww = w.clone().requires_grad_(True), w.double().requires_grad_(True)
    a = cr.eff_distloss_native(wg, m, iv)
    b = oo.eff_distloss_native(ww, m.double(), iv.double())
    _scalar_close("eff_distloss_native %s" % (shape,), a, b)
    a.backward()
    b.backward()
    _close("d distloss / d w %s" % (shape,), wg.grad, ww.grad)


def _render_step(objective, cfg, is_train=True):
  """render_rays_mono on the seeded scene + supervision, then objective(ret, ray_batch).backward(); returns the
  gradients of every trainable parameter and feature map."""
  from dynibar_b200 import render_ray as rr
  from dynibar_b200.projection import Projector
  batch, feat_c, _, frame, t, offs, model, args = scenes.build(cfg)
  with torch.no_grad():
    model.motion_mlp.coeff_linear.weight.normal_(0.0, 0.05)
  dev = torch.device(DEV)
  m = synthetic.model_to(model, dev)
  mods = (m.net_coarse_dy, m.net_coarse_st, m.motion_mlp)
  for mod in mods:
    mod.requires_grad_(True)
  fd = tuple(f.to(dev).requires_grad_(True) for f in feat_c)
  b = synthetic.make_supervision(synthetic.to_device(batch, dev), n_flow=6, seed=cfg["seed"])
  ret = rr.render_rays_mono(frame, t, offs, b, m, fd, Projector(dev), cfg["N_samples"], args,
                            inv_uniform=cfg["inv_uniform"], det=True, is_train=is_train, num_vv=cfg["num_vv"],
                            precision="fp32")
  objective(ret, b).backward()
  out = {}
  for name, mod in (("net_coarse_dy", m.net_coarse_dy), ("net_coarse_st", m.net_coarse_st),
                    ("motion_mlp", m.motion_mlp)):
    for k, p in mod.named_parameters():
      out["%s.%s" % (name, k)] = p.grad
  for i, f in enumerate(fd):
    out["featmaps[%d]" % i] = f.grad
  return out


def _double(ret):
  return {o: ({k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in d.items()}
              if d is not None else None) for o, d in ret.items()}


@pytest.mark.parametrize("epoch", [3, 55])
def test_training_step_with_objective_matches_oracle_objective(epoch):
  """render_rays_mono(is_train=True) -> dynibar_objective -> backward against the same step with the fp64 oracle
  objective.  Bar 1e-4: the render backward itself reduces with float atomics."""
  from dynibar_b200 import criterion as cr
  cfg = dict(scenes.GOLDEN_CONFIGS["mono_train"])
  args = _args(True)
  got = _render_step(lambda ret, b: cr.dynibar_objective(ret, b, args, epoch)[0], cfg)
  bd = lambda b: {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in b.items()}
  want = _render_step(lambda ret, b: oo.objective(_double(ret), bd(b), args, epoch)[0], cfg)
  for k in want:
    if want[k] is None:
      assert got[k] is None, k
      continue
    _close(k, got[k], want[k], tol=1e-4, floor=1e-9)


def test_bootstrap_step_matches_oracle():
  from dynibar_b200 import criterion as cr
  cfg = dict(scenes.GOLDEN_CONFIGS["mono_train"])
  got = _render_step(cr.static_bootstrap_loss, cfg, is_train=False)
  bd = lambda b: {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in b.items()}
  want = _render_step(lambda ret, b: oo.static_bootstrap_loss(_double(ret), bd(b)), cfg, is_train=False)
  for k in want:
    if want[k] is None:
      assert got[k] is None, k
      continue
    _close(k, got[k], want[k], tol=1e-4, floor=1e-9)


def slice_rays(ret, batch, lo, hi):
  sl = lambda k, v: v[:, lo:hi] if k in _KEYS1 else v[lo:hi]
  r = {o: {k: sl(k, v) for k, v in d.items()} for o, d in ret.items()}
  b = {k: (v[:, lo:hi] if k in ("flows", "masks") else v[lo:hi]) for k, v in batch.items()}
  return r, b


@pytest.mark.parametrize("epoch", [3, 55])
def test_sharded_totals_give_full_batch_loss_and_gradients(epoch):
  from dynibar_b200 import criterion as cr
  R, args = 1001, _args(True)
  ret, batch = make_ret(R, 64, 6, seed=31)
  full = leaves(ret)
  loss_full, terms_full = cr.dynibar_objective(full, batch, args, epoch)
  loss_full.backward()
  lg = leaves(ret)
  halves = [slice_rays(lg, batch, 0, 500), slice_rays(lg, batch, 500, R)]
  totals = sum(cr.objective_sums(r, b, args, epoch) for r, b in halves)
  losses = []
  for r, b in halves:
    loss, terms = cr.dynibar_objective(r, b, args, epoch, totals=totals)
    _scalar_close("sharded loss", loss, loss_full, rtol=1e-6, atol=0)
    for k in terms:
      _scalar_close("sharded " + k, terms[k], terms_full[k], rtol=1e-6, atol=1e-12)
    losses.append(loss)
  (losses[0] + losses[1]).backward()
  for key, gw in grads(full).items():
    torch.testing.assert_close(grads(lg)[key], gw, rtol=1e-6, atol=1e-12, msg=str(key))


def _free_port():
  s = socket.socket()
  s.bind(("127.0.0.1", 0))
  p = s.getsockname()[1]
  s.close()
  return p


def _nccl_worker(rank, world, port, q):
  from dynibar_b200 import criterion as cr, distributed as dd
  os.environ["MASTER_ADDR"] = "127.0.0.1"
  os.environ["MASTER_PORT"] = str(port)
  dev = torch.device("cuda", rank)
  torch.cuda.set_device(dev)
  dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
  R, args = 777, _args(True)
  ret, batch = make_ret(R, 64, 6, seed=41, device=dev)
  params = leaves(ret)  # replicated "parameters": every rank renders its block of rays from them
  lo, hi = dd.shard_bounds(R, rank, world)
  r, b = slice_rays(params, batch, lo, hi)
  loss, _ = cr.dynibar_objective(r, b, args, 55, group=dist.group.WORLD)
  loss.backward()
  plist = [params[o][k] for o, ks in _DIFF.items() for k in ks]
  dd.allreduce_gradients(plist, average=False)
  if rank == 0:
    full = leaves(ret)
    want, _ = cr.dynibar_objective(full, batch, args, 55)
    want.backward()
    ok = abs(loss.item() - want.item()) <= 1e-6 * abs(want.item())
    for key, gw in grads(full).items():
      ok = ok and torch.allclose(params[key[0]][key[1]].grad, gw, rtol=1e-6, atol=1e-12)
    q.put(bool(ok))
  dist.barrier()
  dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_nccl_objective_matches_full_batch():
  ctx = mp.get_context("spawn")
  q = ctx.Queue()
  port = _free_port()
  procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
  for p in procs:
    p.start()
  ok = q.get(timeout=300)
  for p in procs:
    p.join(timeout=300)
    assert p.exitcode == 0
  assert ok


def test_rejects_bad_inputs_before_any_launch():
  from dynibar_b200 import criterion as cr
  from dynibar_b200._lib import lib
  ret, batch = make_ret(50, 16, 6, seed=2)
  args = _args(False)

  def bad(where, key, value, match, b=None):
    r = {o: dict(d) for o, d in ret.items()}
    if where == "ray_batch":
      b = dict(batch)
      b[key] = value
    else:
      r[where][key] = value
    n0 = lib.dyn_launch_count(0)
    with pytest.raises(RuntimeError, match=match):
      cr.dynibar_objective(r, b if b is not None else batch, args, 3)
    assert lib.dyn_launch_count(0) == n0

  ref = ret["outputs_coarse_ref"]
  bad("outputs_coarse_ref", "rgb", ref["rgb"].cpu(), r"outputs_coarse_ref\['rgb'\] is a cpu tensor")
  bad("ray_batch", "disp", batch["disp"].cpu(), r"ray_batch\['disp'\] is a cpu tensor")
  bad("outputs_coarse_ref", "depth", torch.rand(51, device=DEV), r"outputs_coarse_ref\['depth'\] has shape")
  bad("outputs_coarse_ref", "weights_dy", torch.rand(50, 17, device=DEV),
      r"outputs_coarse_ref\['weights_dy'\] has shape")
  bad("outputs_coarse_anchor", "pts_traj_anchor", torch.rand(5, 50, 16, 3, device=DEV),
      r"outputs_coarse_anchor\['pts_traj_anchor'\] has shape")
  bad("outputs_coarse_ref", "rgb", ref["rgb"].double(), r"outputs_coarse_ref\['rgb'\] has dtype torch.float64")
  bad("ray_batch", "masks", batch["masks"].long(), r"ray_batch\['masks'\] has dtype torch.int64")
  bad("outputs_coarse_anchor", "sf_seq", None, r"outputs_coarse_anchor\['sf_seq'\] is missing")
  with pytest.raises(RuntimeError, match="totals must be"):
    cr.dynibar_objective(ret, batch, args, 3, totals=torch.zeros(32, device=DEV))
