"""The torch restatement of the training objective (tests/objective_oracle.py) on CPU: its criterion functions
against outputs and input gradients of the unmodified ibrnet/criterion.py stored in tests/golden/criterion.pt
(tests/golden/make_golden_criterion.py), and its eff_distloss_native against the pairwise definition of the
mip-NeRF 360 distortion loss."""

import types

import pytest
import torch

import objective_oracle as oo

CRITERION_SEED = 23
CRITERION_RAYS = 37


def criterion_inputs(seed=CRITERION_SEED, R=CRITERION_RAYS, n_flow=6):
  """Seeded inputs of the criterion fixture (fp32, CPU)."""
  g = torch.Generator().manual_seed(seed)
  return {
      "pred_rgb": torch.rand(R, 3, generator=g),
      "mask": (torch.rand(R, generator=g) > 0.3).float(),
      "occ_weight_map": torch.rand(R, generator=g),
      "gt_rgb": torch.rand(R, 3, generator=g),
      "motion_mask": (torch.rand(R, generator=g) > 0.5).float(),
      "render_flow": torch.randn(n_flow, R, 2, generator=g),
      "gt_flow": torch.randn(n_flow, R, 2, generator=g),
      "flow_mask": (torch.rand(n_flow, R, 1, generator=g) > 0.4).float(),
  }


def checksum(x):
  return float(sum(v.double().abs().sum() for _, v in sorted(x.items())))


def run_criterion_cases(ns, x):
  """Value and input gradients of each case.  `ns` provides criterion(outputs, ray_batch, motion_mask=None),
  compute_rgb_loss, compute_temporal_rgb_loss and compute_flow_loss (the reference's or the oracle's)."""
  out = {}

  def case(name, fn, inputs):
    leaves = {k: x[k].clone().requires_grad_(True) for k in inputs}
    v = fn(leaves)
    v.backward()
    out[name] = {"value": v.detach(), "grad": {k: t.grad for k, t in leaves.items()}}

  batch = lambda: {"rgb": x["gt_rgb"]}
  case("criterion", lambda l: ns.criterion({"rgb": l["pred_rgb"], "mask": x["mask"]}, batch()), ["pred_rgb"])
  case("criterion_motion", lambda l: ns.criterion({"rgb": l["pred_rgb"], "mask": x["mask"]}, batch(),
                                                  motion_mask=x["motion_mask"]), ["pred_rgb"])
  case("compute_rgb_loss", lambda l: ns.compute_rgb_loss(l["pred_rgb"], batch(), x["mask"] * x["motion_mask"]),
       ["pred_rgb"])
  tmp = lambda l: {"rgb": l["pred_rgb"], "mask": x["mask"], "occ_weight_map": x["occ_weight_map"]}
  case("temporal", lambda l: ns.compute_temporal_rgb_loss(tmp(l), batch()), ["pred_rgb"])
  case("temporal_motion", lambda l: ns.compute_temporal_rgb_loss(tmp(l), batch(), motion_mask=x["motion_mask"]),
       ["pred_rgb"])
  case("flow", lambda l: ns.compute_flow_loss(l["render_flow"], x["gt_flow"], x["mask"][None, :, None] *
                                              x["flow_mask"]), ["render_flow"])
  return out


def test_oracle_criterion_matches_reference_fixture(golden):
  fx = golden("criterion")
  x = criterion_inputs()
  assert abs(checksum(x) - fx["checksum"]) < 1e-6 * fx["checksum"], "seeded inputs drifted"
  got = run_criterion_cases(types.SimpleNamespace(criterion=oo.criterion, compute_rgb_loss=oo.compute_rgb_loss,
                                                  compute_temporal_rgb_loss=oo.compute_temporal_rgb_loss,
                                                  compute_flow_loss=oo.compute_flow_loss), x)
  assert sorted(got) == sorted(fx["cases"])
  for name, want in fx["cases"].items():
    torch.testing.assert_close(got[name]["value"], want["value"], rtol=1e-6, atol=0, msg=name)
    assert sorted(got[name]["grad"]) == sorted(want["grad"])
    for k, gw in want["grad"].items():
      torch.testing.assert_close(got[name]["grad"][k], gw, rtol=1e-6, atol=1e-12, msg="%s d/d %s" % (name, k))


@pytest.mark.parametrize("R,N", [(1, 2), (7, 2), (5, 33), (3, 64), (4, 129)])
def test_oracle_distloss_equals_pairwise_definition(R, N):
  g = torch.Generator().manual_seed(R * 1000 + N)
  w = torch.rand(R, N, generator=g, dtype=torch.float64)
  w[0] = 0.0  # a ray whose weights are all zero
  s = torch.sort(torch.rand(R, N + 1, generator=g, dtype=torch.float64), dim=-1).values
  m, iv = (s[:, 1:] + s[:, :-1]) * 0.5, s[:, 1:] - s[:, :-1]
  got = oo.eff_distloss_native(w, m, iv)
  want = oo.eff_distloss_pairwise(w, m, iv)
  assert abs(got.item() - want.item()) <= 1e-12 * abs(want.item()) + 1e-300, (got.item(), want.item())
  # and the gradients in w
  wa, wb = w.clone().requires_grad_(True), w.clone().requires_grad_(True)
  oo.eff_distloss_native(wa, m, iv).backward()
  oo.eff_distloss_pairwise(wb, m, iv).backward()
  assert (wa.grad - wb.grad).abs().max().item() <= 1e-12 * wb.grad.abs().max().item() + 1e-300


def test_oracle_distloss_all_zero_weights_is_zero():
  w = torch.zeros(3, 5, dtype=torch.float64)
  m = torch.arange(5, dtype=torch.float64).expand(3, 5)
  assert oo.eff_distloss_native(w, m, torch.ones(3, 5, dtype=torch.float64)).item() == 0.0


def test_make_supervision_layout_shards_unchanged():
  from dynibar_b200 import distributed as dd, synthetic
  batch = {"ray_o": torch.zeros(11, 3), "ray_d": torch.ones(11, 3), "uv_grid": torch.zeros(11, 2)}
  b = synthetic.make_supervision(batch, n_flow=6, seed=4)
  assert b["rgb"].shape == (11, 3) and b["disp"].shape == (11,) and b["flows"].shape == (6, 11, 2)
  assert b["masks"].shape == (6, 11, 1) and b["motion_mask"].shape == (11,) and b["static_mask"].shape == (11,)
  for k in ("motion_mask", "static_mask", "masks"):
    assert set(b[k].unique().tolist()) <= {0.0, 1.0}
  assert torch.equal(synthetic.make_supervision(batch, seed=4)["flows"], b["flows"])
  lo_part, (lo, hi) = dd.shard_ray_batch(b, 1, 2)
  for k in ("rgb", "disp", "motion_mask", "static_mask"):
    assert torch.equal(lo_part[k], b[k][lo:hi])
  for k in ("flows", "masks"):
    assert torch.equal(lo_part[k], b[k][:, lo:hi])


def test_objective_rejects_cpu_tensors_without_gpu():
  from dynibar_b200 import criterion as cr
  w = torch.rand(2, 4)
  with pytest.raises(RuntimeError, match="eff_distloss_native: w is a cpu tensor"):
    cr.eff_distloss_native(w, w, w)
