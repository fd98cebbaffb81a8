"""Host logic of the training path that needs no GPU: slicing of large ray batches and the merge of the per-slice
output dicts (dynibar_b200.render_ray._render_mono_train_chunked), routing of render_rays_mono."""

from collections import OrderedDict
from types import SimpleNamespace

import torch

from dynibar_b200 import render_ray as rr


def _fake_train(frame_idx, time_embedding, time_offset, ray_batch, model, featmaps, N_samples, args, inv_uniform, det,
                is_train, num_vv, jitter, train=True):
  """Stands in for the CUDA path: every output is a per-ray function of ray_o, in the reference's layouts."""
  assert train
  o = ray_batch["ray_o"]
  R = o.shape[0]
  s = o.sum(-1)
  out = OrderedDict(rgb=o * 2, depth=s, weights=s[:, None].expand(R, N_samples) * 1.0, mask=s > 0,
                    render_flows=torch.stack([o[:, :2] + k for k in range(6)]), exp_sf=o + 1)
  anchor = OrderedDict(rgb=o * 3, pts_traj_ref=torch.stack([o[:, None, :].expand(R, N_samples, 3) + k for k in range(4)]),
                       pts_traj_anchor=torch.stack([o[:, None, :].expand(R, N_samples, 3) - k for k in range(4)]),
                       sf_seq=torch.stack([o[:, None, :].expand(R, N_samples, 3) * k for k in range(6)]),
                       occ_weight_map=s * 0.5)
  if jitter is not None:
    out["jit"] = jitter.sum(1)
  return {"outputs_coarse": None, "outputs_fine": None, "outputs_coarse_ref": out, "outputs_coarse_anchor": anchor}


def test_training_slices_are_merged_along_the_ray_axis(monkeypatch):
  monkeypatch.setattr(rr, "_render_mono", _fake_train)
  g = torch.Generator().manual_seed(0)
  R, S, V = 23, 4, 3
  batch = {"ray_o": torch.randn(R, 3, generator=g), "ray_d": torch.randn(R, 3, generator=g),
           "uv_grid": torch.randn(R, 2, generator=g), "src_cameras": torch.zeros(1, V, 34),
           "static_src_cameras": torch.zeros(1, 2, 34), "anchor_src_cameras": torch.zeros(1, V, 34)}
  jit = torch.rand(R, S, generator=g)
  args = (None, None, None, batch, None, None, S, SimpleNamespace(), True, False, True, 2, jit)
  whole = _fake_train(*args)
  monkeypatch.setattr(rr, "TRAIN_ROWS_LIMIT", 5 * S * V)  # slices of 5 rays: 5 + 5 + 5 + 5 + 3
  got = rr._render_mono_train_chunked(*args)
  assert got["outputs_coarse"] is None and got["outputs_fine"] is None
  for name in ("outputs_coarse_ref", "outputs_coarse_anchor"):
    assert list(got[name].keys()) == list(whole[name].keys())
    for k, v in whole[name].items():
      assert got[name][k].shape == v.shape, (name, k)
      assert torch.equal(got[name][k], v), (name, k)
  monkeypatch.setattr(rr, "TRAIN_ROWS_LIMIT", 10 ** 9)  # one slice: the call is passed through untouched
  one = rr._render_mono_train_chunked(*args)
  assert torch.equal(one["outputs_coarse_ref"]["rgb"], whole["outputs_coarse_ref"]["rgb"])


def test_wants_grad_routing():
  lin = torch.nn.Linear(2, 2)
  model = SimpleNamespace(net=lin, basis=torch.zeros(3))
  fm = (torch.zeros(1), None, torch.zeros(1))
  assert rr._wants_grad(model, fm)
  with torch.no_grad():
    assert not rr._wants_grad(model, fm)
  lin.requires_grad_(False)
  assert not rr._wants_grad(model, fm)
  assert rr._wants_grad(model, (torch.zeros(1, requires_grad=True), None, torch.zeros(1)))
