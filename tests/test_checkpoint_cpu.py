"""Checkpoint ingest (row f4): dicts / files in the reference's save layout (ibrnet/model.py:177-232,
:424-468) load strictly into the parameter containers, reproduce the flat parameter blob the CUDA library
packs, and checkpoints laid out as the REFERENCE's own nn.Modules write them load too."""

import os
from types import SimpleNamespace

import pytest
import torch

from dynibar_b200 import model as dmodel, synthetic, weights


def _args():
  a = synthetic.make_args(1, 0)
  a.N_samples, a.N_importance, a.coarse_feat_dim, a.fine_feat_dim = 16, 16, 32, 32
  return a


def _same_blobs(m1, m2):
  for k, v in vars(m1).items():
    w = getattr(m2, k)
    if isinstance(v, torch.nn.Module):
      assert torch.equal(weights.flatten(v), weights.flatten(w)), k
      assert list(v.state_dict().keys()) == list(w.state_dict().keys())
    else:
      assert torch.equal(v, w), k


def test_round_trip_through_files(tmp_path):
  args = _args()
  model, _ = synthetic.make_model(16, 16, args=args, seed=5)
  coarse, fine = dmodel.checkpoint_dicts(model, global_step=1234)
  coarse["optimizer"], coarse["scheduler"] = {"state": {}}, {"last_epoch": 3}  # present in real files; ignored
  pc, pf = str(tmp_path / "coarse_001234.pth"), str(tmp_path / "model_001234.pth")
  torch.save(coarse, pc)
  torch.save(fine, pf)
  got, info = dmodel.model_from_checkpoints(args, coarse=pc, fine=pf)
  assert info["coarse_step"] == 1234 and info["fine_step"] == 1234
  _same_blobs(model, got)
  assert got.net_coarse_dy.shift == 0.0 and got.net_fine_st.n_samples == 32


def test_mono_checkpoint_and_dataparallel_prefix():
  args = _args()
  model, _ = synthetic.make_model(16, 0, args=args, seed=6, mono=True)
  coarse, fine = dmodel.checkpoint_dicts(model)
  assert fine is None
  coarse["net_coarse_st"] = {"module." + k: v for k, v in coarse["net_coarse_st"].items()}
  coarse["feature_net"] = {"conv1.weight": torch.zeros(1)}
  got, info = dmodel.model_from_checkpoints(args, coarse=coarse, mono=True)
  _same_blobs(model, got)
  assert got.net_coarse_dy.shift == 5.0 and "feature_net" in info["encoders"]


def test_strict_loading_rejects_a_wrong_layout():
  args = _args()
  model, _ = synthetic.make_model(16, 16, args=args, seed=7)
  coarse, _ = dmodel.checkpoint_dicts(model)
  del coarse["net_coarse_dy"]["vis_fc.2.weight"]
  with pytest.raises(RuntimeError):
    dmodel.model_from_checkpoints(args, coarse=coarse)


def test_checkpoint_written_by_the_reference_modules_loads():
  """State dicts laid out exactly as the reference's own modules write them: names, order, shapes and dtypes
  (tests/golden/checkpoint_layout.pt from make_golden_checks.py), filled with seeded values."""
  layout = torch.load(os.path.join(os.path.dirname(__file__), "golden", "checkpoint_layout.pt"), weights_only=False)
  g = torch.Generator().manual_seed(3)

  def state_dict(entries):
    return {name: torch.randn(shape, generator=g).to(getattr(torch, dtype.split(".")[1]))
            for name, shape, dtype in entries}

  args = _args()
  fine = {"net_fine_st": state_dict(layout["net_fine_st"]),
          "net_fine_dy": state_dict(layout["net_fine_dy"]),
          "motion_mlp_fine": state_dict(layout["motion_mlp_fine"]),
          "traj_basis_fine": dmodel.init_dct_basis(6, 24), "global_step": 7}
  got, info = dmodel.model_from_checkpoints(args, fine=fine)
  for key, name in (("net_fine_st", "net_fine_st"), ("net_fine_dy", "net_fine_dy"), ("motion_mlp_fine", "motion_mlp_fine")):
    want = torch.cat([v.reshape(-1).float() for v in fine[key].values()])
    assert torch.equal(weights.flatten(getattr(got, name)), want), key
