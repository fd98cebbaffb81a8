"""2-D feature encoder (row f1) against the reference's own ResNet (ibrnet/feature_network.py:179-311):
committed fixtures of the unmodified reference module on the same weights (tests/golden/encoder.pt, and
tests/golden/encoder_shapes.pt from make_golden_checks.py)."""

import os

import pytest
import torch

from dynibar_b200 import feature_network as fn

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(__file__), "golden", "encoder.pt")
GOLD_SHAPES = os.path.join(os.path.dirname(__file__), "golden", "encoder_shapes.pt")
SAMPLE = 2048  # elements of each output map stored in GOLD_SHAPES


def _model(seed):
  torch.manual_seed(seed)
  m = fn.ResNet()
  with torch.no_grad():  # non-trivial affine parameters / biases (defaults are 1 / 0)
    for name, p in m.named_parameters():
      if name.endswith("bn1.weight") or name.endswith("bn2.weight") or name.endswith("downsample.1.weight"):
        p.uniform_(0.5, 1.5)
      elif name.endswith(".bias"):
        p.uniform_(-0.3, 0.3)
  return m.requires_grad_(False)


def _input(N, H, W):
  return torch.rand(N, 3, H, W, generator=torch.Generator().manual_seed(N * 1000 + H + 1))


def _sample_index(numel, seed):
  return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:SAMPLE]


def test_encoder_matches_reference_fixture():
  fx = torch.load(GOLD, weights_only=False)
  m = _model(fx["seed"])
  g = torch.Generator().manual_seed(fx["seed"] + 1)
  x = torch.rand(*fx["shape"], generator=g)
  assert abs(float(x.double().sum()) - fx["input_sum"]) < 1e-6 * fx["input_sum"]
  c, f = m.to(DEV)(x.to(DEV))
  torch.cuda.synchronize()
  assert c.shape == fx["coarse"].shape and f.shape == fx["fine"].shape
  torch.testing.assert_close(c.cpu(), fx["coarse"], rtol=2e-4, atol=2e-4)
  torch.testing.assert_close(f.cpu(), fx["fine"], rtol=2e-4, atol=2e-4)


@pytest.mark.parametrize("N,H,W", [(2, 288, 512), (3, 37, 53), (1, 135 * 4 // 4, 240)])
def test_encoder_matches_live_reference(N, H, W):
  """The reference ResNet's outputs on these weights and inputs, a seeded sample of each map."""
  fx = torch.load(GOLD_SHAPES, weights_only=False)[(N, H, W)]
  m = _model(N * 1000 + H)
  x = _input(N, H, W)
  assert abs(float(x.double().sum()) - fx["input_sum"]) < 1e-6 * fx["input_sum"]
  c, f = m.to(DEV)(x.to(DEV))
  torch.cuda.synchronize()
  for name, out, seed in (("coarse", c, 1), ("fine", f, 2)):
    assert tuple(out.shape) == fx[name + "_shape"], name
    idx = _sample_index(out.numel(), seed)
    torch.testing.assert_close(out.cpu().reshape(-1)[idx], fx[name], rtol=2e-4, atol=2e-4)


def test_encoder_feeds_the_renderer_layout():
  """[V,3,H,W] images -> [V,32,H/4,W/4] maps, the `featmaps` layout render_rays_* take."""
  m = _model(1).to(DEV)
  c, f = m(torch.rand(8, 3, 288, 512, device=DEV))
  assert c.shape == (8, 32, 72, 128) and f.shape == (8, 32, 72, 128) and torch.isfinite(c).all()


@pytest.mark.parametrize("N,H,W,prec", [(2, 60, 84, "fp32"), (3, 37, 53, "fp32"), (2, 192, 256, "bf16")])
def test_encoder_backward_matches_oracle_autograd(N, H, W, prec):
  """Row f2: gradients of every executed encoder parameter against torch autograd through the oracle's restatement of
  ResNet.forward (pinned to the reference by tests/test_oracle_golden.py).  fp32: 2e-3 relative L2 per tensor
  (InstanceNorm + ReLU network; the ReLU kinks make a few units flip with the summation order); bf16 products
  (tcgen05): 1e-1."""
  from dynibar_b200 import render_ray as rr
  from oracle import dynibar_oracle as orc
  m = _model(N * 100 + H).requires_grad_(True)
  g = torch.Generator().manual_seed(N + H)
  x = torch.rand(N, 3, H, W, generator=g)
  w = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items() if k in fn._EXECUTED}
  wc, wf = orc.encoder_forward(w, x)
  gc, gf = torch.randn(wc.shape, generator=g), torch.randn(wf.shape, generator=g)
  ((wc * gc).sum() + (wf * gf).sum()).backward()
  md = m.to(DEV)
  with rr.precision_scope(prec):
    c, f = md(x.to(DEV))
    assert c.requires_grad and f.requires_grad
    ((c * gc.to(DEV)).sum() + (f * gf.to(DEV)).sum()).backward()
  torch.testing.assert_close(c.detach().cpu(), wc.detach(), rtol=2e-4, atol=2e-4)
  tol = 2e-3 if prec == "fp32" else 1e-1
  sd = md.state_dict(keep_vars=True)
  for k in fn._EXECUTED:
    assert sd[k].grad is not None, k
    d = (sd[k].grad.cpu().double() - w[k].grad.double()).norm().item()
    assert d <= tol * w[k].grad.double().norm().item() + 1e-6, (k, d, w[k].grad.norm().item())
  for k, p in md.named_parameters():  # parameters the reference builds but never runs get no gradient
    if k not in fn._EXECUTED:
      assert p.grad is None, k
