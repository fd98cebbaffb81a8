"""Fixtures of the checks that compare against the UNMODIFIED reference on inputs of their own
(run where the reference sources are, after build()):

    python tests/golden/make_golden_checks.py

  mv_seed77.pt          render_rays_mv on a second seeded scene (ibrnet/render_ray.py)
  sampler_17x23.pt      RaySamplerSingleImage.get_all at render_stride 1 and 3 (ibrnet/sample_ray.py:165-211)
  checkpoint_layout.pt  state_dict layout (names, order, shapes, dtypes) of the reference's DynibarStatic,
                        DynibarDynamic and MotionMLP (ibrnet/mlp_network.py) -- the values are random
                        initialisations and are regenerated from a seed by the test
  encoder_shapes.pt     the reference ResNet (ibrnet/feature_network.py:179-311) at three image shapes;
                        a fixed seeded sample of 2048 elements of each output map

Like make_golden.py the fixtures hold reference OUTPUTS only; inputs and weights are regenerated from
seeds and guarded by a checksum.
"""

import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import make_golden as mg  # noqa: E402
import scenes  # noqa: E402

MV_CFG = dict(scenes.GOLDEN_CONFIGS["mv_small"], seed=77, rays=16, V_dy=7, V_st=4)
SAMPLER_CFG = dict(scenes.GOLDEN_CONFIGS["mv_small"], H=17, W=23, rays=None, seed=91)
SAMPLER_STRIDES = (1, 3)
ENCODER_SHAPES = ((2, 288, 512), (3, 37, 53), (1, 135, 240))


def main():
  from test_checkpoint_cpu import _args as checkpoint_args
  from test_encoder_gpu import _input as encoder_input, _model, _sample_index as encoder_sample_index
  ref = mg.import_reference()
  from ibrnet import feature_network as ref_fn
  torch.set_grad_enabled(False)

  # ---- render_rays_mv on a second scene ----
  batch, feat_c, feat_f, frame, t, offs, model, args = scenes.build(MV_CFG)
  mref = mg.reference_model(ref, model, args, False)
  ret = ref.rr.render_rays_mv(frame, t, offs, batch, mref, ref.proj.Projector("cpu"), feat_c, feat_f,
                              MV_CFG["N_samples"], args, inv_uniform=True, N_importance=MV_CFG["N_importance"],
                              det=True, is_train=False)
  fx = {"cfg": MV_CFG, "checksum": mg.checksum(batch, [feat_c, feat_f])}
  for k in ("outputs_coarse_ref", "outputs_fine_ref", "outputs_fine_ref_dy"):
    fx[k] = mg.clean(ret[k])
  torch.save(fx, os.path.join(HERE, "mv_seed77.pt"))

  # ---- ray sampler ----
  batch = scenes.build(SAMPLER_CFG)[0]
  data = scenes.sampler_data(batch, SAMPLER_CFG["H"], SAMPLER_CFG["W"], SAMPLER_CFG["seed"])
  fx = {"cfg": SAMPLER_CFG}
  for stride in SAMPLER_STRIDES:
    fx[stride] = mg.clean(ref.sr.RaySamplerSingleImage(data, "cpu", render_stride=stride).get_all())
    for k, v in fx[stride].items():  # tensors equal at every stride are stored once
      w = fx[SAMPLER_STRIDES[0]][k]
      if torch.is_tensor(v) and v.shape == w.shape and torch.equal(v, w):
        fx[stride][k] = w
  torch.save(fx, os.path.join(HERE, "sampler_17x23.pt"))

  # ---- checkpoint layout ----
  a = checkpoint_args()
  fx = {}
  for key, mod in (("net_fine_st", ref.mlp.DynibarStatic(a, 32, 32)), ("net_fine_dy", ref.mlp.DynibarDynamic(a, 32, 32)),
                   ("motion_mlp_fine", ref.mlp.MotionMLP(num_basis=6))):
    fx[key] = [(name, tuple(v.shape), str(v.dtype)) for name, v in mod.state_dict().items()]
  torch.save(fx, os.path.join(HERE, "checkpoint_layout.pt"))

  # ---- encoder ----
  fx = {}
  for N, H, W in ENCODER_SHAPES:
    m = _model(N * 1000 + H)
    r = ref_fn.ResNet(coarse_out_ch=32, fine_out_ch=32, coarse_only=False)
    r.load_state_dict(m.state_dict(), strict=True)
    x = encoder_input(N, H, W)
    c, f = r.eval()(x)
    e = {"input_sum": float(x.double().sum()), "coarse_shape": tuple(c.shape), "fine_shape": tuple(f.shape)}
    for name, out, seed in (("coarse", c, 1), ("fine", f, 2)):
      e[name] = out.reshape(-1)[encoder_sample_index(out.numel(), seed)].clone()
    fx[(N, H, W)] = e
  torch.save(fx, os.path.join(HERE, "encoder_shapes.pt"))
  for n in ("mv_seed77", "sampler_17x23", "checkpoint_layout", "encoder_shapes"):
    print(n + ".pt", os.path.getsize(os.path.join(HERE, n + ".pt")) // 1024, "KB")


if __name__ == "__main__":
  main()
