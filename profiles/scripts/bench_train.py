#!/usr/bin/env python
"""Times the training step of BASELINE config 3 (N_rand = 1024 rays, 64 coarse samples, render_rays_mono with the
cross-time branch, forward + backward + Adam step) through the differentiable fp32 path.  Secondary measurement,
not bench.py's metric.  Usage: python profiles/scripts/bench_train.py [steps] [rays] [bf16|fp32] [encoder]
[--objective standin|dynibar|torch]

--objective: `standin` (default) is the four-term loss bench.py's training-step line uses; `dynibar` is
dynibar_b200.criterion.dynibar_objective, the loss of train.py:300-458 on csrc/objective.cu; `torch` is the same
loss as the reference writes it in torch (tests/objective_oracle.py) on the GPU tensors.  --profile-objective DIR
writes the torch.profiler kernel count of the objective region (forward + backward of the loss alone) there."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import argparse  # noqa: E402

import torch  # noqa: E402

from dynibar_b200 import criterion, render_ray as rr, synthetic  # noqa: E402
from dynibar_b200.projection import Projector  # noqa: E402
from dynibar_b200._lib import lib  # noqa: E402
import objective_oracle  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("steps", nargs="?", type=int, default=5)
ap.add_argument("rays", nargs="?", type=int, default=1024)
ap.add_argument("prec", nargs="?", default="bf16", choices=("bf16", "fp32"))
ap.add_argument("encoder", nargs="?", default="", choices=("", "encoder"))
ap.add_argument("--objective", default="standin", choices=("standin", "dynibar", "torch"))
ap.add_argument("--epoch", type=int, default=0, help="training epoch the objective's schedule is evaluated at")
ap.add_argument("--profile-objective", default=None, metavar="DIR")
cli = ap.parse_args()
steps, rays, prec = cli.steps, cli.rays, cli.prec
with_encoder = cli.encoder == "encoder"  # feature maps = ResNet(source images), trained too
# multi-GPU (torchrun): the N_rand rays are block-partitioned over the ranks (weights replicated), every rank runs
# forward + backward on its share and ONE flat all-reduce sums the parameter gradients (distributed.allreduce_gradients)
world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
dev = torch.device("cuda", local)
torch.cuda.set_device(dev)
if world > 1:
  import torch.distributed as dist
  from dynibar_b200 import distributed as dd
  dist.init_process_group("nccl", device_id=dev)
batch, feat_c, _, frame, t, offs = synthetic.make_scene(H=288, W=512, V_dy=8, V_st=8, num_vv=2, seed=3, rays=rays,
                                                        anchor_offset=2)
if world > 1:
  batch, (lo, hi) = dd.shard_ray_batch(batch, rank, world)
  rays_local = hi - lo
else:
  rays_local = rays
args = synthetic.make_args(1, 1, 0)
model, args = synthetic.make_model(64, 0, args=args, seed=3, mono=True)
model = synthetic.model_to(model, dev)
mods = [model.net_coarse_dy, model.net_coarse_st, model.motion_mlp]
params = []
for m in mods:
  m.requires_grad_(True)
  params += list(m.parameters())
b = synthetic.to_device(batch, dev)
if with_encoder:
  from dynibar_b200 import feature_network
  torch.manual_seed(5)
  enc = feature_network.ResNet().to(dev)
  enc.requires_grad_(True)
  imgs = [b[k][0].permute(0, 3, 1, 2).contiguous() for k in ("src_rgbs", "anchor_src_rgbs", "static_src_rgbs")]
  opt = torch.optim.Adam(params + list(enc.parameters()), lr=1e-4)
else:
  feat = tuple(f.to(dev).requires_grad_(True) for f in feat_c)
  opt = torch.optim.Adam(params + list(feat), lr=1e-4)
torch.manual_seed(11)
target = torch.rand(rays, 3, device=dev)
if world > 1:
  target = target[lo:hi]
b = synthetic.make_supervision(b, n_flow=6, seed=11)  # seeded per-ray supervision for the dynibar / torch objectives
proj = Projector(dev)
group = None
if world > 1 and cli.objective == "dynibar":
  group = dist.group.WORLD


def objective(ret):
  if cli.objective == "dynibar":
    return criterion.dynibar_objective(ret, b, args, cli.epoch, group=group)[0]
  if cli.objective == "torch":
    return objective_oracle.objective(ret, b, args, cli.epoch)[0]
  # Loss terms are a stand-in (bench.py's training-step line)
  loss = ((ret["outputs_coarse_ref"]["rgb"] - target) ** 2).mean()
  loss = loss + ((ret["outputs_coarse_anchor"]["rgb"] - target) ** 2).mean()
  loss = loss + 1e-3 * ret["outputs_coarse_ref"]["render_flows"].abs().mean()
  return loss + 1e-2 * ret["outputs_coarse_anchor"]["sf_seq"].abs().mean()


def step():
  opt.zero_grad(set_to_none=True)
  if with_encoder:  # train.py:264-281: coarse feature maps of the reference / anchor / static source views
    with rr.precision_scope(prec):
      fm = tuple(enc(im)[0] for im in imgs)
  else:
    fm = feat
  ret = rr.render_rays_mono(frame, t, offs, b, model, fm, proj, 64, args, inv_uniform=True, det=False, is_train=True,
                            num_vv=2, precision=prec)
  loss = objective(ret)
  loss.backward()
  if world > 1:  # the dynibar objective normalises with the global sums: its gradients add up, not average
    dd.allreduce_gradients([p for g in opt.param_groups for p in g["params"]], average=cli.objective != "dynibar")
  opt.step()
  return loss


def objective_launches():
  """Kernels of the objective alone (forward + backward of the loss on one step's detached outputs)."""
  fm = tuple(enc(im)[0] for im in imgs) if with_encoder else feat
  with rr.precision_scope(prec):
    ret = rr.render_rays_mono(frame, t, offs, b, model, fm, proj, 64, args, inv_uniform=True, det=False,
                              is_train=True, num_vv=2, precision=prec)
  det = {o: ({k: (v.detach().requires_grad_(v.is_floating_point()) if torch.is_tensor(v) else v)
              for k, v in d.items()} if d is not None else None) for o, d in ret.items()}
  objective(det).backward()  # warm
  torch.cuda.synchronize()
  n0 = lib.dyn_launch_count(0)
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    objective(det).backward()
    torch.cuda.synchronize()
  dyn = lib.dyn_launch_count(0) - n0
  kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
             and not e.name.startswith(("Memset", "Memcpy"))]
  os.makedirs(cli.profile_objective, exist_ok=True)
  names = sorted({e.name for e in kernels})
  with open(os.path.join(cli.profile_objective, "objective_%s.txt" % cli.objective), "w") as f:
    f.write("\n".join(names) + "\n")
  return {"objective_cuda_kernels": len(kernels), "objective_dyn_launches": dyn}


for _ in range(2):
  l0 = step()
torch.cuda.synchronize()
if world > 1:
  dist.barrier()
n0 = lib.dyn_launch_count(0)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(steps):
  l1 = step()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / steps
if world > 1:
  tms = torch.tensor([ms], device=dev)
  dist.all_reduce(tms, op=dist.ReduceOp.MAX)
  ms = float(tms.item())
extra = objective_launches() if cli.profile_objective else {}
if rank == 0:
  print(json.dumps({"objective": cli.objective, "epoch": cli.epoch, **extra, "what": "training step, BASELINE config 3 shape (render_rays_mono is_train=True, fwd + bwd + Adam)",
                  "rays": rays, "n_gpus": world, "samples": 64, "views": "6+2 dynamic, 8 static, 6+2 anchor", "precision": prec, "encoder_in_step": with_encoder,
                  "ms_per_step": ms, "rays_per_s": rays / ms * 1e3, "loss_first": float(l0), "loss_last": float(l1),
                  "kernel_launches_per_step": (lib.dyn_launch_count(0) - n0) / steps,
                  "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30}))
if world > 1:
  dist.destroy_process_group()
