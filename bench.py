#!/usr/bin/env python
"""Benchmark of the DynIBaR per-ray IBR hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W              # this repo (CUDA)
  python bench.py --impl reference --gpus N --steps K ...    # CPU reference arm

One "step" = one synthetic 512x288 frame (147 456 rays, the reference's 8192-ray chunks, 64 coarse +
64 fine samples, 8 dynamic + 8 static source views) through `render_rays_mv`.

Multi-GPU (`--scaling strong`, the default and the north_star case): the frame's rays are block-
partitioned over the ranks (dynibar_b200.distributed.shard_bounds); inside the timed region rank 0
broadcasts the source images and feature maps of the frame (as the rank that ran the 2-D encoder would),
every rank renders its block with no further communication, and ONE NCCL gather brings rgb / depth /
mask to rank 0.  `--scaling weak` renders a whole frame on every rank (N frames per step) instead; at
N > 1 the strong line carries the weak measurement as `weak_scaling`.  At N = 1 both are the same job.

The headline, end-to-end and extra lines each time --steps steps (the per-kernel profiling pass at most 2).
Prints ONE JSON line on rank 0.  `--dump-outputs DIR` also writes the frame the last headline step rendered
(rgb / depth / mask, float32 .npy): the inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""

import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

KERNEL_CLASSES = ["view_static", "view_dynamic", "motion", "point1", "point2", "rgbhead", "attention",
                  "gather"]
# DRAM bytes per (point, view) row of the static per-view kernel from the committed ncu capture
# (dram__bytes_read.sum + dram__bytes_write.sum per launch / rows); see profiles/
NCU_DRAM_BYTES_PER_ROW = {"view_static": 298.0}  # profiles/r02_view_twin_ncu.md (156.2 MB / 524 288 rows)

WORKLOAD = dict(H=288, W=512, V_dy=8, V_st=8, N_samples=64, N_importance=64, chunk=8192, seed=0)
METRIC = "rays/sec (64+64 samples x 8 src views)"


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=3)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
  ap.add_argument("--rays", type=int, default=147456, help="rays of the frame (147456 = 512x288)")
  ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"])
  ap.add_argument("--ref-rays", type=int, default=512, help="rays per step of the CPU reference arm (one 512-ray chunk)")
  ap.add_argument("--cpu-rays", type=int, default=512, help="rays per timed chunk of the in-line cpu_baseline")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-extras", action="store_true", help="skip the kernel-timing pass, the 7+11-view line and weak_scaling")
  ap.add_argument("--chunk", type=int, default=WORKLOAD["chunk"],
                  help="rays per render_rays_mv call (the reference's chunk_size knob: 'decrease if running out "
                       "of memory', config.py:168; results do not depend on it)")
  ap.add_argument("--view-kernel", default="default", choices=["default", "twin", "quad", "pipe"],
                  help="per-view stage kernel: library default, twin-warp, quad schedule, or sub-round pipelined twin")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="after the timed steps, write the frame the last headline step rendered as DIR/{rgb,depth,mask}.npy")
  a = ap.parse_args()
  if a.steps < 1:
    ap.error("--steps must be at least 1")
  return a


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(path, px, cap_bytes=DUMP_CAP_BYTES):
  """Writes one rendered frame, [rays, 5] = the rgb / depth / mask of render_rays_mv's outputs_fine_ref, as float32
  DIR/rgb.npy [N, 3], depth.npy [N], mask.npy [N].  A frame above `cap_bytes` is cut to a fixed seeded sample of
  rays (in ray order), so that two builds run with the same arguments write the same rays."""
  import numpy as np
  px = px.detach().float().cpu()
  keep = cap_bytes // (px.shape[1] * 4)
  if px.shape[0] > keep:
    idx = torch.randperm(px.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
    px = px[idx]
  os.makedirs(path, exist_ok=True)
  for name, v in (("rgb", px[:, 0:3]), ("depth", px[:, 3]), ("mask", px[:, 4])):
    np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(v.numpy(), dtype=np.float32))


def peaks():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(p):
    d = json.load(open(p))
    return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                source="measured (MEASURED_PEAKS.json)")
  return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
  """Samples SM clock + throttle reasons of one GPU every 200 ms via NVML."""

  REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
             0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
    self._halt = threading.Event()
    self.ok = False
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
      self.ok = True
    except Exception as e:  # NVML missing: report that instead of clocks
      self.err = repr(e)

  def run(self):
    if not self.ok:
      return
    while not self._halt.is_set():
      try:
        self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
        r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, name in self.REASONS.items():
          if r & bit:
            self.reasons.add(name)
      except Exception:
        pass
      self._halt.wait(0.2)

  def finish(self):
    self._halt.set()
    if self.is_alive():
      self.join()
    if not self.ok or not self.samples:
      return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
    s = sorted(self.samples)
    return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
            "samples": len(s)}


def build_scene(rays, V_dy=None, V_st=None):
  from dynibar_b200 import synthetic
  w = WORKLOAD
  batch, feat_c, feat_f, frame, t, offs = synthetic.make_scene(
      H=w["H"], W=w["W"], V_dy=V_dy or w["V_dy"], V_st=V_st or w["V_st"], seed=w["seed"], rays=rays)
  model, args = synthetic.make_model(w["N_samples"], w["N_importance"], seed=w["seed"])
  return batch, feat_c, feat_f, frame, t, offs, model, args


def cpu_threads():
  """Threads of the CPU arm: torch's intra-op pool stops scaling on these small GEMMs well before all
  cores of the 100+-core GPU hosts (where it collapses to ~2 rays/s), so the arm uses min(cores, 32)
  and reports that number as `cores`."""
  return min(os.cpu_count() or 1, 32)


def make_cpu_runner():
  """The reference's CPU implementation of the path on the same synthetic frame: the UNMODIFIED reference
  (oracle/_ref, byte-compiled from /root/reference by oracle/build_ref.py) when it has been built,
  else the oracle port (oracle/dynibar_oracle.py).  Returns (kind, fn(n_rays) -> None)."""
  torch.set_num_threads(cpu_threads())
  w = WORKLOAD
  full = w["H"] * w["W"]
  batch, feat_c, feat_f, frame, t, offs, model, args = build_scene(None)
  g = torch.Generator().manual_seed(1)
  perm = torch.randperm(full, generator=g)
  state = {"pos": 0}

  def chunk(n):  # consecutive blocks of a seeded permutation of the frame's pixels
    idx = perm[state["pos"]:state["pos"] + n]
    state["pos"] = (state["pos"] + n) % (full - n)
    cb = dict(batch)
    for k in ("ray_o", "ray_d", "uv_grid"):
      cb[k] = batch[k][idx]
    return cb

  from oracle import build_ref
  if build_ref.available():
    ref = build_ref.load()
    mref = build_ref.reference_model(ref, model, args)
    P = ref.proj.Projector("cpu")

    def run(n):
      with torch.no_grad():
        ref.rr.render_rays_mv(frame, t, offs, chunk(n), mref, P, feat_c, feat_f, w["N_samples"], args,
                              inv_uniform=True, N_importance=w["N_importance"], det=True, is_train=False)
    return "reference", run

  from oracle import dynibar_oracle as orc

  def run(n):
    with torch.no_grad():
      orc.render_rays_mv(frame, t, offs, chunk(n), model, None, feat_c, feat_f, w["N_samples"], args,
                         inv_uniform=True, N_importance=w["N_importance"], det=True, is_train=False)
  return "port", run


def train_step_line(dev, precision, rays=1024, steps=3):
  """Secondary line: BASELINE configs[2] -- one training step of N_rand = 1024 rays x 64 samples through the
  differentiable render_rays_mono (cross-time branch included), 2-D encoder forward + backward over the 24 source
  images, Adam step; synthetic 512x288 scene.  Loss terms are a stand-in (two photometric + flow + scene-flow)."""
  from dynibar_b200 import feature_network, render_ray as rr, synthetic
  from dynibar_b200.projection import Projector
  batch, _, _, frame, t, offs = synthetic.make_scene(H=288, W=512, V_dy=8, V_st=8, num_vv=2, seed=3, rays=rays,
                                                     anchor_offset=2)
  args = synthetic.make_args(1, 1, 0)
  model, args = synthetic.make_model(64, 0, args=args, seed=3, mono=True)
  model = synthetic.model_to(model, dev)
  params = []
  for m in (model.net_coarse_dy, model.net_coarse_st, model.motion_mlp):
    m.requires_grad_(True)
    params += list(m.parameters())
  torch.manual_seed(5)
  enc = feature_network.ResNet().to(dev).requires_grad_(True)
  b = synthetic.to_device(batch, dev)
  imgs = [b[k][0].permute(0, 3, 1, 2).contiguous() for k in ("src_rgbs", "anchor_src_rgbs", "static_src_rgbs")]
  opt = torch.optim.Adam(params + list(enc.parameters()), lr=1e-4)
  target = torch.rand(rays, 3, device=dev)
  proj = Projector(dev)

  def step():
    opt.zero_grad(set_to_none=True)
    with rr.precision_scope(precision):
      fm = tuple(enc(im)[0] for im in imgs)  # train.py:264-281
      ret = rr.render_rays_mono(frame, t, offs, b, model, fm, proj, 64, args, inv_uniform=True, det=False,
                                is_train=True, num_vv=2)
    loss = ((ret["outputs_coarse_ref"]["rgb"] - target) ** 2).mean()
    loss = loss + ((ret["outputs_coarse_anchor"]["rgb"] - target) ** 2).mean()
    loss = loss + 1e-3 * ret["outputs_coarse_ref"]["render_flows"].abs().mean()
    loss = loss + 1e-2 * ret["outputs_coarse_anchor"]["sf_seq"].abs().mean()
    loss.backward()
    opt.step()
    return loss

  for _ in range(2):
    l0 = step()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(steps):
    l1 = step()
  e1.record()
  torch.cuda.synchronize()
  ms = e0.elapsed_time(e1) / steps
  return {"what": "BASELINE configs[2] shape: training step (encoder + render_rays_mono is_train=True, forward + "
                  "backward + Adam), N_rand %d, 64 samples, 6+2 / 8 / 6+2 views" % rays,
          "precision": precision, "ms_per_step": ms, "value": rays / ms * 1e3, "unit": "rays/s",
          "loss_first": float(l0), "loss_last": float(l1)}


def main():
  a = parse()
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  w = dict(WORKLOAD, chunk=a.chunk)
  config = {"workload": "BASELINE configs[1] shape: synthetic 512x288 frame, 64 coarse + 64 fine "
                        "samples (fine pass evaluates 128), 8 dynamic + 8 static source views, "
                        "render_rays_mv, det=True, inv_uniform=True, chunk %d" % a.chunk,
            "rays_per_frame": a.rays, "precision": a.precision,
            "l2": "per-step working set (source maps 66 MB + GBs of per-chunk intermediates) exceeds the "
                  "126 MB L2; plus an explicit 256 MB flush between steps"}

  if a.impl == "reference":
    if rank != 0:
      return 0
    kind, run = make_cpu_runner()
    for _ in range(max(1, min(a.warmup, 2))):  # warm-up on a quarter chunk: page-in, thread pool, allocator
      run(max(64, a.ref_rays // 4))
    t0 = time.perf_counter()
    for _ in range(a.steps):
      run(a.ref_rays)
    sec = (time.perf_counter() - t0) / a.steps
    val = a.ref_rays / sec
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": a.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(config, rays_per_step=a.ref_rays,
                           note="CPU arm: the unmodified reference render_rays_mv (oracle/_ref) when kind is "
                                "'reference', else the oracle port; each step is one 512-ray chunk of the same "
                                "frame (a full frame would take > 30 min); rays/s extrapolates linearly"),
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cpu_threads(), "kind": kind,
                             "sample": "%d steps x %d rays of the same frame" % (a.steps, a.ref_rays)},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0

  import torch.distributed as dist
  from dynibar_b200 import _lib, distributed as dd, flops, render_ray as rr, synthetic
  from dynibar_b200.projection import Projector
  dev = torch.device("cuda", local)
  torch.cuda.set_device(dev)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  rr.set_precision(a.precision)
  _lib.lib.dyn_debug_set_view_kernel({"default": -1, "twin": 0, "quad": 1, "pipe": 2}[a.view_kernel])
  pin = lambda x: x.pin_memory() if torch.is_tensor(x) else x
  P = Projector(dev)
  SRC_KEYS = ("src_rgbs", "static_src_rgbs")

  class Frame(object):
    """Pinned host inputs of one frame + their device copies for one (mode, view-count) setting."""

    def __init__(self, mode, V_dy=None, V_st=None):
      self.mode = mode
      full = w["H"] * w["W"]
      batch, feat_c, feat_f, self.frame, self.t, self.offs, model, self.args = build_scene(
          None if a.rays >= full else a.rays, V_dy, V_st)
      n_all = a.rays
      for k in ("ray_o", "ray_d", "uv_grid"):
        reps = (n_all + batch[k].shape[0] - 1) // batch[k].shape[0]
        batch[k] = batch[k].repeat(reps, 1)[:n_all].contiguous()
      # strong: this rank's block of the frame; weak: the whole frame on every rank
      self.lo, self.hi = dd.shard_bounds(n_all, rank, world) if mode == "strong" else (0, n_all)
      self.n_local, self.n_total = self.hi - self.lo, (n_all if mode == "strong" else n_all * world)
      host = dict(batch)
      for k in ("ray_o", "ray_d", "uv_grid"):
        host[k] = batch[k][self.lo:self.hi].contiguous()
      self.host = {k: pin(v) for k, v in host.items()}
      self.host_fc = tuple(pin(x) if x is not None else None for x in feat_c)
      self.host_ff = tuple(pin(x) if x is not None else None for x in feat_f)
      self.model = synthetic.model_to(model, dev)
      self.b_dev = synthetic.to_device(self.host, dev)
      self.fc_dev = synthetic.to_device(self.host_fc, dev)
      self.ff_dev = synthetic.to_device(self.host_ff, dev)
      self.out_host = torch.empty(self.n_local, 5, pin_memory=True)

    def sources(self, b, fc, ff):
      return [b[k] for k in SRC_KEYS] + [x for x in fc + ff if x is not None]

    def render(self, b, fc, ff):
      rr.new_frame()  # every step is a new frame: its source views are packed again (once per frame)
      if self.mode == "strong" and world > 1:
        # once per frame: the rank that produced the source views (2-D encoder) hands them to the others
        dd.broadcast_frame_inputs(self.sources(b, fc, ff), src=0)
      outs = []
      for i in range(0, self.n_local, w["chunk"]):
        cb = dict(b)
        for k in ("ray_o", "ray_d", "uv_grid"):
          cb[k] = b[k][i:i + w["chunk"]]
        r = rr.render_rays_mv(self.frame, self.t, self.offs, cb, self.model, P, fc, ff, w["N_samples"],
                              self.args, inv_uniform=True, N_importance=w["N_importance"], det=True,
                              is_train=False)["outputs_fine_ref"]
        outs.append(torch.cat([r["rgb"], r["depth"][:, None], r["mask"][:, None].float()], 1))
      px = torch.cat(outs, 0)
      if world > 1:  # the path's one exchange step: rendered pixels -> rank 0 over NVLink
        if self.mode == "strong":
          dd.gather_pixels(px, self.n_total)
        else:
          dd.gather_pixels(px, px.shape[0] * world)
      return px

    def step_resident(self):
      flush.zero_()
      return self.render(self.b_dev, self.fc_dev, self.ff_dev)

    def step_e2e(self):
      flush.zero_()
      up = lambda x: x.to(dev, non_blocking=True) if torch.is_tensor(x) else x
      src_here = self.mode == "weak" or world == 1 or rank == 0  # strong: sources enter through rank 0
      b = {}
      for k, v in self.host.items():
        if k in SRC_KEYS and not src_here:
          b[k] = torch.empty(v.shape, device=dev)
        else:
          b[k] = up(v)
      fm = lambda tup: tuple((up(x) if src_here else torch.empty(x.shape, device=dev)) if x is not None else None
                             for x in tup)
      px = self.render(b, fm(self.host_fc), fm(self.host_ff))
      self.out_host.copy_(px, non_blocking=True)
      return px

    def h2d_bytes(self):
      n = sum(v.numel() * v.element_size() for k, v in self.host.items()
              if torch.is_tensor(v) and (k not in SRC_KEYS or self.mode == "weak" or world == 1 or rank == 0))
      if self.mode == "weak" or world == 1 or rank == 0:
        n += sum(x.numel() * x.element_size() for x in self.host_fc + self.host_ff if x is not None)
      return n

  def timed(fn, steps):
    """(ms of `steps` calls of fn, what the last call returned)"""
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
      out = fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
      dist.barrier()
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return ms.item(), out

  flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
  fr = Frame(a.scaling)
  for _ in range(max(a.warmup, 3)):
    fr.step_resident()
  torch.cuda.synchronize()

  # ---- headline: inputs resident in HBM, no profiling hooks ----
  sampler = ClockSampler(local)
  sampler.start()
  _lib.lib.dyn_launch_count(1)
  ms, px_last = timed(fr.step_resident, a.steps)
  launches = int(_lib.lib.dyn_launch_count(0))
  clocks = sampler.finish()
  # ---- end to end: pinned host buffers in, pinned host pixels out, every step ----
  fr.step_e2e()
  ms_e2e, _ = timed(fr.step_e2e, a.steps)
  h2d = torch.tensor([float(fr.h2d_bytes())], device=dev)
  d2h = torch.tensor([float(fr.out_host.numel() * fr.out_host.element_size())], device=dev)
  if world > 1:
    dist.all_reduce(h2d)
    dist.all_reduce(d2h)

  # ---- separate pass: per-kernel device time (CUDA events around every launch of the big kernels) ----
  kernel_ms, prof_steps = {}, 0
  if not a.no_extras:
    prof_steps = min(a.steps, 2)
    _lib.lib.dyn_profile_enable(1)
    ms_prof, _ = timed(fr.step_resident, prof_steps)
    for cls, name in enumerate(KERNEL_CLASSES):
      tot, n = ctypes.c_float(), ctypes.c_int()
      _lib.check(_lib.lib.dyn_profile_read(cls, ctypes.byref(tot), ctypes.byref(n)))
      if n.value:
        kernel_ms[name] = (tot.value, n.value)
    _lib.lib.dyn_profile_enable(0)

  extras = {}
  if not a.no_extras and world > 1 and a.scaling == "strong":
    fw = Frame("weak")
    for _ in range(2):
      fw.step_resident()
    ms_w, _ = timed(fw.step_resident, a.steps)
    extras["weak_scaling"] = {"value": a.rays * world * a.steps / (ms_w / 1e3), "unit": "rays/s",
                              "ms_per_step": ms_w / a.steps, "note": "every rank renders a whole frame"}
    del fw
  if not a.no_extras and world == 1:
    # the view counts eval_nvidia.py really uses (7 dynamic + 11 static, eval_nvidia.py:92-119): 11 static
    # views occupy 16 view slots per point in the per-view kernel
    fe = Frame(a.scaling, 7, 11)
    for _ in range(2):
      fe.step_resident()
    ms_e, _ = timed(fe.step_resident, a.steps)
    fpr_e = flops.flop_per_ray(w["N_samples"], w["N_samples"] + w["N_importance"], 7, 11)
    extras["eval_shape"] = {"views": "7 dynamic + 11 static", "value": a.rays * a.steps / (ms_e / 1e3),
                            "unit": "rays/s", "ms_per_step": ms_e / a.steps, "flop_per_ray": fpr_e,
                            "tflops": a.rays * a.steps / (ms_e / 1e3) * fpr_e / 1e12}
    del fe

  if not a.no_extras and world == 1:
    extras["train_step"] = train_step_line(dev, a.precision, steps=a.steps)

  if a.dump_outputs:
    if world > 1 and a.scaling == "strong":  # rank 0's block -> the whole frame on rank 0
      px_last = dd.gather_pixels(px_last, fr.n_total)
    if rank == 0:
      dump_outputs(a.dump_outputs, px_last)

  total_rays = fr.n_total * a.steps
  value = total_rays / (ms / 1e3)
  e2e_val = total_rays / (ms_e2e / 1e3)

  if rank == 0:
    pk = peaks()
    S_c, S_f = w["N_samples"], w["N_samples"] + w["N_importance"]
    fpr = flops.flop_per_ray(S_c, S_f, w["V_dy"], w["V_st"])
    achieved = value / world * fpr / 1e12  # per GPU
    # per-kernel roofline, from the profiling pass on rank 0 (rank 0 renders fr.n_local rays per step)
    S_tot = S_c + S_f
    n_loc = fr.n_local
    mv_d, mv_s = flops.mac_per_point_view("dynamic"), flops.mac_per_point_view("static")
    mac_pt_head = lambda kind, S: flops.mac_per_point(kind, S)
    # algorithmic MACs per step of each kernel class (reference layer widths, dynibar_b200/flops.py);
    # `essential` drops what a kernel hoists out of the per-(point, view) loop: the dynamic net's
    # ray_dir_fc (depends on the frame time only) and the static net's ref_feature_fc (per ray)
    geo = 257 * 256 + 256 * 128
    qkv = 3 * 128 * 128
    macs = {
        "view_static": n_loc * S_tot * w["V_st"] * (mv_s - (261 * 128 + 128 * 64 + 64)),
        "view_dynamic": n_loc * S_tot * w["V_dy"] * mv_d,
        "rgbhead": n_loc * S_tot * w["V_st"] * (261 * 128 + 128 * 64 + 64),
        "motion": n_loc * S_tot * flops.mac_per_point("motion", 0),
        "point1": 2 * n_loc * S_tot * (geo + qkv),
        "attention": 2 * n_loc * (S_c * 2 * S_c * 128 + S_f * 2 * S_f * 128),
        "point2": n_loc * S_tot * ((128 * 128 + 128 * 128 + 128) +  # static: fc, out_geometry_fc
                                   (128 * 128 + (161 * 256 + 256 * 128) + 128 * 128 + 128 + 155 * 128 + 128 * 64 + 192)),
    }
    essential = {"view_static": n_loc * S_tot * w["V_st"] * (mv_s - (261 * 128 + 128 * 64 + 64) - 66 * 35),
                 "view_dynamic": n_loc * S_tot * w["V_dy"] * (mv_d - (21 * 256 + 256 * 35))}
    # rgb_fc.0's per-point part (128 x 128 of its 261 input columns) runs in point2, the rest in rgbhead
    kernels = {}
    for name, (tot_ms, n) in kernel_ms.items():
      k = {"ms_per_step": tot_ms / prof_steps, "launches_per_step": n / prof_steps,
           "share_of_step": tot_ms / ms_prof}
      if name in macs:
        k["tflops"] = macs[name] * prof_steps * 2 / (tot_ms / 1e3) / 1e12
        k["frac_of_peak"] = k["tflops"] / pk["tf_sustained"]
      if name in essential:
        k["tflops_essential"] = essential[name] * prof_steps * 2 / (tot_ms / 1e3) / 1e12
      kernels[name] = k
    dom = max((n for n in kernels if n in macs), key=lambda n: kernels[n]["ms_per_step"], default=None)
    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": a.steps,
        "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": a.scaling, "vs_baseline": None, "dtype": "f32" if a.precision == "fp32" else "bf16",
        "data": "synthetic",
        "config": dict(config, parallelism=("1 GPU" if world == 1 else
                                             ("rays of ONE frame split over %d GPUs; source maps broadcast from rank 0 "
                                              "and pixels gathered to rank 0 inside the timed region" % world
                                              if a.scaling == "strong" else "%d frames, one per GPU" % world)),
                       view_kernel=a.view_kernel),
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": e2e_val, "unit": "rays/s", "h2d_bytes_per_step": int(h2d.item()),
                "d2h_bytes_per_step": int(d2h.item()), "ms_per_step": ms_e2e / a.steps},
        "roofline_step": {"bound": "tensor", "achieved": achieved, "peak": pk["tf_sustained"],
                          "unit": "TFLOP/s", "frac": achieved / pk["tf_sustained"],
                          "flop_per_ray": fpr, "flop_per_ray_essential": fpr - 2 * (S_tot * (
                              w["V_dy"] * (21 * 256 + 256 * 35) + w["V_st"] * 66 * 35)),
                          "peak_source": pk["source"] + ", sustained bf16",
                          "scope": "whole step (all kernels of render_rays_mv), per GPU"},
        "kernels": kernels,
        "kernels_how": "separate pass of %d step(s) after the headline run with dyn_profile_enable(1): CUDA events "
                       "recorded by the library on the launching stream around every launch (rank 0)" % prof_steps,
    }
    line.update(extras)
    if dom is not None:
      kd = kernels[dom]
      rows_step = {"view_static": n_loc * S_tot * w["V_st"]}.get(dom)
      line["roofline"] = {
          "kernel": dom, "bound": "tensor", "achieved": kd["tflops"], "peak": pk["tf_sustained"],
          "unit": "TFLOP/s", "frac": kd["tflops"] / pk["tf_sustained"],
          "achieved_essential": kd.get("tflops_essential"),
          "traffic": (NCU_DRAM_BYTES_PER_ROW[dom] * rows_step / kd["launches_per_step"]
                      if dom in NCU_DRAM_BYTES_PER_ROW and rows_step else None),
          "algorithmic_flop_per_launch": macs[dom] * 2 / kd["launches_per_step"],
          "avg_launch_ms": kd["ms_per_step"] / kd["launches_per_step"],
          "peak_source": pk["source"] + ", sustained bf16 (kernel timed inside a long step)",
          "how": "CUDA events recorded by the library on the launching stream around every launch of "
                 "this kernel (dyn_profile_*), in a separate pass right after the timed region"}
    if world == 1 and not a.no_cpu_baseline:
      kind, run = make_cpu_runner()
      run(128)  # warm-up
      t0 = time.perf_counter()
      run(a.cpu_rays)
      run(a.cpu_rays)
      csec = time.perf_counter() - t0
      line["cpu_baseline"] = {"value": 2 * a.cpu_rays / csec, "unit": "rays/s", "cores": cpu_threads(), "kind": kind,
                              "sample": "2 timed chunks of %d rays of the same frame after a 128-ray warm-up "
                                        "(%.1f s); a full frame extrapolates linearly" % (a.cpu_rays, csec)}
    print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()
  return 0


if __name__ == "__main__":
  sys.exit(main())
