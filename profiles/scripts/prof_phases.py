"""Phase timestamps (clock64) of block 0 of the static per-view kernel (csrc/view_twin3.cu).

    python profiles/scripts/prof_phases.py > gpurun_out/phases.txt
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), 'tests'))
from dynibar_b200 import _lib, synthetic, render_ray as rr

NAMES = ["geom+F1 operand", "gather", "wait F1", "F1 epi", "wait F2", "F2 epi+pool1", "wait F3",
         "F3 epi", "wait F4", "F4 epi", "wait F5", "F5 epi", "wait F6", "F6 epi", "wait F7",
         "F7 epi", "pool2+out"]


def main():
  DEV = "cuda:0"
  rr.set_precision("bf16")
  R, S = 8192, 128
  batch, feat_c, feat_f, frame, t, offs = synthetic.make_scene(rays=R, seed=0)
  model, args = synthetic.make_model(64, 64)
  d = lambda x: synthetic.to_device(x, DEV)
  b, ff = d(batch), d(feat_f)
  m = synthetic.model_to(model, DEV)
  pts, z, s = rr.sample_along_camera_ray(b["ray_o"], b["ray_d"], b["depth_range"], S, True, True)
  fcl = rr.featmaps_channels_last(ff[2])
  run = lambda: rr.net_static_fused(m.net_fine_st, pts, b["ray_o"], b["ray_d"], b["camera"],
                                    b["static_src_rgbs"], b["static_src_cameras"], fcl)
  run(); run()
  torch.cuda.synchronize()
  buf = torch.zeros(2 * 64 + 8 + 480, dtype=torch.int64, device=DEV)
  _lib.lib.dyn_debug_set_view_timestamps(buf.data_ptr())
  run()
  torch.cuda.synchronize()
  _lib.lib.dyn_debug_set_view_timestamps(None)
  allv = buf.cpu()
  iss = allv[128:131].tolist()
  print('issuer: lifetime %d cycles, waiting for A operands %.1f%%, waiting for weight chunks %.1f%%, issuing %.1f%%' % (iss[0], 100.0*iss[1]/iss[0], 100.0*iss[2]/iss[0], 100.0*(iss[0]-iss[1]-iss[2])/iss[0]))
  t = allv[:128].view(2, 64)
  base = int(t[0, 0])
  ch = allv[136:136 + 480].view(120, 4) - base
  print('issuer per chunk (cycles relative to twin0 iter0 start): start, A ready, weights ready, issued | waitA waitW issue')
  for i in range(120):
    a, b, c, d = ch[i].tolist()
    print('  chunk %3d  %8d %8d %8d %8d | %6d %6d %6d' % (i, a, b, c, d, b - a, c - b, d - c))
  print('epilogue timestamps twin0 (relative):', (t[0][:36] - base).tolist())
  print('epilogue timestamps tile1 twin? n/a')
  for tw in range(2):
    ts = t[tw]
    n = int((ts != 0).sum())
    print("twin", tw, "timestamps", n)
    per = 18
    for it in range(n // per):
      seg = ts[it * per:(it + 1) * per]
      d = (seg[1:] - seg[:-1]).tolist()
      tot = int(seg[-1] - seg[0])
      print(" iter", it, "total", tot)
      for nm, x in zip(NAMES, d):
        print("   %-18s %7d  %5.1f%%" % (nm, x, 100.0 * x / tot))
      if (it + 1) * per < n:
        print("   -> next iteration gap", int(ts[(it + 1) * per] - seg[-1]))


if __name__ == "__main__":
  main()
