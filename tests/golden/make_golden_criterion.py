"""Fixture of the training criteria, from the UNMODIFIED ibrnet/criterion.py (run where the reference sources are):

    python tests/golden/make_golden_criterion.py

  criterion.pt   value and input gradients of Criterion (with and without motion_mask), compute_rgb_loss,
                 compute_temporal_rgb_loss (with and without motion_mask) and compute_flow_loss on the seeded
                 inputs of tests/test_criterion_cpu.py:criterion_inputs

ibrnet/criterion.py imports utils.py, which imports matplotlib for its plotting helpers; the criteria use none of
it, so matplotlib is stubbed in sys.modules (as make_golden.import_reference stubs kornia).  Like the other
fixtures it holds reference OUTPUTS only; the inputs are regenerated from the seed and guarded by a checksum.
"""

import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import make_golden as mg  # noqa: E402


def import_reference_criterion():
  if mg.REF not in sys.path:
    sys.path.insert(0, mg.REF)
  if "matplotlib" not in sys.modules:  # utils.py:4-7 (plotting helpers only)
    mpl = types.ModuleType("matplotlib")
    cm = types.ModuleType("matplotlib.cm")
    backends = types.ModuleType("matplotlib.backends")
    agg = types.ModuleType("matplotlib.backends.backend_agg")
    agg.FigureCanvasAgg = object
    figure = types.ModuleType("matplotlib.figure")
    figure.Figure = object
    mpl.cm, mpl.backends, mpl.figure, backends.backend_agg = cm, backends, figure, agg
    sys.modules.update({"matplotlib": mpl, "matplotlib.cm": cm, "matplotlib.backends": backends,
                        "matplotlib.backends.backend_agg": agg, "matplotlib.figure": figure})
  from ibrnet import criterion  # noqa
  return criterion


def main():
  from test_criterion_cpu import checksum, criterion_inputs, run_criterion_cases
  ref = import_reference_criterion()
  crit = ref.Criterion()
  ns = types.SimpleNamespace(criterion=lambda o, b, motion_mask=None: crit(o, b, motion_mask=motion_mask),
                             compute_rgb_loss=ref.compute_rgb_loss,
                             compute_temporal_rgb_loss=ref.compute_temporal_rgb_loss,
                             compute_flow_loss=ref.compute_flow_loss)
  x = criterion_inputs()
  fx = {"checksum": checksum(x), "cases": run_criterion_cases(ns, x)}
  torch.save(fx, os.path.join(HERE, "criterion.pt"))
  print("wrote criterion.pt:", {k: float(v["value"]) for k, v in fx["cases"].items()})


if __name__ == "__main__":
  main()
