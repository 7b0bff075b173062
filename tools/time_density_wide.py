"""Time the density entry points (cnfot_density_grid / cnfot_density_mc) on the wide-conditioner engine.

  python tools/time_density_wide.py [--rounds R] [--reps K] [--out FILE]

Four calls, each timed with CUDA events over K back-to-back calls after a warm-up call:
  snapshots  utils.plot_density_snapshot: ten 100 x 100 grids on [-6, 6]^2
  grid500    utils.rmse_grid_loss_fn: one 500 x 500 grid with the reference error
  mc1e6      utils.rmse_mc_loss_fn: 10^6 Monte-Carlo samples with the reference error
  evaluate   solvers.evaluate for fp at its default sizes (the two calls above plus host work)
on two flows: dim 2, 2 layers, 2 x 128, 5 bins (wide engine only), and the config/mfc.yaml flow (2 x 16), there with
CNFOT_ENGINE=wide and with the fused kernels, alternated within each round.  Every working set fits in L2.
Prints one JSON line per (flow, engine, call) with the median over the rounds, and the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402

from cnf_ot_b200 import _lib, random, solvers, utils  # noqa: E402
from cnf_ot_b200.flows import FlowModel, ParamTree  # noqa: E402
from cnf_ot_b200.layout import FlowShape  # noqa: E402


def card():
  name = torch.cuda.get_device_name()
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", f"-i={torch.cuda.current_device()}"],
                       capture_output=True, text=True, timeout=30)
    power = q.stdout.strip() or "unknown"
  except (OSError, subprocess.SubprocessError):
    power = "unknown"
  return name, power


def calls(model, P):
  cfg = {"general": {"type": "fp", "dim": 2}, "fp": {"T": 1, "a": 1}}
  key = random.PRNGKey(3)
  return {
    "snapshots": lambda: utils.plot_density_snapshot(model.apply.log_prob, P),
    "grid500": lambda: utils.rmse_grid_loss_fn(model.apply.log_prob, P, 1, 500),
    "mc1e6": lambda: utils.rmse_mc_loss_fn(model, P, 1, key, 1000000),
    "evaluate": lambda: solvers.evaluate(cfg, model, P, key, verbose=False),
  }


def time_call(fn, reps):
  fn()   # warm-up: module loads, workspace allocation
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(reps):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / reps


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--rounds", type=int, default=3)
  ap.add_argument("--reps", type=int, default=5)
  ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
  args = ap.parse_args()
  torch.cuda.set_device(0)
  g = torch.Generator(device="cuda").manual_seed(0)
  # (label, shape, engine setting: "wide" forces the wide engine, None leaves the library's choice)
  runs = [("2x128", FlowShape(2, 2, 2, 128, 5), None), ("mfc.yaml", FlowShape(2, 2, 2, 16, 5), "wide"),
          ("mfc.yaml", FlowShape(2, 2, 2, 16, 5), None)]
  blobs = {}
  for label, shape, _ in runs:
    if label not in blobs:
      blobs[label] = torch.randn(shape.blob_size, device="cuda", generator=g) * 0.02
  times = {}
  engines = {}
  for _ in range(args.rounds):
    for label, shape, force in runs:
      if force:
        os.environ["CNFOT_ENGINE"] = force
      else:
        os.environ.pop("CNFOT_ENGINE", None)
      model = FlowModel(shape, "cuda")
      P = ParamTree(shape, blobs[label])
      for name, fn in calls(model, P).items():
        ms = time_call(fn, args.reps)
        eng = _lib.last_launch_info()["engine"]
        engines[(label, force, name)] = eng
        times.setdefault((label, force, name), []).append(ms)
  os.environ.pop("CNFOT_ENGINE", None)
  name, power = card()
  lines = []
  for (label, force, call), ts in times.items():
    ts = sorted(ts)
    lines.append(json.dumps({"flow": label, "engine": engines[(label, force, call)], "call": call,
                             "ms_median": round(ts[len(ts) // 2], 4), "ms_all": [round(t, 4) for t in ts],
                             "reps": args.reps, "gpu": name, "power_limit": power}))
  print("\n".join(lines))
  if args.out:
    with open(args.out, "w") as f:
      f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
  main()
