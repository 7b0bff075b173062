"""Time per training update on the wide-conditioner engine: the host-driven update() loop of solvers.make_update (a key
split on the host, four cnfot_philox_rows launches, the engine's step, cnfot_adam_update) against the device-resident
cnfot_mfc_update replayed from CUDA graphs (what solvers.main runs on one GPU).

Both loops train their own copy of the same flow; they alternate within one process, `--rounds` rounds, each timing
`--updates` updates after a warm-up (graph capture included there).  A window ends with a device synchronise: wall =
host clock around the window, device = CUDA events around it.  A separate profiled pass counts the device activities
(kernels, memsets, copies) of one update of each loop.

  python tools/time_wide_update.py [--rounds 3] [--out result.json]
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# hidden-64 flows of small dim also fit the fused kernels: every flow here runs on the wide engine
os.environ["CNFOT_ENGINE"] = "wide"

import torch  # noqa: E402
import yaml  # noqa: E402

from cnf_ot_b200 import _lib, applications, ops, random, solvers  # noqa: E402

# the flows of tools/train_wide.py, and one flow of BASELINE config 5's shape (dim 32, 16 layers, 2 x 512) at a batch
# that fits one row chunk
FLOWS = [
  ("ot", dict(dim=2, hidden=64, layers=2, B=4096), 10),
  ("rwpo", dict(dim=2, hidden=64, layers=2, B=2048), 10),
  ("ot", dict(dim=2, hidden=512, layers=2, B=4096), 10),
  ("ot", dict(dim=32, hidden=512, layers=16, B=4096), 2),
]


def config(typ, f):
  cfg = yaml.safe_load(open(os.path.join(ROOT, "cnf_ot_b200", "config", "mfc.yaml")))
  c = copy.deepcopy(cfg)
  c["general"]["type"] = typ
  c["general"]["dim"] = f["dim"]
  c["cnf"]["hidden_size"] = f["hidden"]
  c["cnf"]["flow_num_layers"] = f["layers"]
  c["train"]["batch_size"] = f["B"]
  return c


class HostLoop:
  """solvers.main's make_update loop: one key split per update on the host."""

  def __init__(self, cfg):
    model, loss_fn, _ = solvers.build(cfg)
    dim = cfg["general"]["dim"]
    self.rng = random.PRNGKey(cfg["general"]["seed"])
    model_rng, self.rng = random.split(self.rng)
    self.params = model.init(model_rng, torch.zeros(1, dim), torch.zeros(1))
    self.opt = solvers.AdamState(self.params)
    tr = cfg["train"]
    self.lam, self.B = tr["_lambda"], tr["batch_size"]
    self.update = solvers.make_update(loss_fn, tr["lr"], self.B)

  def warm(self):
    self.run(2)

  def run(self, n):
    for _ in range(n):
      k, self.rng = random.split(self.rng)
      self.update(self.params, k, self.lam, self.opt)


class GraphLoop:
  """solvers.main's device-resident loop: K updates per CUDA graph, replayed."""

  def __init__(self, cfg, K):
    model, loss_fn, _ = solvers.build(cfg)
    dim = cfg["general"]["dim"]
    rng = random.PRNGKey(cfg["general"]["seed"])
    model_rng, rng = random.split(rng)
    self.params = model.init(model_rng, torch.zeros(1, dim), torch.zeros(1))
    sc = applications._step_config(loss_fn)
    tr = cfg["train"]
    B = tr["batch_size"]
    self.K = K
    state = ops.TrainState(model.shape, self.params.blob, 12345, rows_B=B, rows_b=B // 32)
    self.one = lambda: ops.mfc_update(model.shape, sc["problem"], state, self.params.blob, cfg["general"]["t_batch_size"],
                                      tr["_lambda"], B, B // 32, tr["lr"])
    self.graph = None

  def warm(self):
    self.one()   # outside the capture: sets the kernels' shared-memory limits
    self.graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(self.graph):
      for _ in range(self.K):
        self.one()
    self.graph.replay()

  def run(self, n):
    for _ in range(n // self.K):
      self.graph.replay()


def window(loop, n):
  s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  s.record()
  loop.run(n)
  e.record()
  torch.cuda.synchronize()
  return (time.perf_counter() - t0) * 1e3 / n, s.elapsed_time(e) / n


def activities_per_update(loop, n):
  from torch.profiler import ProfilerActivity, profile
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    loop.run(n)
    torch.cuda.synchronize()
  kinds = {}
  for ev in prof.events():
    if ev.device_type == torch.autograd.DeviceType.CUDA:
      name = ev.name.lower()
      kind = "memset" if "memset" in name else ("memcpy" if "memcpy" in name else "kernel")
      kinds[kind] = kinds.get(kind, 0) + 1
  return {k: v / n for k, v in sorted(kinds.items())}


def card():
  try:
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True, timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
  except Exception:
    return torch.cuda.get_device_name()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--rounds", type=int, default=3)
  ap.add_argument("--out", default=None)
  args = ap.parse_args()
  torch.cuda.set_device(0)
  print(f"card: {card()}", flush=True)
  results = []
  for typ, f, K in FLOWS:
    cfg = config(typ, f)
    loops = {"host update()": HostLoop(cfg), "graph mfc_update": GraphLoop(cfg, K)}
    for lp in loops.values():
      lp.warm()
    n = 2 * K
    times = {name: [] for name in loops}
    for _ in range(args.rounds):
      for name, lp in loops.items():
        times[name].append(window(lp, n))
    variant = _lib.last_launch_variant()["plan"]
    row = {"type": typ, **f, "K": K, "updates_per_window": n, "plan": variant}
    for name, lp in loops.items():
      wall = [w for w, _ in times[name]]
      dev = [d for _, d in times[name]]
      row[name] = {"wall_ms": statistics.median(wall), "wall_range": [min(wall), max(wall)],
                   "device_ms": statistics.median(dev), "device_range": [min(dev), max(dev)],
                   "activities_per_update": activities_per_update(lp, K)}
    results.append(row)
    h, g = row["host update()"], row["graph mfc_update"]
    print(f"{typ} dim {f['dim']} L {f['layers']} hidden {f['hidden']} B {f['B']} ({variant}): "
          f"host loop wall {h['wall_ms']:.3f} ms [{h['wall_range'][0]:.3f}, {h['wall_range'][1]:.3f}] device {h['device_ms']:.3f}, "
          f"{h['activities_per_update']}; graph wall {g['wall_ms']:.3f} ms [{g['wall_range'][0]:.3f}, {g['wall_range'][1]:.3f}] "
          f"device {g['device_ms']:.3f}, {g['activities_per_update']}; speed-up (wall) {h['wall_ms'] / g['wall_ms']:.2f}x",
          flush=True)
    del loops
    torch.cuda.empty_cache()
  if args.out:
    with open(args.out, "w") as fh:
      json.dump({"card": card(), "results": results}, fh, indent=1)


if __name__ == "__main__":
  main()
