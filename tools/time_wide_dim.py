"""Time the wide-conditioner engine across flow dimensions: the ot/free train step (cnfot_mfc_step on explicit rows)
and the device-resident update (cnfot_mfc_update: on-chip draws + step + Adam) at dim 32, 64, 128 and 255, for a flow
of 4 layers with 2 x 512 conditioners, at B = 4 096 and 32 768 rows (b = B / 32 kinetic rows, one time per step).

    python tools/time_wide_dim.py [--dims 32,64,128,255] [--batches 4096,32768] [--steps 3] [--rounds 3] [--out FILE]

CUDA events around `--steps` calls after one warm-up call of each shape; `--rounds` rounds, the dims alternated inside
each round, the median round reported.  Each shape's buffers are freed before the next shape is built (dim 255 at
B = 32 768 takes ~80 GB of workspace with the activation stash).  Algorithmic conditioner FLOPs come from the shapes:
a flow pass costs 2 L sum_{d=1}^{D-1} [(d+1) H + (M-1) H^2 + 16 H] FLOPs per row, a train step 3x that (forward, input
adjoints, weight gradients) over its 2 B fit rows and 2 b kinetic rows.  The card's name and power limit are read in
the same run."""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402

from cnf_ot_b200 import _lib, ops  # noqa: E402
from cnf_ot_b200.layout import FlowShape  # noqa: E402

L, M, H, LAM, LR = 4, 2, 512, 5000.0, 1e-4


def step_flops(D, B):
  per_row_pass = 2 * L * sum((d + 1) * H + (M - 1) * H * H + 16 * H for d in range(1, D))
  return 3 * per_row_pass * (2 * B + 2 * (B // 32))


def card():
  name = torch.cuda.get_device_name(0)
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30)
    power = q.stdout.strip() if q.returncode == 0 else "unknown"
  except (OSError, subprocess.SubprocessError):
    power = "unknown"
  return name, power


def free_all():
  ops._workspaces.clear()
  gc.collect()
  torch.cuda.empty_cache()


def time_calls(fn, steps):
  fn()   # warm-up: module loads, shared-memory attributes, workspace growth
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(steps):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / steps


def measure(D, B, steps):
  shape = FlowShape(D, L, M, H, 5)
  b = B // 32
  g = torch.Generator(device="cuda").manual_seed(D)
  W = torch.randn(shape.blob_size, device="cuda", generator=g) * 0.005
  cfg = {"general": {"type": "ot", "dim": D, "dx": 0.01, "dt": 0.01, "t_batch_size": 1}, "ot": {"subtype": "free"}}
  prob = ops.problem_desc(cfg)
  src = torch.randn(B, D, device="cuda", generator=g) - 3.0
  tgt = torch.randn(B, D, device="cuda", generator=g)
  sub = torch.randn(b, D, device="cuda", generator=g)
  out = torch.empty(shape.blob_size + 8, device="cuda")
  ms_step = time_calls(lambda: ops.mfc_step(shape, prob, W, None, sub, src, tgt, [0.37], LAM, B, b, out=out), steps)
  engine = _lib.last_launch_info()["engine"]
  loss = float(out[shape.blob_size])
  del src, tgt, sub, out
  free_all()
  state = ops.TrainState(shape, W, 12345, rows_B=B, rows_b=b)
  ms_update = time_calls(lambda: ops.mfc_update(shape, prob, state, W, 1, LAM, B, b, LR), steps)
  plan = _lib.last_launch_variant()["plan"]
  del state, W
  free_all()
  return {"ms_step": ms_step, "ms_update": ms_update, "engine": engine, "plan": plan, "loss": loss}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--dims", default="32,64,128,255")
  ap.add_argument("--batches", default="4096,32768")
  ap.add_argument("--steps", type=int, default=3)
  ap.add_argument("--rounds", type=int, default=3)
  ap.add_argument("--out", default=None, help="write the results as JSON here")
  a = ap.parse_args()
  if not torch.cuda.is_available():
    sys.exit("time_wide_dim.py needs a CUDA device")
  dims = [int(v) for v in a.dims.split(",")]
  batches = [int(v) for v in a.batches.split(",")]
  name, power = card()
  print(f"card: {name}; power limit, max SM clock: {power}", flush=True)
  runs = {(D, B): [] for D in dims for B in batches}
  for r in range(a.rounds):
    for B in batches:
      order = dims if r % 2 == 0 else dims[::-1]
      for D in order:
        m = measure(D, B, a.steps)
        runs[(D, B)].append(m)
        print(f"round {r} B {B} D {D}: step {m['ms_step']:.2f} ms, update {m['ms_update']:.2f} ms "
              f"(engine {m['engine']}, plan {m['plan']}, loss {m['loss']:.6g})", flush=True)
  rows = []
  for B in batches:
    base = None
    for D in dims:
      ms = statistics.median(m["ms_step"] for m in runs[(D, B)])
      mu = statistics.median(m["ms_update"] for m in runs[(D, B)])
      fl = step_flops(D, B)
      if base is None:
        base = (ms, fl)
      rows.append({"D": D, "B": B, "ms_step": ms, "ms_update": mu, "samples_per_s": B / ms * 1e3,
                   "tflops_step": fl / ms / 1e9, "time_ratio": ms / base[0], "flop_ratio": fl / base[1],
                   "spread_step_ms": [round(m["ms_step"], 3) for m in runs[(D, B)]],
                   "engine": runs[(D, B)][0]["engine"]})
  print(f"\n{name}, power limit / max SM clock {power}; L {L}, M {M}, H {H}, ot/free, b = B/32, one time per step")
  print("| D | B | step ms | update ms | samples/s | conditioner TFLOP/s | time / D=32 | FLOP / D=32 |")
  print("|---|---|---|---|---|---|---|---|")
  for q in rows:
    print(f"| {q['D']} | {q['B']} | {q['ms_step']:.2f} | {q['ms_update']:.2f} | {q['samples_per_s']:.3g} | "
          f"{q['tflops_step']:.1f} | {q['time_ratio']:.2f} | {q['flop_ratio']:.2f} |")
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump({"card": name, "power_limit_max_sm_clock": power, "L": L, "M": M, "H": H, "rows": rows}, f, indent=1)


if __name__ == "__main__":
  main()
