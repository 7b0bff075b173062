"""bench.py contract checks that need no GPU: the reference arm prints exactly ONE JSON line on stdout with the keys the
driver reads, and the committed lines of our arm (profiles/r01_bench_*_final.json, plain runs on B200) carry the
roofline / cpu_baseline / e2e / clocks objects."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def test_reference_arm_prints_one_json_line():
  r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                     capture_output=True, text=True, timeout=900, cwd=ROOT)
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, r.stdout
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and BASE_KEYS <= set(d)
  assert d["unit"] == "samples/s" and d["higher_is_better"] is True and d["value"] > 0
  assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
  assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
  assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.gpu
def test_bench_times_k_steps_and_dumps_the_last_one(tmp_path):
  """--steps K times steps 0 .. K-1 however many blocks --reps splits them into, and --dump-outputs writes the
  [gradient | loss slots] buffer the last of them returned.  Step i reads its own seeded input set and time, so the dump
  tells which step ran last: runs that end on the same step agree, a run one step longer does not."""
  import numpy as np

  def run(out, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "1", "--no-oracle",
                        "--dump-outputs", str(out), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    g, s = np.load(out / "gradient.npy"), np.load(out / "loss_slots.npy")
    assert g.dtype == s.dtype == np.float32 and s.shape == (8, ) and np.isfinite(g).all()
    return json.loads(r.stdout), np.concatenate([g, s]).astype(np.float64)

  def headline(steps, reps):
    d, v = run(tmp_path / f"k{steps}_r{reps}", "--steps", str(steps), "--reps", str(reps), "--no-per-config")
    assert d["steps"] == steps and d["spread"]["reps"] == min(steps, reps) and v.size == d["config"]["params"] + 8
    assert v[-8] == np.float32(d["run"]["loss_last_step"])
    return v

  rel = lambda a, b: np.abs(a - b).max() / np.abs(b).max()
  k3, k3_one_block, k4 = headline(3, 3), headline(3, 1), headline(4, 1)
  assert rel(k3, k3_one_block) < 1e-5   # the same step: equal up to the order of the kernel's float additions
  assert rel(k4, k3_one_block) > 1e-4   # another input set and time
  d, v = run(tmp_path / "only", "--only", "cfg1", "--steps", "2")
  assert v.size == d["entry"]["params"] + 8 and v[-8] == np.float32(d["entry"]["loss_last_step"])


def test_dump_outputs_stays_within_64_mib(tmp_path):
  """bench.dump_outputs on the CPU: a buffer within 64 MiB is written whole, a larger one (cfg 5's gradient alone is
  530 MiB) as the same seeded sample of gradient entries every time, with their indices; all files within 64 MiB."""
  import numpy as np
  import torch
  cap = 64 << 20
  sizes = (1200, cap // 4)   # the second: [gradient | 8 loss slots] just over the cap
  code = ("import sys, types, torch\nsys.path.insert(0, sys.argv[1])\nimport bench\n"
          "for n in map(int, sys.argv[3:]):\n"
          "  out = torch.rand(n + 8, generator=torch.Generator().manual_seed(n))\n"
          "  for run in 'ab':\n"
          "    bench.dump_outputs(f'{sys.argv[2]}/{n}{run}', types.SimpleNamespace(blob_size=n), out)\n")
  r = subprocess.run([sys.executable, "-c", code, ROOT, str(tmp_path), *map(str, sizes)], capture_output=True, text=True,
                     timeout=600)
  assert r.returncode == 0, r.stderr[-2000:]
  for n in sizes:
    out = torch.rand(n + 8, generator=torch.Generator().manual_seed(n)).numpy()
    d = tmp_path / f"{n}a"
    files = {f.name: np.load(f) for f in d.iterdir()}
    assert sum(f.stat().st_size for f in d.iterdir()) <= cap
    assert all(v.dtype in (np.float32, np.float64) for v in files.values())
    assert np.array_equal(files["loss_slots.npy"], out[n:])
    if (n + 8) * 4 <= cap:
      assert set(files) == {"gradient.npy", "loss_slots.npy"} and np.array_equal(files["gradient.npy"], out[:n])
    else:
      idx = files["gradient_index.npy"]
      assert idx.size == files["gradient.npy"].size == 1 << 20 and (np.diff(idx) > 0).all() and 0 <= idx[0] <= idx[-1] < n
      assert np.array_equal(files["gradient.npy"], out[:n][idx.astype(np.int64)])
    for name, v in files.items():
      assert np.array_equal(v, np.load(tmp_path / f"{n}b" / name))


@pytest.mark.parametrize("name", ["r01_bench_n1_final.json", "r01_bench_n2_final.json", "r01_bench_n8_final.json"])
def test_committed_bench_lines_follow_the_contract(name):
  d = json.loads(open(os.path.join(ROOT, "profiles", name)).read())
  assert BASE_KEYS | {"gpu_launches", "clocks", "roofline"} <= set(d)
  assert d["gpu_launches"] == 2 * d["steps"] and d["scaling"] == "weak" and d["vs_baseline"] is None
  rf = d["roofline"]
  assert rf["bound"] in ("hbm", "tensor") and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
  assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
  assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
  if d["n_gpus"] == 1:
    assert d["cpu_baseline"]["kind"] == "port" and 0.5 < min(v["frac"] for v in d["roofline_spline"].values()) < 1.0


@pytest.mark.parametrize("name", ["r02_bench_n1_final.json", "r02_bench_n2_final.json", "r02_bench_n8_final.json"])
def test_committed_round2_bench_lines_follow_the_contract(name):
  """Round 2: one kernel launch per step (reduction, all-reduce in its tail), repetitions with spread, full-size
  parity, the per-config block, the kernel's own timeline; at N > 1 the fused all-reduce checked against NCCL."""
  d = json.loads([l for l in open(os.path.join(ROOT, "profiles", name)) if l.startswith("{")][0])
  assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "spread", "parity", "per_config", "step_timeline",
                      "train_loop"} <= set(d)
  assert d["gpu_launches"] == d["steps"] * d["spread"]["reps"] and d["scaling"] == "weak" and d["vs_baseline"] is None
  assert d["spread"]["min_ms"] <= d["spread"]["median_ms"] <= d["spread"]["max_ms"]
  rf = d["roofline"]
  assert rf["bound"] == "hbm" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
  assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
  assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
  assert set(d["per_config"]) == {"cfg1", "cfg3", "cfg4", "cfg5"}
  tl = d["step_timeline"]
  assert tl["kernel_span"] < d["ms_per_step"] * 1e3 * 1.05 and tl["reduction_tail"] < 20
  for t in d["train_loop"]:
    assert t["wall_over_device"] < 1.1 and t["loss_last"] < t["loss_first"]
  if d["n_gpus"] == 1:
    assert d["parity"]["rows"] == 262144 and d["parity"]["loss_rel"] < 2e-5 and d["parity"]["grad_rel"] < 5e-5
    assert d["cpu_baseline"]["kind"] == "port"
  else:
    assert d["dp_check"]["identical_on_all_ranks"] is True and d["dp_check"]["dp_check_rel_err"] < 2e-6


def test_traffic_json_belongs_to_the_committed_kernel_sources():
  """profiles/traffic.json (ncu-derived constants bench.py reports) is regenerated by tools/make_traffic.py after every
  change under cnf_ot_b200/csrc; a file captured from other sources is ignored by bench.py -- and fails here."""
  sys.path.insert(0, ROOT)
  sys.path.insert(0, os.path.join(ROOT, "tools"))
  import make_traffic
  tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
  assert tj["csrc_sha16"] == make_traffic.fingerprint()
  assert tj["mfc_step_kernel_warp_insts_per_launch"] > 1e7 and tj["mfc_step_kernel_dram_bytes_per_launch"] > 4e6
