#!/usr/bin/env python
"""Benchmark of the cnf_ot flow train step (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--reps R] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one evaluation of the configured MFC loss and its parameter gradient
(all flow passes forward + inverse + log-det + loss terms + backward; optimiser
excluded, SURVEY.md §8d) over one synthetic batch.  Headline workload = BASELINE.json
configs[1]: mfc.yaml type=ot subtype=obstacle, 2-D, RQS flow (2 layers, 2x16
conditioner, 5 bins), batch 2^18 per GPU (weak scaling), lambda=5000, dt=0.01.

  value       samples/s with the batch already resident in HBM (CUDA events, max over ranks;
              K timed steps split into --reps blocks, median of the blocks, min / max in `spread`)
  --dump-outputs DIR : [gradient | loss slots] of the last timed step (headline workload, or the --only
              config) as DIR/gradient.npy and DIR/loss_slots.npy (float32); seeded inputs, so two builds
              compare output for output.  At most 64 MiB: a larger gradient is written as a fixed, seeded
              sample of 2^20 entries, their indices in DIR/gradient_index.npy
  e2e         the same through the C-ABI call with HOST (pinned) buffers: H2D of the inputs
              and the weights, the step, D2H of [gradient | loss] inside the timed region
  parity      the SAME parameter blob and the SAME 2^18-row input set evaluated by the CPU
              oracle (oracle/, torch f64): relative loss / gradient error of the timed path
  dp_check    N > 1: the fused step + all-reduce (cnfot_mfc_step_dp) against step + NCCL
              all-reduce on the same inputs, and whether every rank holds identical bytes
  per_config  the other BASELINE configs (cfg 1 B=4096; cfg 3 rwpo/double_well 2^20; cfg 4
              fp/nongradient d=10, 2^22 rows over the GPUs; cfg 5 d=32 16x(2x512), reduced
              rows), each with ms/step, samples/s, a roofline object and a small-batch
              oracle check
  --impl reference : the CPU restatement of the reference step (oracle/, torch f64,
              all host threads) on a bounded sample of the same workload.
"""
import argparse
import hashlib
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
  if _p not in sys.path:
    sys.path.insert(0, _p)

import torch  # noqa: E402

METRIC = "flow train-step samples/s (fwd+inv+logdet+loss+grad)"
UNIT = "samples/s"
B_PER_GPU = 1 << 18
SIGMA = 0.3  # parameter perturbation (BASELINE.md §2)


# stdout carries exactly ONE line (the JSON): everything a library writes to file descriptor 1 (NCCL prints its
# version banner there) is sent to stderr, the JSON goes to a private copy of the original stdout
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
  _JSON_OUT.write(json.dumps(line) + "\n")
  _JSON_OUT.flush()


def log(msg):
  print(f"[bench] {msg}", file=sys.stderr, flush=True)


# ---------------------------------------------------------------- workloads (BASELINE.json configs)
def mfc_cfg(typ, sub, dim, batch, H=16, L=2, M=2, K=5, lam=5000.0):
  """mfc.yaml-shaped dict (config/mfc.yaml:6-40) of one BASELINE config."""
  cfg = {
    "general": {"type": typ, "dim": dim, "dx": 0.01, "dt": 0.01, "t_batch_size": 1, "seed": 42},
    "ot": {"subtype": "obstacle"},
    "rwpo": {"T": 1, "beta": 1, "a": 1, "pot_type": "double_well"},
    "fp": {"T": 1, "a": 1, "sigma": 0.5, "velocity_field_type": "nongradient"},
    "cnf": {"flow_num_layers": L, "mlp_num_layers": M, "hidden_size": H, "num_bins": K},
    "train": {"epochs": 1, "lr": 1e-3, "_lambda": lam, "batch_size": batch, "eval_frequency": 100},
  }
  cfg[typ][{"ot": "subtype", "rwpo": "pot_type", "fp": "velocity_field_type"}[typ]] = sub
  return cfg


# name -> (BASELINE label, type, subtype, dim, (H, L, M, K), rows rule, param sigma)
#   rows rule: ("weak", rows per GPU) or ("strong", global rows shared by the GPUs)
WORKLOADS = {
  "cfg1": ("mfc.yaml type=ot subtype=free, 2-D Gaussian->Gaussian, batch 4096 (BASELINE configs[0])",
           "ot", "free", 2, (16, 2, 2, 5), ("strong", 4096), 0.3),
  "cfg2": ("mfc.yaml type=ot subtype=obstacle (BASELINE configs[1])",
           "ot", "obstacle", 2, (16, 2, 2, 5), ("weak", B_PER_GPU), 0.3),
  "cfg3": ("mfc.yaml type=rwpo pot_type=double_well T=1 beta=1 a=1, batch 2^20 per GPU (BASELINE configs[2])",
           "rwpo", "double_well", 2, (16, 2, 2, 5), ("weak", 1 << 20), 0.3),
  "cfg4": ("mfc.yaml type=fp velocity_field_type=nongradient sigma=0.5, d=10, batch 2^22 over the GPUs (BASELINE configs[3])",
           "fp", "nongradient", 10, (16, 2, 2, 5), ("strong", 1 << 22), 0.05),
  "cfg5": ("synthetic scale-out, ot/free structure, d=32, 16 layers, conditioner 2x512 (BASELINE configs[4], reduced rows)",
           "ot", "free", 32, (512, 16, 2, 5), ("weak", 1 << 15), 0.0),
}


def mlp_flops_per_row_eval(D, L, M, H, Pp=16):
  """2 L sum_{d=1}^{D-1} [(d+1) H + (M-1) H^2 + H P] (SURVEY.md §8)."""
  return 2 * L * sum((d + 1) * H + (M - 1) * H * H + H * Pp for d in range(1, D))


def flow_evals_per_step(typ, sub, D, B, b):
  """Rows pushed through the flow per step (SURVEY.md §8 table)."""
  if typ == "ot":
    return 2 * B + (3 if sub == "obstacle" else 2) * b
  if typ == "rwpo":
    return 2 * B + (3 + 2 * D) * b
  return B + (3 + 2 * D) * b


def config_block(n_gpus):
  """`config` of the JSON line: identical in both arms (our arm's run details go to `run`)."""
  return {
    "workload": WORKLOADS["cfg2"][0],
    "dim": 2, "flow_num_layers": 2, "mlp": "2x16", "num_bins": 5, "params": 1200,
    "batch_per_gpu": B_PER_GPU, "global_batch": B_PER_GPU * n_gpus, "sub_batch": "batch//32",
    "t_batch_size": 1, "lambda": 5000.0, "param_sigma": SIGMA,
    "rows_through_flow_per_step": "2B log-prob dir + 3(B/32) sample dir",
    "parallelism": f"dp{n_gpus} (rows sharded, one all-reduce of [grad|loss])",
    "l2_policy": "rotating input sets, > 2x L2 in aggregate (every step streams its batch from HBM)",
  }


# ---------------------------------------------------------------- clocks (NVML, in-process)
class ClockSampler:
  def __init__(self, index):
    self.samples, self.reasons, self.max_mhz = [], set(), None
    self._stop = threading.Event()
    self._t = None
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
    except Exception:  # no NVML: report nulls
      self.nv = None

  def _loop(self):
    nv = self.nv
    names = {
      getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
      getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
      getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
      getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
    }
    while not self._stop.is_set():
      try:
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for bit, name in names.items():
          if r & bit:
            self.reasons.add(name)
      except Exception:
        pass
      time.sleep(0.002)

  def __enter__(self):
    if self.nv:
      self._t = threading.Thread(target=self._loop, daemon=True)
      self._t.start()
    return self

  def __exit__(self, *a):
    self._stop.set()
    if self._t:
      self._t.join()

  def summary(self):
    s = sorted(self.samples)
    return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------- CPU oracle legs (checker / baseline only)
def oracle_params_from_blob(shape, blob):
  """The haiku-shaped float64 parameter dict the oracle takes, from the blob the GPU arm runs."""
  from cnf_ot_b200.layout import unpack
  from oracle import flow as oflow
  spec = oflow.FlowSpec(shape.dim, shape.num_layers, [shape.hidden] * shape.mlp_layers, shape.num_bins)
  # the reference's dtypes: float64 everywhere, the shared `first` leaf float32 (flows.py:47-55)
  return unpack(shape, blob.detach().cpu(), like=oflow.init_params(spec, seed=0))


def oracle_value_and_grad(cfg, shape, blob, inputs):
  """loss (float), gradient (float64 blob) of the CPU restatement on explicit inputs."""
  from cnf_ot_b200.layout import pack
  from oracle import losses as olosses
  spec = olosses.spec_from_config(cfg)
  params = oracle_params_from_blob(shape, blob)
  t0 = time.perf_counter()
  loss, grads = olosses.value_and_grad(cfg, spec, params, inputs)
  dt = time.perf_counter() - t0
  return float(loss), pack(shape, grads, torch.float64), dt


def parity_against_oracle(cfg, shape, blob, inputs_dev, t_batch, lam, out_dev):
  """Relative loss / gradient error of a device result against the oracle on the same blob and inputs."""
  dbl = lambda x: None if x is None else x.detach().cpu().double()
  inputs = {"t_batch": torch.tensor(list(t_batch), dtype=torch.float64)}
  for k in ("latent", "latent_sub", "src", "tgt"):
    if inputs_dev.get(k) is not None:
      inputs[k] = dbl(inputs_dev[k])
  if "latent" not in inputs:          # ot: the oracle's sub-batch rows
    inputs["latent"] = inputs["latent_sub"]
  loss, G, dt = oracle_value_and_grad(cfg, shape, blob, inputs)
  out = out_dev.detach().cpu().double()
  n = shape.blob_size
  return {"loss_rel": abs(float(out[n]) - loss) / abs(loss),
          "grad_rel": float((out[:n] - G).abs().max() / G.abs().max()),
          "loss": float(out[n]), "oracle_loss": loss, "oracle_seconds": dt}


def cpu_baseline(budget_s=15.0):
  """The oracle (port of the reference step) timed on the host cores on a bounded sample."""
  from oracle import losses as olosses
  from util import make_inputs, make_params
  torch.set_num_threads(os.cpu_count() or 1)

  def timer(rows):
    cfg = mfc_cfg("ot", "obstacle", 2, rows)
    spec, params = make_params(cfg, SIGMA)
    inputs = make_inputs(cfg)

    def step():
      t0 = time.perf_counter()
      olosses.value_and_grad(cfg, spec, params, inputs)
      return time.perf_counter() - t0
    return step

  probe = timer(1 << 13)
  probe()
  rate = (1 << 13) / probe()
  rows = 1 << 13
  while rows < B_PER_GPU and (rows * 2) / rate * 3 < budget_s:
    rows *= 2
  step = timer(rows)
  step()
  best = min(step() for _ in range(2))
  return {"value": rows / best, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
          "sample": f"oracle (torch f64 restatement of the reference step) on {rows} rows of the "
                    f"same workload, best of 2 after 1 warm-up"}


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  from oracle import losses as olosses
  from util import make_inputs, make_params
  torch.set_num_threads(os.cpu_count() or 1)

  def timer(rows):
    cfg = mfc_cfg("ot", "obstacle", 2, rows)
    spec, params = make_params(cfg, SIGMA)
    inputs = make_inputs(cfg)
    return lambda: olosses.value_and_grad(cfg, spec, params, inputs)

  # bounded sample per step so K + W steps end within minutes
  probe = timer(1 << 12)
  probe()
  t0 = time.perf_counter()
  probe()
  rate = (1 << 12) / (time.perf_counter() - t0)
  total = args.steps + args.warmup
  rows = 1 << 12
  while rows < B_PER_GPU and (rows * 2) / rate * total < 120.0:
    rows *= 2
  step = timer(rows)
  for _ in range(args.warmup):
    step()
  t0 = time.perf_counter()
  for _ in range(args.steps):
    step()
  el = time.perf_counter() - t0
  value = rows * args.steps / el
  sample = (f"reference step restated on CPU (oracle/, torch f64, autograd), {rows} rows per step "
            f"(bounded sample of the 2^18-row workload), {torch.get_num_threads()} threads")
  emit({
    "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
    "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3,
    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
    "data": "synthetic", "config": config_block(args.gpus),
    "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                     "sample": sample},
    "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "gpu_launches": 0, "run": {"rows_per_step_cpu": rows},
  })


# ---------------------------------------------------------------- our arm
def make_blob(shape, device, sigma, seed=43):
  """Reference init (FlowModel.init) + N(0, sigma^2) on biases, output layers and `first`."""
  from cnf_ot_b200 import random as crandom
  from cnf_ot_b200.flows import FlowModel
  model = FlowModel(shape, device)
  params = model.init(crandom.PRNGKey(3))
  g = torch.Generator(device="cpu").manual_seed(seed)
  if sigma > 0:
    for mod, leaves in params.items():
      for name, v in leaves.items():
        if name == "w" and mod.startswith("mlp_"):
          continue
        v.add_((torch.randn(v.shape, generator=g) * sigma).to(device))
  return params.blob


def peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    with open(path) as f:
      return json.load(f), "measured (MEASURED_PEAKS.json)"
  return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "bf16_tflops_sustained": 1392.5}, "fallback (B200_PROFILING.md)"


def time_region(fn, n, stream_sync, first=0):
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  stream_sync()
  e0.record()
  for i in range(first, first + n):
    fn(i)
  e1.record()
  stream_sync()
  return e0.elapsed_time(e1) / 1e3  # seconds


class Dist:
  """Rank plumbing of one bench process."""

  def __init__(self):
    import torch.distributed as td
    self.td = td
    self.world = int(os.environ.get("WORLD_SIZE", "1"))
    self.rank = int(os.environ.get("RANK", "0"))
    self.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
      raise SystemExit("bench.py needs a CUDA device: cnf_ot_b200 has no CPU path")
    torch.cuda.set_device(self.local)
    self.dev = torch.device("cuda", self.local)
    if self.world > 1:
      os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the ONE JSON line
      td.init_process_group("nccl", device_id=self.dev)

  def sync(self):
    if self.world > 1:
      self.td.barrier()
    torch.cuda.synchronize()

  def max_over_ranks(self, seconds):
    t = torch.tensor(list(seconds), dtype=torch.float64, device=self.dev)
    if self.world > 1:
      self.td.all_reduce(t, op=self.td.ReduceOp.MAX)
    return t.tolist()

  def close(self):
    if self.world > 1:
      self.td.barrier()
      self.td.destroy_process_group()


def timed_reps(dist, step, steps, reps):
  """`steps` consecutive timed steps (indices 0 .. steps-1) in `reps` blocks (fewer when steps < reps); per-step
  seconds of each block, max over ranks.  The blocks are delimited by events recorded between the steps, with no
  synchronise between them, so only the first block starts from an idle device."""
  reps = max(1, min(reps, steps))
  sizes = [steps // reps + (r < steps % reps) for r in range(reps)]
  ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
  dist.sync()
  ev[0].record()
  i = 0
  for r, n in enumerate(sizes):
    for _ in range(n):
      step(i)
      i += 1
    ev[r + 1].record()
  dist.sync()
  return dist.max_over_ranks([ev[r].elapsed_time(ev[r + 1]) / 1e3 / n for r, n in enumerate(sizes)])


def spread(per_step_s):
  return {"median_ms": statistics.median(per_step_s) * 1e3, "min_ms": min(per_step_s) * 1e3,
          "max_ms": max(per_step_s) * 1e3, "reps": len(per_step_s)}


class Workload:
  """One BASELINE config on this rank: shapes, parameter blob, rotating synthetic input sets, the step closure."""

  def __init__(self, name, dist, max_sets_bytes=2 * 126 * 2**20 + 2**20, oracle_rows=None, rows_override=None):
    from cnf_ot_b200 import ops
    from cnf_ot_b200.layout import FlowShape
    label, typ, sub, D, (H, L, M, K), (rule, rows), sigma = WORKLOADS[name]
    self.name, self.label, self.typ, self.sub, self.D, self.rule, self.sigma = name, label, typ, sub, D, rule, sigma
    self.dist = dist
    dev, world, rank = dist.dev, dist.world, dist.rank
    if oracle_rows is not None:     # the small-batch oracle check: one GPU's worth, whole batch on this rank
      self.gB, self.B = oracle_rows, oracle_rows
    elif rows_override:             # --only cfgN --rows-per-gpu R (e.g. cfg 5 at its BASELINE size, 2^21 rows per GPU)
      self.gB, self.B, self.rule = rows_override * world, rows_override, "weak"
    elif rule == "weak":
      self.gB, self.B = rows * world, rows
    else:
      self.gB, self.B = rows, rows // world
    self.gb, self.b = self.gB // 32, self.B // 32
    self.lam = 5000.0
    self.cfg = mfc_cfg(typ, sub, D, self.gB, H, L, M, K, self.lam)
    self.shape = FlowShape(D, L, M, H, K)
    self.problem = ops.problem_desc(self.cfg)
    if name == "cfg5":
      # haiku-like scale for the hidden matrices (1/sqrt(fan_in) ~ 0.04 at 512), small output layers: a well-conditioned flow
      g = torch.Generator(device=dev).manual_seed(43)
      self.W = torch.randn(self.shape.blob_size, device=dev, generator=g) * 0.02
    else:
      self.W = make_blob(self.shape, dev, sigma)
    if world > 1:
      dist.td.broadcast(self.W, 0)
    row_bytes = D * 4
    per_set = ((2 if typ == "ot" else 1) * self.B + self.b) * row_bytes
    self.bytes_per_set = per_set
    self.n_sets = 1 if oracle_rows is not None else max(2, min(64, max_sets_bytes // max(per_set, 1) + 1))
    if per_set > 126 * 2**20:
      self.n_sets = 2
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    centres = torch.tensor([[0., 5.], [5., 0.], [0., -5.], [-5., 0.], [3., 4.], [3., -4.], [-3., -4.], [-3., 4.]], device=dev)
    self.sets = []
    for _ in range(self.n_sets):
      s = {"latent_sub": torch.randn(self.b, D, device=dev, generator=g)}
      if typ == "ot":
        z = torch.randn(self.B, D, device=dev, generator=g)
        if sub == "obstacle" and D == 2:   # the live 8-mode mixture source (applications.py:34-71)
          s["src"] = z + centres[torch.randint(0, 8, (self.B, ), device=dev, generator=g)]
        else:                               # Gaussian -> Gaussian (applications.py:28-32, ot.py:72-80)
          s["src"] = z - 3.0
        s["tgt"] = z
      else:
        s["latent"] = torch.randn(self.B, D, device=dev, generator=g)
      self.sets.append(s)
    horizon = 1.0 if typ == "ot" else float(self.cfg[typ]["T"])
    self.t_vals = (torch.rand(4096, generator=torch.Generator().manual_seed(42)) * horizon).tolist()
    self.out = torch.empty(self.shape.blob_size + 8, dtype=torch.float32, device=dev)
    self.px, self.transport = None, "none"
    self.wide = H > 64

  def attach_peer_exchange(self):
    """N > 1: fused all-reduce over peer-mapped memory where the library supports it, else NCCL."""
    if self.dist.world == 1:
      return
    if self.wide:
      self.transport = f"NCCL all-reduce ({self.shape.blob_size * 4 >> 20} MiB)"
      return
    if self.shape.blob_size + 8 > 9000:
      # the exchange kernel needs all its blocks co-resident (ADVICE r1): larger buffers go through NCCL
      self.transport = "NCCL all-reduce"
      return
    try:
      from cnf_ot_b200 import dist as cdist
      self.px = cdist.PeerExchange(self.shape, self.dist.dev)
      self.transport = "fused in the step's reduction over peer-mapped memory (NVLink/NVSwitch)"
    except Exception as exc:  # symmetric memory unavailable
      log(f"PeerExchange unavailable ({exc!r}); using NCCL all-reduce")
      self.transport = "NCCL all-reduce"

  def args_of(self, s, i):
    return (s.get("latent"), s["latent_sub"], s.get("src"), s.get("tgt"), [self.t_vals[i % 4096]])

  def step(self, i, peers="default", out=None):
    from cnf_ot_b200 import ops
    s = self.sets[i % self.n_sets]
    lat, sub, src, tgt, tb = self.args_of(s, i)
    px = self.px if peers == "default" else peers
    out = self.out if out is None else out
    ops.mfc_step(self.shape, self.problem, self.W, lat, sub, src, tgt, tb, self.lam, self.gB, self.gb, out=out, peers=px)
    if self.dist.world > 1 and px is None:
      self.dist.td.all_reduce(out)
    return out

  def flops_per_step(self):
    H, L, M = self.shape.hidden, self.shape.num_layers, self.shape.mlp_layers
    evals = flow_evals_per_step(self.typ, self.sub, self.D, self.B, self.b)
    return evals * 3.0 * mlp_flops_per_row_eval(self.D, L, M, H), evals


def oracle_check_small(name, dist, rows):
  """Small-batch parity of one config against the CPU oracle (rank 0, its own GPU only)."""
  from cnf_ot_b200 import ops
  w = Workload(name, dist_single(dist), oracle_rows=rows)
  s = w.sets[0]
  lat, sub, src, tgt, tb = w.args_of(s, 0)
  out = ops.mfc_step(w.shape, w.problem, w.W, lat, sub, src, tgt, tb, w.lam, w.gB, w.gb)
  torch.cuda.synchronize()
  r = parity_against_oracle(w.cfg, w.shape, w.W, s, tb, w.lam, out)
  return {"rows": rows, "loss_rel": r["loss_rel"], "grad_rel": r["grad_rel"], "oracle_seconds": r["oracle_seconds"]}


class _Single:
  """A world-size-1 view of a Dist (rank 0's own GPU)."""

  def __init__(self, dist):
    self.dev, self.world, self.rank, self.local, self.td = dist.dev, 1, 0, dist.local, dist.td

  def sync(self):
    torch.cuda.synchronize()

  def max_over_ranks(self, seconds):
    return list(seconds)


def dist_single(dist):
  return _Single(dist)


def fused_rooflines(w, t_step, pk, pk_src):
  """The three views of the fused step kernel: HBM (contract), fp32 CUDA-core peak on algorithmic FLOPs."""
  hbm = float(pk["hbm_gbs"])
  clk = float(pk.get("sm_max_mhz", 1965.0)) * 1e6
  n = w.shape.blob_size
  alg_bytes = w.bytes_per_set + n * 4 + (n + 8) * 4
  flops, evals = w.flops_per_step()
  fp32_peak = 148 * 128 * 2 * clk / 1e12
  ach = alg_bytes / t_step / 1e9
  return {
    "roofline": {"bound": "hbm", "kernel": "mfc_step_kernel", "achieved": ach, "peak": hbm, "unit": "GB/s",
                 "frac": ach / hbm, "traffic": None, "peak_source": pk_src, "algorithmic_bytes_per_launch": alg_bytes},
    "roofline_fp32": {"bound": "fp32", "kernel": "mfc_step_kernel", "achieved": flops / t_step / 1e12, "peak": fp32_peak,
                      "unit": "TFLOP/s", "frac": flops / t_step / 1e12 / fp32_peak, "flops_per_launch": flops,
                      "rows_through_flow_per_launch": evals},
  }


def kernel_fingerprint():
  """Identity of the loaded library: the profile-derived constants in profiles/traffic.json are only
  trusted when they were captured from the same kernels (tools/ncu_summary.py records the same hash)."""
  from cnf_ot_b200 import _lib
  h = hashlib.sha256()
  csrc = os.path.join(ROOT, "cnf_ot_b200", "csrc")
  for fn in sorted(os.listdir(csrc)):
    if fn.endswith((".cu", ".cuh", ".h")):
      with open(os.path.join(csrc, fn), "rb") as f:
        h.update(fn.encode())
        h.update(f.read())
  return h.hexdigest()[:16]


def profile_constants():
  """(dram bytes per launch, warp instructions per launch, note) of mfc_step_kernel from profiles/traffic.json, or
  Nones when the file was captured from other kernel sources than the ones built here."""
  tpath = os.path.join(ROOT, "profiles", "traffic.json")
  if not os.path.exists(tpath):
    return None, None, "no profiles/traffic.json"
  with open(tpath) as f:
    tj = json.load(f)
  fp = kernel_fingerprint()
  if tj.get("csrc_sha16") != fp:
    return None, None, f"profiles/traffic.json was captured from other kernel sources ({tj.get('csrc_sha16')} != {fp}): not used"
  return (tj.get("mfc_step_kernel_dram_bytes_per_launch"), tj.get("mfc_step_kernel_warp_insts_per_launch"),
          tj.get("source"))


def spline_rooflines(peak_gbs):
  """Stand-alone spline kernels (seam 2), HBM-bound: algorithmic bytes 4P+12 / 8P+16 per row."""
  from cnf_ot_b200 import _lib
  lib = _lib.load()
  n, K, P = 1 << 24, 5, 16
  theta = torch.randn(n, P, device="cuda") * SIGMA
  v = torch.randn(n, device="cuda") * 3
  y, ld = torch.empty_like(v), torch.empty_like(v)
  go, gl = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
  gi, gp = torch.empty_like(v), torch.empty_like(theta)
  s = torch.cuda.current_stream().cuda_stream
  calls = {
    "rqs_forward": (lambda i: lib.cnfot_rqs_forward(s, v.data_ptr(), theta.data_ptr(), n, K, -10., 10., 1e-4, 1e-4, y.data_ptr(), ld.data_ptr(), 0), 4 * P + 12),
    "rqs_inverse": (lambda i: lib.cnfot_rqs_inverse(s, v.data_ptr(), theta.data_ptr(), n, K, -10., 10., 1e-4, 1e-4, y.data_ptr(), ld.data_ptr(), 0), 4 * P + 12),
    "rqs_forward_vjp": (lambda i: lib.cnfot_rqs_forward_vjp(s, v.data_ptr(), theta.data_ptr(), go.data_ptr(), gl.data_ptr(), n, K, -10., 10., 1e-4, 1e-4, gi.data_ptr(), gp.data_ptr()), 8 * P + 16),
    "rqs_inverse_vjp": (lambda i: lib.cnfot_rqs_inverse_vjp(s, v.data_ptr(), theta.data_ptr(), go.data_ptr(), gl.data_ptr(), n, K, -10., 10., 1e-4, 1e-4, gi.data_ptr(), gp.data_ptr()), 8 * P + 16),
  }
  out = {}
  for name, (fn, bpr) in calls.items():
    for i in range(3):
      fn(i)
    el = time_region(fn, 10, torch.cuda.synchronize) / 10
    gbs = n * bpr / el / 1e9
    out[name] = {"bound": "hbm", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s",
                 "frac": gbs / peak_gbs, "rows": n, "bytes_per_row": bpr, "us": el * 1e6}
  return out


def dense_roofline(dev, pk, pk_src):
  """cfg 5's dominant kernel (hidden-layer GEMM rows x 512 x 512, 3xTF32 on tcgen05), timed alone on one row chunk."""
  from cnf_ot_b200 import ops
  H, rows = 512, 4 * 148 * 128
  X = torch.randn(rows, H, device=dev)
  P = ops.PreparedDense(torch.randn(H, H, device=dev) / H**0.5)
  bias = torch.zeros(H, device=dev)
  Y = torch.empty(rows, H, device=dev)
  fn = lambda i: ops.dense_forward(X, P, bias=bias, epilogue="bias_relu", out=Y)
  for i in range(3):
    fn(i)
  tk = time_region(fn, 20, torch.cuda.synchronize) / 20
  tf32_peak = float(pk.get("bf16_tflops_sustained", 1392.5)) / 2.0
  pipe = 3 * 2.0 * rows * H * H / tk / 1e12   # tf32 MMA flops issued (3 per fp32-fidelity product)
  traffic, tsrc = None, "no profiles/traffic.json entry"
  tpath = os.path.join(ROOT, "profiles", "traffic.json")
  if os.path.exists(tpath):
    with open(tpath) as f:
      tj = json.load(f)
    if tj.get("csrc_sha16") == kernel_fingerprint() and tj.get("dense_tc_kernel_256_1_dram_bytes_per_launch"):
      # captured on 2^18 rows: the kernel streams X once and writes Y once, so the bytes scale with the rows
      traffic = int(tj["dense_tc_kernel_256_1_dram_bytes_per_launch"] * rows / float(1 << 18))
      tsrc = tj.get("dense_tc_kernel_source", "") + f", 2^18 rows, scaled to {rows} rows"
    else:
      tsrc = "profiles/traffic.json was captured from other kernel sources: not used"
  return {"bound": "tensor", "kernel": "dense_tc_kernel<256,1> (hidden layer, rows x 512 x 512, timed alone)",
          "achieved": pipe, "peak": tf32_peak, "unit": "TFLOP/s", "frac": pipe / tf32_peak, "traffic": traffic,
          "traffic_source": tsrc, "algorithmic_bytes_per_launch": 2 * rows * H * 4 + 2 * H * H * 4,
          "peak_source": pk_src + ": bf16_tflops_sustained / 2 (tf32)", "fp32_fidelity_tflops": pipe / 3,
          "us_per_launch": tk * 1e6}


def train_loop_block(dist, batch):
  """The reference's training loop (solvers.py:99-106) at its own batch size: device-resident updates (draws +
  value_and_grad + all-reduce + Adam in one kernel), 100 updates per CUDA graph.  Wall clock per update (host
  timer around replay + synchronize) next to the device time of the same updates."""
  from cnf_ot_b200 import ops
  from cnf_ot_b200.layout import FlowShape
  shape = FlowShape(2, 2, 2, 16, 5)
  cfg = mfc_cfg("rwpo", "double_well", 2, batch)
  cfg["rwpo"].update(T=2, beta=10)          # config/mfc.yaml as shipped
  problem = ops.problem_desc(cfg)
  W = make_blob(shape, dist.dev, 0.0)       # the reference's initialisation
  rank, world = dist.rank, dist.world
  B, b = batch, batch // 32
  rs = slice(rank * B // world, (rank + 1) * B // world)
  ss = slice(rank * b // world, (rank + 1) * b // world)
  px = None
  if world > 1:
    from cnf_ot_b200 import applications
    px = applications.peer_exchange(shape, dist.dev)
  state = ops.TrainState(shape, W, 42, peers=px)
  K = 100
  hist = torch.zeros(K * 8, device=dist.dev)
  one = lambda: ops.mfc_update(shape, problem, state, W, 1, 5000.0, B, b, 1e-3, rows_B=rs, rows_b=ss, loss_hist=hist)
  for _ in range(5):
    one()
  dist.sync()
  t0 = time.perf_counter()
  for _ in range(K):
    one()
  dist.sync()
  eager = (time.perf_counter() - t0) / K
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g):
    for _ in range(K):
      one()
  state.steps_issued -= K
  if px is not None:
    px.epoch -= K

  def replay():
    g.replay()
    state.steps_issued += K
    if px is not None:
      px.epoch += K

  replay()
  dist.sync()
  walls, devs = [], []
  for _ in range(5):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.sync()
    t0 = time.perf_counter()
    e0.record()
    replay()
    e1.record()
    torch.cuda.synchronize()
    walls.append((time.perf_counter() - t0) / K)
    devs.append(e0.elapsed_time(e1) / 1e3 / K)
  wall, dev = dist.max_over_ranks([statistics.median(walls), statistics.median(devs)])
  losses = hist[:state.step_count()].cpu()
  return {"batch": batch, "updates_per_graph": K, "wall_us_per_update": wall * 1e6, "device_us_per_update": dev * 1e6,
          "eager_wall_us_per_update": eager * 1e6, "wall_over_device": wall / dev, "samples_per_s": batch / wall,
          "loss_first": float(losses[0]), "loss_last": float(losses[-1]), "updates_run": int(losses.numel()),
          "workload": "config/mfc.yaml (rwpo / double_well, T=2, beta=10), reference initialisation, lr 1e-3",
          "api": "cnfot_mfc_update: draws + value_and_grad + all-reduce + Adam in ONE kernel launch per update"}


def density_block(dev):
  """SURVEY.md 8f row 3: the density consumers after training, one launch each -- ten 500 x 500 grids of
  exp(log_prob) (the reference: 100 x 100 snapshots, utils.py:572-595, and a 500 x 500 grid, solvers.py:282-301) and
  the 10^6-sample Monte-Carlo L2 error (solvers.py:254-278)."""
  from cnf_ot_b200 import ops
  from cnf_ot_b200.layout import FlowShape
  shape = FlowShape(2, 2, 2, 16, 5)
  W = make_blob(shape, dev, SIGMA)
  ts = torch.linspace(0, 1, 10).tolist()
  grid = lambda i: ops.density_grid(shape, W, ts, [-6, 6, -6, 6], 500, 500)
  mc = lambda i: ops.density_mc(shape, W, 1.0, 1234 + i, 1000000, ref=(1.0, 4.0, 0.6353352832366127))
  out = {}
  for name, fn, pts in (("grid_10x500x500", grid, 10 * 500 * 500), ("mc_rmse_1e6", mc, 1000000)):
    for i in range(3):
      fn(i)
    el = time_region(fn, 10, torch.cuda.synchronize) / 10
    out[name] = {"us": el * 1e6, "points_per_s": pts / el}
  out["api"] = "cnfot_density_grid / cnfot_density_mc: one kernel launch, grid points and latent rows generated on chip"
  return out


def per_config_entry(name, dist, args, pk, pk_src):
  """Timing + roofline + small-batch oracle check of one BASELINE config other than the headline one."""
  steps = {"cfg1": 250, "cfg2": 100, "cfg3": 50, "cfg4": 9, "cfg5": 2}[name]
  reps = {"cfg1": 5, "cfg2": 5, "cfg3": 5, "cfg4": 3, "cfg5": 1}[name]
  if args.only:
    steps, reps = args.steps, args.reps
  w = Workload(name, dist, rows_override=args.rows_per_gpu if args.only else None)
  w.attach_peer_exchange()
  for i in range(3 if name != "cfg5" else 1):
    w.step(i)
  per = timed_reps(dist, w.step, steps, reps)
  if args.only and args.dump_outputs and dist.rank == 0:
    dump_outputs(args.dump_outputs, w.shape, w.out)
  t_step = statistics.median(per)
  entry = {
    "workload": w.label, "dim": w.D, "params": w.shape.blob_size, "batch_per_gpu": w.B, "global_batch": w.gB,
    "scaling": w.rule, "steps": steps, "ms_per_step": t_step * 1e3, "spread": spread(per),
    "value": w.gB / t_step, "unit": UNIT, "all_reduce": w.transport, "param_sigma": w.sigma,
    "input_sets": w.n_sets, "input_set_bytes": w.bytes_per_set,
    "loss_last_step": float(w.out[w.shape.blob_size]),
  }
  if dist.rank == 0:
    if w.wide:
      entry["roofline"] = dense_roofline(dist.dev, pk, pk_src)
      flops, evals = w.flops_per_step()
      entry["roofline"]["step_algorithmic_tflops"] = flops / t_step / 1e12
    else:
      entry.update(fused_rooflines(w, t_step, pk, pk_src))
  del w
  torch.cuda.empty_cache()
  if dist.rank == 0 and not args.no_oracle:
    rows = {"cfg1": 4096, "cfg3": 4096, "cfg4": 512, "cfg5": 64}[name]
    try:
      entry["oracle_check"] = oracle_check_small(name, dist, rows)
    except Exception as exc:   # keep the line: a failed check is reported, not hidden
      entry["oracle_check"] = {"error": repr(exc)}
    torch.cuda.empty_cache()
  return entry


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 20


def dump_outputs(path, shape, out):
  """The buffer the last timed step returned to its caller, [gradient | loss slots] (include/cnfot.h), as
  path/gradient.npy and path/loss_slots.npy (float32): the inputs are seeded, so two builds compare output for output.
  A buffer over DUMP_MAX_BYTES (cfg 5: 139 M parameters) keeps the files under it: gradient.npy then holds the entries
  at DUMP_SAMPLE indices drawn without replacement from a fixed seed, written in ascending order to
  gradient_index.npy (float64, exact)."""
  import numpy as np
  os.makedirs(path, exist_ok=True)
  n = shape.blob_size
  grad = out.detach()[:n]
  if out.numel() * 4 > DUMP_MAX_BYTES:
    idx = np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    grad = grad[torch.from_numpy(idx).to(grad.device)]
    np.save(os.path.join(path, "gradient_index.npy"), idx.astype(np.float64))
  np.save(os.path.join(path, "gradient.npy"), grad.float().cpu().numpy())
  np.save(os.path.join(path, "loss_slots.npy"), out.detach()[n:].float().cpu().numpy())


def timeline_block(w, n=24):
  """Where one step's time goes: %globaltimer stamps written by the kernel itself (cnfot_debug_step_timeline)."""
  from cnf_ot_b200 import _lib
  lib = _lib.load()
  dev = w.out.device
  init = torch.tensor([-1, 0, -1, 0, 0, 0, 0, 0], dtype=torch.int64)
  words = torch.empty(n, 8, dtype=torch.int64, device=dev)
  for i in range(n):
    words[i].copy_(init)
  torch.cuda.synchronize()
  try:
    for i in range(n):
      lib.cnfot_debug_step_timeline(words[i].data_ptr())
      w.step(i)
  finally:
    lib.cnfot_debug_step_timeline(None)
  torch.cuda.synchronize()
  t = words.cpu().double()[4:]
  med = lambda x: float(x.median()) / 1e3
  return {"unit": "us", "kernel_span": med(t[:, 5] - t[:, 0]), "cta_setup": med(t[:, 1] - t[:, 0]),
          "tiles_until_first_cta_idle": med(t[:, 2] - t[:, 1]), "tiles_until_last_cta_idle": med(t[:, 3] - t[:, 1]),
          "flush": med(t[:, 4] - t[:, 3]), "reduction_tail": med(t[:, 5] - t[:, 4]),
          "gap_to_next_kernel": med(t[1:, 0] - t[:-1, 5]),
          "note": "medians over 20 consecutive steps of the timed workload, stamped by the kernel (tools/step_timeline.py); the "
                  "tail is reduction (+ all-reduce at N > 1), measured from the last CTA's arrival to the last CTA's exit"}



def run_ours(args):
  from cnf_ot_b200 import _lib, ops
  dist = Dist()
  td, world, rank, dev = dist.td, dist.world, dist.rank, dist.dev
  _lib.load()
  pk, pk_src = peaks()

  w = Workload("cfg2", dist)
  w.attach_peer_exchange()
  shape, n = w.shape, w.shape.blob_size
  warm = max(args.warmup, 3)
  for i in range(warm):
    w.step(i)
  with ClockSampler(dist.local) as clk:
    per = timed_reps(dist, w.step, args.steps, args.reps)
  t_step = statistics.median(per)
  value = w.gB / t_step
  loss_dev = float(w.out[n])
  launch = _lib.last_launch_info()
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, shape, w.out)

  # ---- parity at the FULL batch: same blob, same input set, CPU oracle (rank 0's shard as a whole batch)
  parity = None
  if rank == 0 and not args.no_oracle:
    s = w.sets[0]
    lat, sub, src, tgt, tb = w.args_of(s, 0)
    o = ops.mfc_step(shape, w.problem, w.W, lat, sub, src, tgt, tb, w.lam, w.B, w.b)
    torch.cuda.synchronize()
    pcfg = mfc_cfg(w.typ, w.sub, w.D, w.B)
    parity = parity_against_oracle(pcfg, shape, w.W, s, tb, w.lam, o)
    parity["rows"] = w.B
    parity["note"] = ("the timed kernel on input set 0 of this run (this rank's 2^18 rows as one batch) against "
                      "oracle/ (torch f64) on the same parameter blob and rows; tolerance 2e-5 / 5e-5 (tests/test_gpu_step.py)")

  # ---- N > 1: the fused step + all-reduce against step + NCCL all-reduce, same inputs
  dp_check = None
  if world > 1:
    a = torch.empty_like(w.out)
    w.step(0, peers=None, out=a)            # plain step, then NCCL all-reduce
    ref = a.clone()
    if w.px is not None:
      w.step(0, out=a)                      # fused
    torch.cuda.synchronize()
    err = float((a.double() - ref.double()).abs().max() / ref.double().abs().max())
    digest = torch.tensor(list(hashlib.sha256(a.cpu().numpy().tobytes()).digest()[:8]), dtype=torch.int64, device=dev)
    alld = [torch.empty_like(digest) for _ in range(world)]
    td.all_gather(alld, digest)
    dp_check = {"dp_check_rel_err": err, "identical_on_all_ranks": all(bool((d == alld[0]).all()) for d in alld),
                "fused": w.px is not None,
                "note": "cnfot_mfc_step_dp (all-reduce inside the step's reduction kernel) vs cnfot_mfc_step + NCCL all_reduce"}

  # ---- e2e: the call a user of the reference makes -- update(params, key): host weights and the PRNG key in,
  # [gradient | loss] out; the draws are made inside the kernel (the reference draws inside its jitted step too)
  hW = w.W.cpu().contiguous().pin_memory()
  hout = torch.empty(n + 8, dtype=torch.float32).pin_memory()
  dW2 = torch.empty_like(w.W)
  rs, ss = slice(rank * w.B, (rank + 1) * w.B), slice(rank * w.b, (rank + 1) * w.b)

  def step_e2e(i):
    if world == 1:
      ops.mfc_step_rng_host(shape, w.problem, hW, 0x5EED, i, 1, w.lam, w.gB, w.gb, hout, device=dev)
    else:
      dW2.copy_(hW, non_blocking=True)
      ops.mfc_step_rng(shape, w.problem, dW2, 0x5EED, i, 1, w.lam, w.gB, w.gb, rows_B=rs, rows_b=ss, out=w.out, peers=w.px)
      if w.px is None:
        td.all_reduce(w.out)
      hout.copy_(w.out, non_blocking=True)
      torch.cuda.synchronize()

  for i in range(3):
    step_e2e(i)
  per_e = timed_reps(dist, step_e2e, args.steps, args.reps)
  t_e2e = statistics.median(per_e)
  h2d = n * 4 + 16          # weights + key / step
  d2h = (n + 8) * 4

  # the round-1 form of the same call: explicit HOST row arrays (pinned, read in place by the kernel over PCIe)
  n_host = 8
  pin = lambda x: None if x is None else x.cpu().contiguous().pin_memory()
  hsets = [{k: pin(v) for k, v in s.items()} for s in w.sets[:n_host]]

  def step_e2e_rows(i):
    s = hsets[i % n_host]
    lat, sub, src, tgt, tb = w.args_of(s, i)
    if world == 1:
      ops.mfc_step_host(shape, w.problem, hW, lat, sub, src, tgt, tb, w.lam, w.gB, w.gb, hout, device=dev)
    else:
      dW2.copy_(hW, non_blocking=True)
      ops.mfc_step(shape, w.problem, dW2, lat, sub, src, tgt, tb, w.lam, w.gB, w.gb, out=w.out, peers=w.px)
      if w.px is None:
        td.all_reduce(w.out)
      hout.copy_(w.out, non_blocking=True)
      torch.cuda.synchronize()

  for i in range(3):
    step_e2e_rows(i)
  per_er = timed_reps(dist, step_e2e_rows, args.steps, args.reps)
  t_e2e_rows = statistics.median(per_er)
  del hsets

  # ---- the on-chip-draw step and the device-resident update on the same workload (device-timed)
  def step_rng(i):
    ops.mfc_step_rng(shape, w.problem, w.W, 0x5EED, i, 1, w.lam, w.gB, w.gb, rows_B=rs, rows_b=ss, out=w.out, peers=w.px)
    if world > 1 and w.px is None:
      td.all_reduce(w.out)

  for i in range(3):
    step_rng(i)
  t_rng = statistics.median(timed_reps(dist, step_rng, args.steps, args.reps))
  timeline = timeline_block(w)

  line = None
  if rank == 0:
    rf = fused_rooflines(w, t_step, pk, pk_src)
    traffic, insts, tsrc = profile_constants()
    rf["roofline"]["traffic"] = traffic
    rf["roofline"]["traffic_source"] = tsrc
    rf["roofline"]["note"] = ("the fused step kernel is bound neither by HBM nor by the tensor pipe: it is latency-bound at 16 "
                              "warps per SM, half of the issue slots used (SURVEY.md §8d; DESIGN.md §4.2; ncu: profiles/): see "
                              "roofline_issue / roofline_fp32 / step_timeline; the HBM-bound kernels of the path are the "
                              "stand-alone spline kernels in roofline_spline")
    issue_peak = 148 * 4 * float(pk.get("sm_max_mhz", 1965.0)) * 1e6  # warp instructions / s
    line = {
      "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
      "warmup": warm, "ms_per_step": t_step * 1e3, "higher_is_better": True,
      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
      "config": config_block(world),
      "spread": spread(per),
      "run": {"all_reduce": w.transport, "input_sets": w.n_sets, "input_sets_mib": w.n_sets * w.bytes_per_set >> 20,
              "loss_last_step": loss_dev, "launch": launch},
      "e2e": {"value": w.gB / t_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
              "ms_per_step": t_e2e * 1e3, "spread": spread(per_e),
              "api": "cnfot_mfc_step_rng_host (C ABI): host weights + PRNG key in, [grad|loss] out; the step's draws are "
                     "made inside the kernel (Philox), like the reference draws inside its jitted update" if world == 1 else
                     "weights H2D + cnfot_mfc_step_rng (draws on chip, all-reduce in the kernel tail) + [grad|loss] D2H",
              "explicit_host_rows": {"value": w.gB / t_e2e_rows, "ms_per_step": t_e2e_rows * 1e3, "spread": spread(per_er),
                                     "h2d_bytes_per_step": w.bytes_per_set + n * 4, "d2h_bytes_per_step": d2h,
                                     "api": "cnfot_mfc_step_host: pinned host row arrays read in place over PCIe (round-1 form)"}},
      "on_chip_draws": {"value": w.gB / t_rng, "ms_per_step": t_rng * 1e3,
                        "note": "cnfot_mfc_step_rng, device-timed: same step, rows generated in the kernel instead of read from HBM"},
      "gpu_launches": args.steps,  # ONE kernel per step: mfc_step_kernel (reduction, all-reduce in its tail)
      "clocks": clk.summary(),
      "parity": parity, "dp_check": dp_check,
      "step_timeline": timeline,
      "roofline": rf["roofline"],
      "roofline_issue": {"bound": "issue", "kernel": "mfc_step_kernel",
                         "achieved": (insts / t_step / 1e9) if insts else None, "peak": issue_peak / 1e9,
                         "unit": "G warp-inst/s", "frac": (insts / t_step / issue_peak) if insts else None,
                         "warp_insts_per_launch": insts,
                         "note": "executed warp instructions per launch (ncu smsp__inst_executed.sum, profiles/) / "
                                 "live launch time, against 148 SM x 4 schedulers x max clock"},
      "roofline_fp32": rf["roofline_fp32"],
    }
    line["roofline_fp32"]["note"] = ("algorithmic conditioner FLOPs (fwd+dgrad+wgrad) only, against the CUDA-core fp32 peak "
                                     "148 SM x 128 FMA x 2 x max clock; the 16x16 layers run on the tensor pipe (3 MMAs per "
                                     "product for fp32 fidelity), the input layers and splines on CUDA cores")
  del w
  torch.cuda.empty_cache()

  tl = [train_loop_block(dist, bsz) for bsz in (2048, 4096)]
  if rank == 0:
    line["train_loop"] = tl
  if not args.no_per_config:
    pc = {}
    for name in ("cfg1", "cfg3", "cfg4", "cfg5"):
      t0 = time.time()
      try:
        pc[name] = per_config_entry(name, dist, args, pk, pk_src)
      except Exception as exc:
        if world > 1:
          raise           # ranks must stay in lock step
        pc[name] = {"error": repr(exc)}
      log(f"per_config {name}: {time.time() - t0:.1f} s")
    if rank == 0:
      line["per_config"] = pc
  if rank == 0:
    if world == 1:
      line["density_eval"] = density_block(dev)
      line["roofline_spline"] = spline_rooflines(float(pk["hbm_gbs"]))
      if not args.no_oracle:
        line["cpu_baseline"] = cpu_baseline()
    emit(line)
  dist.close()


def run_only(args):
  """One BASELINE config alone (--only cfgN [--rows-per-gpu R]): its per_config entry as the JSON line."""
  from cnf_ot_b200 import _lib
  dist = Dist()
  _lib.load()
  pk, pk_src = peaks()
  with ClockSampler(dist.local) as clk:
    e = per_config_entry(args.only, dist, args, pk, pk_src)
  if dist.rank == 0:
    line = {"metric": METRIC, "value": e["value"], "unit": UNIT, "n_gpus": dist.world, "steps": e["steps"], "warmup": 3,
            "ms_per_step": e["ms_per_step"], "higher_is_better": True, "scaling": e["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": e["workload"], "batch_per_gpu": e["batch_per_gpu"],
                                                            "global_batch": e["global_batch"]},
            "clocks": clk.summary(), "entry": e}
    emit(line)
  dist.close()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=None, help="timed steps K (default 100; 20 for --impl reference)")
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--reps", type=int, default=5, help="blocks the K timed steps are split into (median reported)")
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--no-per-config", action="store_true", help="skip the per_config block (configs 1, 3, 4, 5)")
  ap.add_argument("--no-oracle", action="store_true", help="skip every CPU-oracle leg (parity, cpu_baseline)")
  ap.add_argument("--only", default=None, choices=sorted(WORKLOADS), help="time ONE config alone (builder tool)")
  ap.add_argument("--rows-per-gpu", type=int, default=None, help="--only: rows per GPU (weak scaling)")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write what the last timed step returned as DIR/<name>.npy, at most 64 MiB (a larger "
                       "gradient as a seeded sample); not with --impl reference")
  args = ap.parse_args()
  if args.steps is None:
    args.steps = 20 if args.impl == "reference" else 100
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl == "reference":
    ap.error("--dump-outputs: the reference arm sizes its row sample from a timing probe, so its inputs differ from run to run")
  if args.impl == "reference":
    run_reference(args)
  elif args.only:
    run_only(args)
  else:
    run_ours(args)


if __name__ == "__main__":
  main()
