"""Tensor-level entry points over the C ABI.

torch is used for device memory and the current CUDA stream only; every
computation happens inside libcnfot.so.  All functions require CUDA float32
tensors (they raise otherwise -- there is no CPU path).
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from .layout import FlowShape


def _stream() -> int:
  return torch.cuda.current_stream().cuda_stream


def _dev(t: Optional[torch.Tensor], name: str, dtype=torch.float32) -> Optional[torch.Tensor]:
  if t is None:
    return None
  if not t.is_cuda:
    raise _lib.CnfotError(f"{name}: expected a CUDA tensor (cnf_ot_b200 has no CPU path)")
  if t.dtype != dtype:
    raise _lib.CnfotError(f"{name}: expected dtype {dtype}, got {t.dtype}")
  return t.contiguous()


def _ptr(t: Optional[torch.Tensor]) -> int:
  return 0 if t is None else t.data_ptr()


def _rows(t: Optional[torch.Tensor], name: str) -> Optional[torch.Tensor]:
  """Row buffers of the train step: CUDA tensors, or PINNED host tensors, which the kernel reads in
  place over PCIe (unified addressing: each row is read once, so no staging copy is needed)."""
  if t is not None and not t.is_cuda and t.is_pinned():
    if t.dtype != torch.float32 or not t.is_contiguous():
      raise _lib.CnfotError(f"{name}: expected a contiguous float32 tensor")
    return t
  return _dev(t, name)


# ---------------------------------------------------------------- seam 2: splines
def _rqs(inverse: bool, v, params, num_bins, range_min, range_max, min_bin_size, min_knot_slope,
         want_bins):
  lib = _lib.load()
  v = _dev(v, "input").reshape(-1)
  P = 3 * num_bins + 1
  params = _dev(params, "params").reshape(-1, P)
  rows = v.numel()
  if params.shape[0] != rows:
    raise _lib.CnfotError(f"params has {params.shape[0]} rows, input has {rows}")
  out = torch.empty_like(v)
  ld = torch.empty_like(v)
  bins = torch.empty(rows, dtype=torch.int32, device=v.device) if want_bins else None
  fn = lib.cnfot_rqs_inverse if inverse else lib.cnfot_rqs_forward
  with torch.cuda.device(v.device):
    _lib.check(fn(_stream(), _ptr(v), _ptr(params), rows, num_bins, range_min, range_max,
                  min_bin_size, min_knot_slope, _ptr(out), _ptr(ld), _ptr(bins)))
  return out, ld, bins


def rqs_forward(x, params, num_bins, range_min=-10.0, range_max=10.0, min_bin_size=1e-4,
                min_knot_slope=1e-4, want_bins=False):
  """RationalQuadraticSpline(params).forward_and_log_det(x) for one scalar per row."""
  return _rqs(False, x, params, num_bins, range_min, range_max, min_bin_size, min_knot_slope,
              want_bins)


def rqs_inverse(y, params, num_bins, range_min=-10.0, range_max=10.0, min_bin_size=1e-4,
                min_knot_slope=1e-4, want_bins=False):
  """RationalQuadraticSpline(params).inverse_and_log_det(y)."""
  return _rqs(True, y, params, num_bins, range_min, range_max, min_bin_size, min_knot_slope,
              want_bins)


def rqs_vjp(inverse: bool, v, params, g_out, g_logdet, num_bins, range_min=-10.0, range_max=10.0,
            min_bin_size=1e-4, min_knot_slope=1e-4):
  """Adjoints of (input, params) given adjoints of (output, logdet)."""
  lib = _lib.load()
  v = _dev(v, "input").reshape(-1)
  P = 3 * num_bins + 1
  params = _dev(params, "params").reshape(-1, P)
  g_out = _dev(g_out, "g_out").reshape(-1)
  g_logdet = _dev(g_logdet, "g_logdet").reshape(-1)
  rows = v.numel()
  g_in = torch.empty_like(v)
  g_params = torch.empty_like(params)
  fn = lib.cnfot_rqs_inverse_vjp if inverse else lib.cnfot_rqs_forward_vjp
  with torch.cuda.device(v.device):
    _lib.check(fn(_stream(), _ptr(v), _ptr(params), _ptr(g_out), _ptr(g_logdet), rows, num_bins,
                  range_min, range_max, min_bin_size, min_knot_slope, _ptr(g_in), _ptr(g_params)))
  return g_in, g_params


# ---------------------------------------------------------------- seam 1: the flow
def _cond(cond, rows, device) -> Tuple[torch.Tensor, int]:
  cond = torch.as_tensor(cond, dtype=torch.float32, device=device).reshape(-1).contiguous()
  if cond.numel() == 1:
    return cond, 0
  if cond.numel() != rows:
    raise _lib.CnfotError(f"cond has {cond.numel()} entries, expected 1 or {rows}")
  return cond, 1


def flow_eval(shape: FlowShape, weights, x, cond, inverse: bool, want_logdet=True, add_base=False):
  """flow.bijector.forward/inverse(_and_log_det); with add_base the second output is the
  log-density ConditionalTransformed returns."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  x = _dev(x, "x").reshape(-1, shape.dim)
  rows = x.shape[0]
  c, cs = _cond(cond, rows, x.device)
  out = torch.empty_like(x)
  ld = torch.empty(rows, dtype=torch.float32, device=x.device) if want_logdet else None
  fn = lib.cnfot_flow_inverse_ws if inverse else lib.cnfot_flow_forward_ws
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_flow_workspace_bytes(desc, rows)  # 0 unless the wide-conditioner engine runs
  ws = _workspace(nbytes, x.device) if nbytes > 0 else None
  with torch.cuda.device(x.device):
    _lib.check(fn(_stream(), desc, _ptr(weights), _ptr(x), _ptr(c), cs, rows, _ptr(out), _ptr(ld),
                  1 if add_base else 0, _ptr(ws), 0 if ws is None else ws.numel()))
  return out, ld


_workspaces = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
  """Scratch memory of the calling (device, stream): kernels of different streams never share partial-result rows or
  tile counters, and a buffer is only ever used on the stream whose caching-allocator block it is."""
  device = torch.device(device)
  index = device.index if device.index is not None else torch.cuda.current_device()
  key = (index, torch.cuda.current_stream(index).cuda_stream)
  ws = _workspaces.get(key)
  if ws is None or ws.numel() < nbytes:
    with torch.cuda.device(index):
      ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
    _workspaces[key] = ws
  return ws


_step_workspaces = {}


class _StepWorkspace:
  """A dedicated, registered workspace of the fused train step (cnfot_workspace_register): consecutive steps need no
  memset between them and their launches overlap (see include/cnfot.h)."""

  def __init__(self, buf):
    self.buf = buf

  def __del__(self):
    try:
      _lib.load().cnfot_workspace_release(self.buf.data_ptr())
    except Exception:
      pass


def _step_workspace(shape: FlowShape, desc, nbytes: int, device) -> torch.Tensor:
  """Scratch memory of the train step for the calling (device, stream, flow shape).  Fused per-row engine: a
  persistent registered workspace; wide-conditioner engine: the shared scratch buffer."""
  device = torch.device(device)
  lib = _lib.load()
  if not fused_update_supported(shape):
    return _workspace(nbytes, device)
  index = device.index if device.index is not None else torch.cuda.current_device()
  key = (index, torch.cuda.current_stream(index).cuda_stream, shape)
  ent = _step_workspaces.get(key)
  if ent is None or ent.buf.numel() < nbytes:
    with torch.cuda.device(index):
      buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
      _lib.check(lib.cnfot_workspace_register(_stream(), desc, buf.data_ptr(), buf.numel()))
    ent = _StepWorkspace(buf)
    _step_workspaces[key] = ent
  return ent.buf


def flow_vjp(shape: FlowShape, weights, x, cond, g_out, g_logdet, inverse: bool, add_base=False,
             want_g_in=True):
  """(g_in, g_weights) of flow_eval; g_weights is summed over rows (blob layout)."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  x = _dev(x, "x").reshape(-1, shape.dim)
  rows = x.shape[0]
  c, cs = _cond(cond, rows, x.device)
  g_out = _dev(g_out, "g_out").reshape(-1, shape.dim)
  g_logdet = _dev(g_logdet, "g_logdet")
  g_in = torch.empty_like(x) if want_g_in else None
  g_w = torch.empty(shape.blob_size, dtype=torch.float32, device=x.device)
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_flow_vjp_workspace_bytes(desc, rows)
  ws = _workspace(nbytes, x.device)
  fn = lib.cnfot_flow_inverse_vjp if inverse else lib.cnfot_flow_forward_vjp
  with torch.cuda.device(x.device):
    _lib.check(fn(_stream(), desc, _ptr(weights), _ptr(x), _ptr(c), cs, rows, _ptr(g_out),
                  _ptr(g_logdet), 1 if add_base else 0, _ptr(g_in), _ptr(g_w), ws.data_ptr(),
                  ws.numel()))
  return g_in, g_w


# ---------------------------------------------------------------- seam 3: the train step
def problem_desc(cfg: dict) -> _lib.ProblemDesc:
  """mfc.yaml dict -> cnfot_problem_desc (solvers.py:58-88)."""
  g = cfg["general"]
  typ = g["type"]
  if typ not in _lib.TYPES:
    raise Exception(f"Unknown problem type: {typ}...")
  if typ == "ot":
    sub, T, beta, a, sigma = cfg["ot"]["subtype"], 1.0, 1.0, 0.0, 0.0
  elif typ == "rwpo":
    r = cfg["rwpo"]
    sub, T, beta, a, sigma = r["pot_type"], r["T"], r["beta"], r["a"], 0.0
  else:
    f = cfg["fp"]
    sub, T, beta, a, sigma = f["velocity_field_type"], f["T"], 4.0, f["a"], f["sigma"]
  if sub not in _lib.SUBTYPES[typ]:
    raise Exception(f"Unknown {typ} subtype: {sub}")
  return _lib.ProblemDesc(_lib.TYPES[typ], _lib.SUBTYPES[typ][sub], float(T), float(beta), float(a),
                          float(sigma), float(g["dt"]), float(g["dx"]))


def mfc_step(shape: FlowShape, problem: _lib.ProblemDesc, weights, latent, latent_sub, src, tgt,
             t_batch: Sequence[float], lam: float, global_B: int, global_b: int,
             out: Optional[torch.Tensor] = None, peers=None) -> torch.Tensor:
  """value_and_grad of the configured loss on this GPU's shard.

  Returns the fp32 buffer [gradient (blob_size) | 8 loss slots] (see include/cnfot.h);
  buffers of different ranks sum to the whole-batch result.  With `peers` (a
  dist.PeerExchange) the final reduction kernel also all-reduces the buffer over peer-mapped
  memory (cnfot_mfc_step_dp): the returned buffer is already the whole-batch result."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  device = weights.device
  latent = _rows(latent, "latent")
  latent_sub = _rows(latent_sub, "latent_sub")
  src = _rows(src, "src")
  tgt = _rows(tgt, "tgt")
  rows_B = 0
  for t in (src, latent):
    if t is not None:
      rows_B = t.reshape(-1, shape.dim).shape[0]
      break
  rows_b = 0 if latent_sub is None else latent_sub.reshape(-1, shape.dim).shape[0]
  tb = torch.as_tensor(list(t_batch), dtype=torch.float32)  # host
  n_t = tb.numel()
  if out is None:
    out = torch.empty(shape.blob_size + _lib.NUM_LOSS_SLOTS, dtype=torch.float32, device=device)
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_mfc_step_workspace_bytes(desc, rows_B, rows_b, n_t)
  ws = _step_workspace(shape, desc, nbytes, device)
  with torch.cuda.device(device):
    if peers is None:
      _lib.check(lib.cnfot_mfc_step(_stream(), desc, problem, _ptr(weights), _ptr(latent),
                                    _ptr(latent_sub), _ptr(src), _ptr(tgt), tb.data_ptr(), n_t, rows_B,
                                    rows_b, global_B, global_b, float(lam), _ptr(out), ws.data_ptr(),
                                    ws.numel()))
    else:
      pd = peers.next_desc(shape)
      _lib.check(lib.cnfot_mfc_step_dp(_stream(), desc, problem, _ptr(weights), _ptr(latent),
                                       _ptr(latent_sub), _ptr(src), _ptr(tgt), tb.data_ptr(), n_t, rows_B,
                                       rows_b, global_B, global_b, float(lam), _ptr(out), ws.data_ptr(),
                                       ws.numel(), ctypes.byref(pd)))
  return out


def mfc_step_host(shape: FlowShape, problem: _lib.ProblemDesc, weights, latent, latent_sub, src,
                  tgt, t_batch: Sequence[float], lam: float, global_B: int, global_b: int,
                  out: torch.Tensor, device=None) -> torch.Tensor:
  """Same step with HOST tensors in and out; transfers are inside the call.  Pinned row buffers are
  read in place by the kernel (zero-copy), pageable ones are staged with cudaMemcpyAsync."""
  lib = _lib.load()
  device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
  for name, t in (("weights", weights), ("latent", latent), ("latent_sub", latent_sub),
                  ("src", src), ("tgt", tgt), ("out", out)):
    if t is not None and (t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous()):
      raise _lib.CnfotError(f"{name}: expected a contiguous float32 host tensor")
  rows_B = 0
  for t in (src, latent):
    if t is not None:
      rows_B = t.reshape(-1, shape.dim).shape[0]
      break
  rows_b = 0 if latent_sub is None else latent_sub.reshape(-1, shape.dim).shape[0]
  tb = torch.as_tensor(list(t_batch), dtype=torch.float32)
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_mfc_step_host_workspace_bytes(desc, rows_B, rows_b, tb.numel())
  ws = _workspace(nbytes, device)
  with torch.cuda.device(device):
    _lib.check(lib.cnfot_mfc_step_host(_stream(), desc, problem, _ptr(weights), _ptr(latent),
                                       _ptr(latent_sub), _ptr(src), _ptr(tgt), tb.data_ptr(),
                                       tb.numel(), rows_B, rows_b, global_B, global_b, float(lam),
                                       _ptr(out), ws.data_ptr(), ws.numel()))
  return out


# ---------------------------------------------------------------- the step's draws, made on chip
def philox_rows(key: int, step: int, source: int, global_rows: int, dim: int, device, rows=None) -> torch.Tensor:
  """Rows `rows` (a slice of range(global_rows); default all) of the (global_rows, dim) array the step kernel draws
  for (key, step): `source` is _lib.ROWS_NORMAL or _lib.ROWS_OT_SOURCE."""
  lib = _lib.load()
  rs = slice(0, global_rows) if rows is None else rows
  out = torch.empty(rs.stop - rs.start, dim, dtype=torch.float32, device=device)
  with torch.cuda.device(out.device):
    _lib.check(lib.cnfot_philox_rows(_stream(), int(key) & (2**64 - 1), int(step) & 0xFFFFFFFF, int(source),
                                     int(global_rows), rs.start, rs.stop - rs.start, int(dim), _ptr(out)))
  return out


def philox_times(key: int, step: int, n_t: int, horizon: float):
  """The n_t uniform times horizon * U[0, 1) of step (key, step), as a list of floats (computed on the host)."""
  lib = _lib.load()
  tb = torch.empty(max(n_t, 1), dtype=torch.float32)
  _lib.check(lib.cnfot_philox_times_host(int(key) & (2**64 - 1), int(step) & 0xFFFFFFFF, int(n_t), float(horizon),
                                         tb.data_ptr()))
  return tb[:n_t].tolist()


def mfc_step_rng(shape: FlowShape, problem: _lib.ProblemDesc, weights, key: int, step: int, n_t: int, lam: float,
                 global_B: int, global_b: int, rows_B=None, rows_b=None, out: Optional[torch.Tensor] = None,
                 peers=None) -> torch.Tensor:
  """cnfot_mfc_step with the draws made inside the kernel from (key, step).  rows_B / rows_b: this rank's shard as
  slices of range(global_B) / range(global_b) (default: everything)."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  device = weights.device
  rB = slice(0, global_B) if rows_B is None else rows_B
  rb = slice(0, global_b) if rows_b is None else rows_b
  if out is None:
    out = torch.empty(shape.blob_size + _lib.NUM_LOSS_SLOTS, dtype=torch.float32, device=device)
  desc = _lib.flow_desc(shape)
  ws = _step_workspace(shape, desc, lib.cnfot_mfc_step_workspace_bytes(desc, rB.stop - rB.start, rb.stop - rb.start, n_t), device)
  pd = None if peers is None else peers.next_desc(shape)
  with torch.cuda.device(device):
    _lib.check(lib.cnfot_mfc_step_rng(_stream(), desc, problem, _ptr(weights), int(key) & (2**64 - 1),
                                      int(step) & 0xFFFFFFFF, int(n_t), rB.start, rB.stop - rB.start, rb.start,
                                      rb.stop - rb.start, global_B, global_b, float(lam), _ptr(out), ws.data_ptr(),
                                      ws.numel(), None if pd is None else ctypes.byref(pd)))
  return out


_rng_host_cache = {}


def mfc_step_rng_host(shape: FlowShape, problem: _lib.ProblemDesc, weights_host, key: int, step: int, n_t: int, lam: float,
                      global_B: int, global_b: int, out_host: torch.Tensor, device=None) -> torch.Tensor:
  """The same with HOST weights in and HOST [gradient | loss] out (transfers and a stream synchronisation inside).
  The per-(flow shape, device, stream) set-up (descriptor, persistent workspace) is cached: a call is one ctypes call."""
  for name, t in (("weights", weights_host), ("out", out_host)):
    if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
      raise _lib.CnfotError(f"{name}: expected a contiguous float32 host tensor")
  index = torch.cuda.current_device() if device is None else torch.device(device).index
  if index is None:
    index = torch.cuda.current_device()
  stream = torch.cuda.current_stream(index).cuda_stream
  ck = (shape, index, stream)
  ent = _rng_host_cache.get(ck)
  if ent is None:
    lib = _lib.load()
    desc = _lib.flow_desc(shape)
    nbytes = lib.cnfot_mfc_step_rng_host_workspace_bytes(desc)
    if nbytes < 0:
      _lib.check(1)
    dev = torch.device("cuda", index)
    with torch.cuda.device(index):
      ws = _step_workspace(shape, desc, nbytes, dev)   # persistent: no memset between two calls
    ent = (lib, desc, ws, ws.data_ptr(), ws.numel())
    _rng_host_cache[ck] = ent
  lib, desc, ws, ws_ptr, ws_bytes = ent
  args = (stream, desc, problem, weights_host.data_ptr(), int(key) & (2**64 - 1), int(step) & 0xFFFFFFFF, int(n_t), 0,
          global_B, 0, global_b, global_B, global_b, float(lam), out_host.data_ptr(), ws_ptr, ws_bytes)
  if torch.cuda.current_device() == index:
    rc = lib.cnfot_mfc_step_rng_host(*args)
  else:
    with torch.cuda.device(index):
      rc = lib.cnfot_mfc_step_rng_host(*args)
  _lib.check(rc)
  return out_host


def fused_update_supported(shape: FlowShape) -> bool:
  """True when the fused per-row step kernel (on-chip draws, device-resident update) covers this flow shape;
  False for the wide-conditioner engine."""
  return _lib.load().cnfot_train_state_bytes(_lib.flow_desc(shape)) >= 0


class TrainState:
  """Device-resident state of the fused update (cnfot_mfc_update): key, step count, all-reduce epoch and the step
  kernel's self-cleaning reduction buffers, plus the optax.adam moments (solvers.py:55-56)."""

  def __init__(self, shape: FlowShape, params_blob: torch.Tensor, key: int, step: int = 0, peers=None):
    lib = _lib.load()
    self.shape, self.device = shape, params_blob.device
    self.desc = _lib.flow_desc(shape)
    n = lib.cnfot_train_state_bytes(self.desc)
    if n < 0:
      _lib.check(1)
    self.buf = torch.empty(n, dtype=torch.uint8, device=self.device)
    self.mu = torch.zeros_like(params_blob)
    self.nu = torch.zeros_like(params_blob)
    self.key = int(key) & (2**64 - 1)
    self.peers = peers
    self._peer_desc = None
    epoch0 = 1
    if peers is not None:
      # the state's device-side epoch continues the exchange's host-side count (mfc_update keeps both in step)
      self._peer_desc = peers.peek_desc(shape)
      epoch0 = self._peer_desc.epoch
    with torch.cuda.device(self.device):
      _lib.check(lib.cnfot_train_state_init(_stream(), self.desc, self.buf.data_ptr(), self.buf.numel(), self.key,
                                            int(step), epoch0))
    self.steps_issued = int(step)

  def step_count(self) -> int:
    """Updates completed so far (reads the device counter: synchronises)."""
    return int(self.buf[128 + 8:128 + 16].view(torch.int64)[0])

  def status(self) -> int:
    """0 ok; 1: a peer never arrived in the all-reduce (results are NaN from then on)."""
    return int(self.buf[:64].view(torch.int32)[_lib.STATUS_WORD])


def mfc_update(shape: FlowShape, problem: _lib.ProblemDesc, state: TrainState, weights: torch.Tensor, n_t: int, lam: float,
               global_B: int, global_b: int, lr: float, rows_B=None, rows_b=None, out: Optional[torch.Tensor] = None,
               loss_hist: Optional[torch.Tensor] = None, b1=0.9, b2=0.999, eps=1e-8) -> None:
  """One `update` (solvers.py:90-97): value_and_grad on on-chip draws + all-reduce + Adam in ONE kernel launch.
  Nothing host-side changes between calls, so a run of calls can be captured in a CUDA graph and replayed."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  rB = slice(0, global_B) if rows_B is None else rows_B
  rb = slice(0, global_b) if rows_b is None else rows_b
  adam = _lib.AdamDesc(float(lr), float(b1), float(b2), float(eps))
  pd = state._peer_desc
  with torch.cuda.device(weights.device):
    _lib.check(lib.cnfot_mfc_update(_stream(), state.desc, problem, state.buf.data_ptr(), state.buf.numel(),
                                    _ptr(weights), _ptr(state.mu), _ptr(state.nu), ctypes.byref(adam), int(n_t),
                                    rB.start, rB.stop - rB.start, rb.start, rb.stop - rb.start, global_B, global_b,
                                    float(lam), _ptr(out), _ptr(loss_hist), 0 if loss_hist is None else loss_hist.numel(),
                                    None if pd is None else ctypes.byref(pd)))
  state.steps_issued += 1
  if state.peers is not None:
    state.peers.epoch += 1   # keep the host-side epoch of the exchange in step with the device-side one


def kinetic_energy(shape: FlowShape, weights, latent, t_values: Sequence[float], dt: float = 0.01,
                   with_score: bool = False, kappa: float = 0.0, dx: float = 0.01,
                   latent_blocks: int = 1) -> torch.Tensor:
  """(1/n_t) sum_t mean(v_t^2)/2 * dim over a time grid in ONE forward-only kernel
  (utils.calc_kinetic_energy / calc_score_kinetic_energy, cnf_ot/utils.py:311-389).
  latent: (latent_blocks * batch, D); time i uses block i % latent_blocks.  Returns a 0-d float64
  CUDA tensor."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  latent = _dev(latent, "latent").reshape(-1, shape.dim)
  if latent.shape[0] % latent_blocks:
    raise _lib.CnfotError("latent rows must be a multiple of latent_blocks")
  batch = latent.shape[0] // latent_blocks
  tb = torch.as_tensor(list(t_values), dtype=torch.float32)
  out = torch.empty(1, dtype=torch.float64, device=weights.device)
  desc = _lib.flow_desc(shape)
  ws = _workspace(lib.cnfot_kinetic_energy_workspace_bytes(desc, tb.numel()), weights.device)
  with torch.cuda.device(weights.device):
    _lib.check(lib.cnfot_kinetic_energy(_stream(), desc, _ptr(weights), _ptr(latent), batch, latent_blocks,
                                        tb.data_ptr(), tb.numel(), float(dt), int(with_score), float(kappa),
                                        float(dx), _ptr(out), ws.data_ptr(), ws.numel()))
  return out[0]


def density_grid(shape: FlowShape, weights, t_values: Sequence[float], domain, nx: int, ny: int, ref=None,
                 want_density: bool = True):
  """exp(log_prob) on the grid hstack(meshgrid(linspace(x0, x1, nx), linspace(y0, y1, ny))) for every time of `t_values`
  in ONE kernel launch (cnfot_density_grid; wide flows: one flow pass per row chunk).  domain = (x0, x1, y0, y1).  ref = (mix, var0, var1): also the sum of squared
  errors against (1 - mix) N(0, var0 I) + mix N(0, var1 I).  Returns (density (n_t, ny, nx) or None, sq_err 0-d float64 or None)."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  tb = torch.as_tensor(list(t_values), dtype=torch.float32)
  dens = torch.empty(tb.numel(), ny, nx, dtype=torch.float32, device=weights.device) if want_density else None
  sq = torch.zeros(1, dtype=torch.float64, device=weights.device) if ref is not None else None
  mix, v0, v1 = (0.0, 1.0, 1.0) if ref is None else ref
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_density_workspace_bytes(desc, tb.numel())
  if nbytes < 0:
    _lib.check(1)
  ws = _workspace(nbytes, weights.device)
  x0, x1, y0, y1 = (float(v) for v in domain)
  with torch.cuda.device(weights.device):
    _lib.check(lib.cnfot_density_grid(_stream(), desc, _ptr(weights), tb.data_ptr(), tb.numel(), x0, x1, y0, y1, int(nx), int(ny),
                                      _ptr(dens), int(ref is not None), float(mix), float(v0), float(v1), _ptr(sq),
                                      ws.data_ptr(), ws.numel()))
  return dens, (None if sq is None else sq[0])


def density_mc(shape: FlowShape, weights, cond: float, key: int, n: int, ref=None, want_samples: bool = False,
               want_density: bool = False, step: int = 0):
  """sample_and_log_prob at time `cond` for the NORMAL (n, dim) latent draw of (key, step), made on chip
  (cnfot_density_mc).  Returns (samples or None, density = exp(log_prob) or None, sq_err or None); see density_grid."""
  lib = _lib.load()
  weights = _dev(weights, "weights")
  dev = weights.device
  smp = torch.empty(n, shape.dim, dtype=torch.float32, device=dev) if want_samples else None
  dens = torch.empty(n, dtype=torch.float32, device=dev) if want_density else None
  sq = torch.zeros(1, dtype=torch.float64, device=dev) if ref is not None else None
  mix, v0, v1 = (0.0, 1.0, 1.0) if ref is None else ref
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_density_workspace_bytes(desc, 0)
  if nbytes < 0:
    _lib.check(1)
  ws = _workspace(nbytes, dev)
  with torch.cuda.device(dev):
    _lib.check(lib.cnfot_density_mc(_stream(), desc, _ptr(weights), float(cond), int(key) & (2**64 - 1), int(step) & 0xFFFFFFFF,
                                    int(n), _ptr(smp), _ptr(dens), int(ref is not None), float(mix), float(v0), float(v1),
                                    _ptr(sq), ws.data_ptr(), ws.numel()))
  return smp, dens, (None if sq is None else sq[0])


class PreparedDense:
  """Weights of one dense layer in the tcgen05 kernels' tile order (hi / lo tf32 split)."""

  def __init__(self, W: torch.Tensor, transpose: bool = False):
    lib = _lib.load()
    W = _dev(W, "W")
    if W.dim() != 2:
      raise _lib.CnfotError("W must be a matrix")
    self.K, self.N = (W.shape[1], W.shape[0]) if transpose else (W.shape[0], W.shape[1])
    n = lib.cnfot_dense_prepared_floats(self.K, self.N)
    if n < 0:
      raise _lib.CnfotError("dense layers need both sizes to be multiples of 16")
    self.buf = torch.empty(n, dtype=torch.float32, device=W.device)
    with torch.cuda.device(W.device):
      _lib.check(lib.cnfot_dense_prepare(_stream(), _ptr(W), self.K, self.N, W.stride(0), int(transpose),
                                         _ptr(self.buf)))


_EPILOGUES = {"bias": 0, "bias_relu": 1, "relu_mask": 2, "none": 3}


def dense_forward(X, prepared: PreparedDense, bias=None, mask_src=None, epilogue: str = "bias", out=None):
  """Y = epilogue(X W + b) on tcgen05 (3xTF32): see include/cnfot.h, cnfot_dense_forward."""
  lib = _lib.load()
  X = _dev(X, "X")
  rows = X.shape[0]
  if X.dim() != 2 or X.shape[1] != prepared.K or X.stride(1) != 1:
    raise _lib.CnfotError("X must be (rows, K) with unit inner stride")
  bias = _dev(bias, "bias")
  mask_src = _dev(mask_src, "mask_src")
  if out is None:
    out = torch.empty(rows, prepared.N, dtype=torch.float32, device=X.device)
  with torch.cuda.device(X.device):
    _lib.check(lib.cnfot_dense_forward(_stream(), _ptr(X), rows, prepared.K, X.stride(0), _ptr(prepared.buf),
                                       prepared.N, _ptr(bias), _ptr(mask_src),
                                       0 if mask_src is None else mask_src.stride(0), _EPILOGUES[epilogue],
                                       _ptr(out), out.stride(0)))
  return out


def dense_wgrad(A, G, dW, db=None) -> None:
  """dW += A^T G, db += column sums of G (tcgen05, 3xTF32): see include/cnfot.h, cnfot_dense_wgrad.
  dW may be a strided view (rows contiguous) of a gradient blob."""
  lib = _lib.load()
  A, G = _dev(A, "A"), _dev(G, "G")
  if not dW.is_cuda or dW.dtype != torch.float32 or dW.stride(1) != 1:
    raise _lib.CnfotError("dW must be a CUDA float32 matrix with unit inner stride")
  if A.shape[0] != G.shape[0] or dW.shape != (A.shape[1], G.shape[1]):
    raise _lib.CnfotError("dense_wgrad: shape mismatch")
  with torch.cuda.device(A.device):
    _lib.check(lib.cnfot_dense_wgrad(_stream(), _ptr(A), A.stride(0), _ptr(G), G.stride(0), A.shape[0], A.shape[1],
                                     G.shape[1], _ptr(dW), dW.stride(0), _ptr(db)))


def mask_tail(y: torch.Tensor, sub_dim: int) -> torch.Tensor:
  """y[:, sub_dim:] = 0 in place (cnf_ot/dr/trainers.py:95,108)."""
  lib = _lib.load()
  y = _dev(y, "y")
  with torch.cuda.device(y.device):
    _lib.check(lib.cnfot_mask_tail(_stream(), _ptr(y), y.shape[0], y.shape[1], int(sub_dim)))
  return y


def recon_head(x: torch.Tensor, xr: torch.Tensor, global_rows: int):
  """(loss contribution, g_xr) of mean_rows sum_dims (x - xr)^2 over this shard (trainers.py:97,110);
  the loss is a 0-d float64 CUDA tensor."""
  lib = _lib.load()
  x, xr = _dev(x, "x"), _dev(xr, "xr")
  g = torch.empty_like(xr)
  loss = torch.zeros(1, dtype=torch.float64, device=x.device)
  with torch.cuda.device(x.device):
    _lib.check(lib.cnfot_recon_head(_stream(), _ptr(x), _ptr(xr), x.shape[0], x.shape[1], 1.0 / float(global_rows),
                                    _ptr(g), _ptr(loss)))
  return loss[0], g


def adam_update(params, grads, m, v, lr, step, b1=0.9, b2=0.999, eps=1e-8) -> None:
  """In-place optax.adam(lr) update of the parameter blob."""
  lib = _lib.load()
  params, grads, m, v = (_dev(t, n) for t, n in ((params, "params"), (grads, "grads"), (m, "m"), (v, "v")))
  with torch.cuda.device(params.device):
    _lib.check(lib.cnfot_adam_update(_stream(), _ptr(params), _ptr(grads), _ptr(m), _ptr(v),
                                     params.numel(), lr, b1, b2, eps, step))
