"""GPU: on-chip draws and the device-resident update on the wide-conditioner engine (cnfot_mfc_step_rng and
cnfot_mfc_update for flows of csrc/wide.cu): the same numbers as the explicit-row step on the arrays of
cnfot_philox_rows / _times_host, the same trajectory as the fused update and as the float64 oracle + Adam, CUDA-graph
replay, solvers.main on a wide flow, and the calls the engine refuses."""
import ctypes

import pytest
import torch

from cnf_ot_b200 import _lib, ops, solvers
from cnf_ot_b200.layout import pack, unpack
from oracle import losses as olosses
from util import make_cfg, make_params, shape_of

pytestmark = pytest.mark.gpu


@pytest.fixture
def wide(monkeypatch):
  """Small hidden-64 flows also fit the fused kernels: run them on the wide engine."""
  monkeypatch.setenv("CNFOT_ENGINE", "wide")


def _explicit_inputs(cfg, shape, key, step, B, rows_B=None, rows_b=None):
  """The arrays of the draws of (key, step) that the step with on-chip draws generates itself."""
  b, D = B // 32, shape.dim
  typ = cfg["general"]["type"]
  horizon = 1.0 if typ == "ot" else float(cfg[typ]["T"])
  inp = {"t_batch": ops.philox_times(key, step, cfg["general"]["t_batch_size"], horizon),
         "latent_sub": ops.philox_rows(key, step, _lib.ROWS_NORMAL, b, D, "cuda", rows=rows_b)}
  if typ == "ot":
    inp["src"] = ops.philox_rows(key, step, _lib.ROWS_OT_SOURCE, B, D, "cuda", rows=rows_B)
    inp["tgt"] = ops.philox_rows(key, step, _lib.ROWS_NORMAL, B, D, "cuda", rows=rows_B)
  else:
    inp["latent"] = ops.philox_rows(key, step, _lib.ROWS_NORMAL, B, D, "cuda", rows=rows_B)
  return inp


def _explicit_step(cfg, shape, pd, W, key, step, lam, B, rows_B=None, rows_b=None):
  inp = _explicit_inputs(cfg, shape, key, step, B, rows_B, rows_b)
  return ops.mfc_step(shape, pd, W, inp.get("latent"), inp["latent_sub"], inp.get("src"), inp.get("tgt"), inp["t_batch"],
                      lam, B, B // 32).clone()


def _rel(a, b):
  return float((a - b).abs().max() / b.abs().max())


def _loss_rel(h, h_ref):
  return float(((h - h_ref).abs() / h_ref.abs()).max())


def _norm_rel(w, w_ref):
  return float((w - w_ref).norm() / w_ref.norm())


CASES = [("ot", "obstacle", 3), ("rwpo", "double_well", 3), ("fp", "nongradient", 4)]


@pytest.mark.parametrize("typ,sub,D", CASES)
def test_on_chip_draws_equal_the_step_on_exported_arrays(typ, sub, D, wide):
  B, lam = 1024, 100.0
  cfg = make_cfg(typ, sub, dim=D, H=64, Tn=2, lam=lam, B=B)
  shape = shape_of(cfg)
  _, params = make_params(cfg, 0.05)
  W = pack(shape, params).cuda()
  pd = ops.problem_desc(cfg)
  key = 0xABCDEF0123456789
  for step in (0, 17):
    a = _explicit_step(cfg, shape, pd, W, key, step, lam, B)
    r = ops.mfc_step_rng(shape, pd, W, key, step, 2, lam, B, B // 32).clone()
    assert _lib.last_launch_variant()["plan"] == "wide"
    # same kernels on the same numbers: only the order of the red.global additions differs
    assert _rel(r, a) < 1e-6, (step, _rel(r, a))
  # a shard draws the rows of its GLOBAL indices: each shard equals the explicit step on its slice, the shards add up
  b = B // 32
  parts = []
  for i in range(3):
    rB, rb = slice(i * B // 3, (i + 1) * B // 3), slice(i * b // 3, (i + 1) * b // 3)
    p = ops.mfc_step_rng(shape, pd, W, key, 17, 2, lam, B, b, rows_B=rB, rows_b=rb).clone()
    assert _rel(p, _explicit_step(cfg, shape, pd, W, key, 17, lam, B, rB, rb)) < 1e-6
    parts.append(p)
  assert _rel(sum(parts), a) < 2e-6


@pytest.mark.parametrize("typ,sub", [("ot", "obstacle"), ("rwpo", "double_well")])
def test_on_chip_draws_in_unstacked_chunks(typ, sub, wide, monkeypatch):
  """Chunks of 128 rows: the kinetic sub-batch (256 rows) is too large for the stacked passes, so run_step takes one
  pass per chunk (kinetic_chunk) over two chunks, with the score passes of rwpo starting from the state r(t)."""
  monkeypatch.setenv("CNFOT_WIDE_CHUNK", "128")
  B, lam = 8192, 100.0
  cfg = make_cfg(typ, sub, dim=3, H=64, Tn=2, lam=lam, B=B)
  shape = shape_of(cfg)
  _, params = make_params(cfg, 0.05)
  W = pack(shape, params).cuda()
  pd = ops.problem_desc(cfg)
  key = 0x0123456789ABCDEF
  a = _explicit_step(cfg, shape, pd, W, key, 5, lam, B)
  r = ops.mfc_step_rng(shape, pd, W, key, 5, 2, lam, B, B // 32).clone()
  assert _rel(r, a) < 1e-6, _rel(r, a)


def _run_updates(shape, pd, W, key, steps, lam, lr, B, n_t=1):
  state = ops.TrainState(shape, W, key, rows_B=B, rows_b=B // 32)
  hist = torch.zeros(steps, device="cuda")
  for _ in range(steps):
    ops.mfc_update(shape, pd, state, W, n_t, lam, B, B // 32, lr, loss_hist=hist)
  return state, hist


def test_wide_engine_follows_the_fused_engine(monkeypatch):
  """The mfc.yaml flow (hidden 16) is covered by both engines: the same key gives the same step, and 20
  device-resident updates from the same state the same trajectory."""
  B, lam, lr, steps = 2048, 50.0, 2e-3, 20
  cfg = make_cfg("ot", "free", B=B, lam=lam)
  shape = shape_of(cfg)
  _, params = make_params(cfg, 0.3)
  pd = ops.problem_desc(cfg)
  key = 0x5EED5EED5EED
  W0 = pack(shape, params).cuda()
  f = ops.mfc_step_rng(shape, pd, W0, key, 3, 1, lam, B, B // 32).clone()
  assert _lib.last_launch_variant()["plan"] != "wide"
  Wf = W0.clone()
  sf, hf = _run_updates(shape, pd, Wf, key, steps, lam, lr, B)
  monkeypatch.setenv("CNFOT_ENGINE", "wide")
  w = ops.mfc_step_rng(shape, pd, W0, key, 3, 1, lam, B, B // 32).clone()
  assert _lib.last_launch_variant()["plan"] == "wide"
  n = shape.blob_size
  assert abs(float(w[n]) - float(f[n])) <= 2e-5 * abs(float(f[n]))
  assert _rel(w[:n], f[:n]) <= 5e-5
  Ww = W0.clone()
  sw, hw = _run_updates(shape, pd, Ww, key, steps, lam, lr, B)
  assert sf.step_count() == sw.step_count() == steps and sw.status() == 0
  rel = (hw.double() - hf.double()).abs() / hf.double().abs()
  dw = (Ww.double() - Wf.double()).abs()
  moved = float((Wf.double() - W0.double()).abs().max())
  assert float(rel[:5].max()) < 5e-5 and float(rel.max()) < 5e-2, rel
  assert float(dw.median()) < 0.01 * moved and float(dw.quantile(0.99)) < 0.2 * moved, (float(dw.quantile(0.99)), moved)


def _oracle_adam_trajectory(cfg, shape, spec, params0, key, steps, lam, lr, B):
  """oracle value_and_grad (float64) + optax-style Adam in float64 on the exported draws of (key, step k)."""
  blob = pack(shape, params0, torch.float64)
  m, v = torch.zeros_like(blob), torch.zeros_like(blob)
  losses = []
  for k in range(steps):
    inp = _explicit_inputs(cfg, shape, key, k, B)
    o_in = {kk: (vv.double().cpu() if torch.is_tensor(vv) else torch.tensor(vv, dtype=torch.float64)) for kk, vv in inp.items()}
    if "latent" not in o_in:
      o_in["latent"] = o_in["latent_sub"]
    p = unpack(shape, blob, params0)
    p = {mod: {n: t.double() for n, t in lv.items()} for mod, lv in p.items()}
    loss, grads = olosses.value_and_grad(cfg, spec, p, o_in, lam)
    g = pack(shape, grads, torch.float64)
    losses.append(float(loss))
    m = 0.9 * m + 0.1 * g
    v = 0.999 * v + 0.001 * g * g
    mh, vh = m / (1 - 0.9**(k + 1)), v / (1 - 0.999**(k + 1))
    blob = blob - lr * mh / (vh.sqrt() + 1e-8)
  return torch.tensor(losses, dtype=torch.float64), blob


@pytest.mark.parametrize("typ,sub", [("ot", "obstacle"), ("rwpo", "double_well")])
def test_wide_updates_follow_the_oracle_adam_trajectory(typ, sub, wide):
  # lr 1e-3: at 2e-3 these hidden-64 trajectories leave the float64 one after ~10 updates on the fused engine just as
  # on the wide one (ot/obstacle: both 19 % loss difference at update 20), which says nothing about either engine
  steps, B, lam, lr = 20, 1024, 50.0, 1e-3
  cfg = make_cfg(typ, sub, dim=2, H=64, Tn=1, lam=lam, B=B)
  shape = shape_of(cfg)
  spec, params = make_params(cfg, 0.1)
  W = pack(shape, params).cuda()
  pd = ops.problem_desc(cfg)
  key = 0x5EED5EED5EED
  state, hist = _run_updates(shape, pd, W, key, steps, lam, lr, B)
  assert _lib.last_launch_variant()["plan"] == "wide"
  assert state.step_count() == steps and state.status() == 0
  l_or, w_or = _oracle_adam_trajectory(cfg, shape, spec, params, key, steps, lam, lr, B)
  rel = (hist.cpu().double() - l_or).abs() / l_or.abs()
  dw = (W.cpu().double() - w_or).abs()
  moved = float((w_or - pack(shape, params, torch.float64)).abs().max())
  print(f"loss rel err: first 5 {float(rel[:5].max()):.2e}, all {float(rel.max()):.2e}; weights moved {moved:.3e}, "
        f"|dw| median {float(dw.median()):.2e} q99 {float(dw.quantile(0.99)):.2e}")
  assert float(rel[:5].max()) < 5e-5, rel[:5]
  assert float(rel.max()) < 5e-2, float(rel.max())
  assert float(dw.median()) < 0.01 * moved and float(dw.quantile(0.99)) < 0.2 * moved, (float(dw.quantile(0.99)), moved)


def test_graph_replays_are_new_updates(wide):
  """One eager update, K = 4 updates captured, the graph replayed twice == nine eager updates: the device-side step
  counter selects draws, Adam's bias correction and the loss slot, so a replay is never a repeat."""
  # lr 1e-3, as in the oracle test: this flow amplifies float32 differences quickly at larger steps
  B, lam, lr = 2048, 50.0, 1e-3
  cfg = make_cfg("ot", "obstacle", dim=2, H=64, lam=lam, B=B)
  shape = shape_of(cfg)
  _, params = make_params(cfg, 0.1)
  pd = ops.problem_desc(cfg)

  def run(graphed):
    W = pack(shape, params).cuda()
    state = ops.TrainState(shape, W, 77, rows_B=B, rows_b=B // 32)
    hist = torch.zeros(9, device="cuda")
    one = lambda: ops.mfc_update(shape, pd, state, W, 1, lam, B, B // 32, lr, loss_hist=hist)
    if graphed:
      one()
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g):
        for _ in range(4):
          one()
      g.replay()
      g.replay()
    else:
      for _ in range(9):
        one()
    torch.cuda.synchronize()
    return state.step_count(), hist.cpu().double(), W.cpu().double()

  n0, h0, w0 = run(False)
  n1, h1, w1 = run(True)
  assert n0 == n1 == 9
  assert bool(torch.isfinite(h1).all()) and len(set(h1.tolist())) == 9
  # The engine sums gradients with red.global, so two EAGER runs already differ in the last bits, and Adam carries
  # that into the weights (measured on B200: ~3e-7 of the loss, ~4e-7 of |w| in norm after nine updates).  The
  # replayed run must be within 1e-6 relative, or as close to the eager run as a second eager run is.
  _, h2, w2 = run(False)
  for name, d, d_eager in (("loss", _loss_rel(h1, h0), _loss_rel(h2, h0)), ("weights", _norm_rel(w1, w0), _norm_rel(w2, w0))):
    assert d <= max(1e-6, 4 * d_eager), (name, d, d_eager)


def test_main_trains_a_wide_flow_device_resident(tmp_path, wide):
  cfg = make_cfg("ot", "obstacle", dim=2, H=64, B=2048, lam=50.0)
  cfg["train"].update(epochs=30, lr=1e-3, eval_frequency=10)
  p, hist = solvers.main(cfg)
  assert _lib.last_launch_variant()["plan"] == "wide"
  h = torch.stack(hist).cpu().double()
  assert h.shape == (30, ) and bool(torch.isfinite(h).all())
  assert float(h[-5:].mean()) < float(h[:5].mean())
  # 15 epochs, checkpoint, 15 more from the checkpoint == 30 in one run (same train key, same step counter)
  path = str(tmp_path / "half.npz")
  c1 = make_cfg("ot", "obstacle", dim=2, H=64, B=2048, lam=50.0)
  c1["train"].update(epochs=15, lr=1e-3, eval_frequency=10, params_out=path)
  solvers.main(c1)
  c2 = make_cfg("ot", "obstacle", dim=2, H=64, B=2048, lam=50.0)
  c2["train"].update(epochs=15, lr=1e-3, eval_frequency=10, params_in=path)
  p2, hist2 = solvers.main(c2)
  h2 = torch.stack(hist2).cpu().double()
  # up to float32 reordering: a second uninterrupted run differs from the first by the red.global order of 30 steps
  # (measured on B200: ~4e-5 of the loss, ~2e-4 of max|w|); the resumed run must be no further away than that
  p3, hist3 = solvers.main(cfg)
  h3 = torch.stack(hist3).cpu().double()
  for name, d, d_again in (("loss", _loss_rel(h2, h[15:]), _loss_rel(h3, h)),
                           ("weights", _norm_rel(p2.blob, p.blob), _norm_rel(p3.blob, p.blob))):
    assert d <= max(2e-4, 4 * d_again), (name, d, d_again)


def test_wide_refusals(wide):
  cfg = make_cfg("ot", "obstacle", dim=2, H=64, B=1024, lam=50.0)
  shape = shape_of(cfg)
  _, params = make_params(cfg, 0.1)
  W = pack(shape, params).cuda()
  pd = ops.problem_desc(cfg)
  lib = _lib.load()
  desc = _lib.flow_desc(shape)
  assert lib.cnfot_train_state_bytes(desc) == -1
  assert lib.cnfot_train_state_bytes_rows(desc, 1024, 32) > 0
  peers = _lib.PeerDesc()
  peers.rank, peers.world, peers.epoch = 0, 2, 1
  out = torch.empty(shape.blob_size + 8, device="cuda")
  ws = torch.empty(lib.cnfot_mfc_step_workspace_bytes(desc, 1024, 32, 1), dtype=torch.uint8, device="cuda")
  with pytest.raises(_lib.CnfotError, match="all-reduce"):
    _lib.check(lib.cnfot_mfc_step_rng(ops._stream(), desc, pd, W.data_ptr(), 1, 0, 1, 0, 1024, 0, 32, 1024, 32, 50.0,
                                      out.data_ptr(), ws.data_ptr(), ws.numel(), ctypes.byref(peers)))
  state = ops.TrainState(shape, W, 1, rows_B=1024, rows_b=32)
  adam = _lib.AdamDesc(1e-3, 0.9, 0.999, 1e-8)
  with pytest.raises(_lib.CnfotError, match="all-reduce"):
    _lib.check(lib.cnfot_mfc_update(ops._stream(), desc, pd, state.buf.data_ptr(), state.buf.numel(), W.data_ptr(),
                                    state.mu.data_ptr(), state.nu.data_ptr(), ctypes.byref(adam), 1, 0, 1024, 0, 32, 1024,
                                    32, 50.0, None, None, 0, ctypes.byref(peers)))
  small = ops.TrainState(shape, W, 1, rows_B=256, rows_b=8)
  with pytest.raises(_lib.CnfotError, match="train state too small"):
    ops.mfc_update(shape, pd, small, W, 1, 50.0, 1024, 32, 1e-3)
  assert small.step_count() == 0
  with pytest.raises(_lib.CnfotError):
    ops.mfc_step_rng_host(shape, pd, W.cpu(), 1, 0, 1, 50.0, 1024, 32, torch.empty(shape.blob_size + 8))
