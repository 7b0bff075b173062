"""Densities on grids / at Monte-Carlo samples (cnfot_density_grid / cnfot_density_mc) on the wide-conditioner engine
(cnf_ot_b200/csrc/wide.cu: wide_density_grid / wide_density_mc): the reference fixture of test_density.py with the
engine forced, flows only the wide engine covers against the oracle, chunking, and the edges of the C ABI."""
import numpy as np
import pytest
import torch

from cnf_ot_b200 import _lib, ops, random, utils
from cnf_ot_b200._lib import CnfotError
from cnf_ot_b200.layout import pack
from oracle import density as odens
from test_density import _load
from util import make_cfg, make_params, shape_of

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _force_wide_engine(monkeypatch):
  """Shapes both engines cover (the fixture's hidden 16) must run on the wide engine here."""
  monkeypatch.setenv("CNFOT_ENGINE", "wide")


def close(a, b, tol):
  """test_density.py's measure: max |a - b| / (|b| + 1e-2)."""
  return float(((a.double().cpu() - b).abs() / (b.abs() + 1e-2)).max()) < tol


def test_reference_fixture_on_the_wide_engine():
  """test_density.py::test_gpu_density_grid_and_mc_match_the_reference, same fixture and tolerances."""
  from cnf_ot_b200.flows import FlowModel, ParamTree
  g, shape, spec, params = _load()
  k = int(g["stride"])
  model = FlowModel(shape, "cuda")
  P = ParamTree(shape, g["blob"].float().cuda())
  snap = utils.plot_density_snapshot(model.apply.log_prob, P)
  assert _lib.last_launch_info()["engine"] == "wide"
  assert snap.shape == (10, 100, 100) and close(snap[:, ::k, ::k], g["snap_sub"], 2e-5)
  assert float(((snap.double().sum((1, 2)).cpu() - g["snap_sum"]) / g["snap_sum"]).abs().max()) < 1e-5
  dens2 = utils.density_on_grid(model.apply.log_prob, P, g["t_traj"].tolist(), g["domain2"].tolist(), 100)
  assert close(dens2[:, ::k, ::k], g["dens2_sub"], 2e-5)
  XY = odens.grid_points([-6, 6, -6, 6], 100, 100).float().cuda()
  lp = model.apply.log_prob(P, XY, cond=torch.tensor([float(np.linspace(0, 1, 10)[3])]))
  assert float((torch.exp(lp).reshape(100, 100) - snap[3]).abs().max()) < 2e-6
  a, T = float(g["fp_a"]), float(g["fp_T"])
  rg = float(utils.rmse_grid_loss_fn(model.apply.log_prob, P, 1.0, int(g["grid_size"]), a=a, T=T))
  assert _lib.last_launch_info()["engine"] == "wide"
  assert abs(rg - float(g["rmse_grid"])) < 2e-5 * float(g["rmse_grid"])
  key = random.PRNGKey(11)
  n = 50000
  rm = float(utils.rmse_mc_loss_fn(model, P, 1.0, key, n, a=a, T=T))
  assert _lib.last_launch_info()["engine"] == "wide"
  lat = ops.philox_rows(key.value, 0, _lib.ROWS_NORMAL, n, 2, "cuda").double().cpu()
  with torch.no_grad():
    want = float(odens.rmse_mc(spec, params, 1.0, lat, a, T))
  assert abs(rm - want) < 2e-5 * want
  smp, dens, _ = ops.density_mc(shape, P.blob, 1.0, key.value, 4096, want_samples=True, want_density=True)
  y, lp = model.apply.sample_and_log_prob(P, cond=torch.ones(4096, 1, device="cuda"), seed=key, sample_shape=(4096, ))
  assert float((smp - y).abs().max()) < 1e-5 and float((dens - torch.exp(lp)).abs().max()) < 1e-6


# (D, L, M, H, sigma): flows the fused kernels do not cover (hidden 128, hidden 48); sigma as in test_gpu_wide.py
WIDE_ONLY = [(2, 2, 2, 128, 0.02), (2, 2, 3, 48, 0.1)]


def _flow(D, L, M, H, sigma):
  cfg = make_cfg(dim=D, L=L, M=M, H=H)
  shape = shape_of(cfg)
  spec, params = make_params(cfg, sigma)
  return shape, spec, params, pack(shape, params).cuda()


@pytest.mark.parametrize("D,L,M,H,sigma", WIDE_ONLY)
def test_grid_matches_the_oracle_and_chunks_agree(D, L, M, H, sigma, monkeypatch):
  shape, spec, params, W = _flow(D, L, M, H, sigma)
  ts, dom, n = [0.0, 0.45, 1.0], [-4.0, 4.0, -4.0, 4.0], 60
  with torch.no_grad():
    want = odens.density_on_grid(spec, params, ts, dom, n)
    want_rg = float(odens.rmse_grid(spec, params, 1.0, 150, 1.0, 1.0))
  v0, v1 = utils._fp_reference_variances(1.0, 1.0)

  def run():
    dens, _ = ops.density_grid(shape, W, ts, dom, n, n)
    assert _lib.last_launch_info()["engine"] == "wide"
    _, sq = ops.density_grid(shape, W, [1.0], [-5, 5, -5, 5], 150, 150, ref=(1.0, v0, v1), want_density=False)
    return dens, float(torch.sqrt(sq / (150 * 150)))

  dens, rg = run()
  assert dens.shape == (3, n, n) and close(dens, want, 2e-5)
  assert abs(rg - want_rg) < 2e-5 * want_rg
  # 1024-row chunks: chunks cross the time boundaries (3600 points per time) and the last one is partial
  monkeypatch.setenv("CNFOT_WIDE_CHUNK", "1024")
  dens_c, rg_c = run()
  assert float((dens_c - dens).abs().max()) <= 1e-6
  assert abs(rg_c - rg) <= 1e-6 * rg


@pytest.mark.parametrize("D,L,M,H,sigma", [WIDE_ONLY[0], (5, 3, 1, 128, 0.01)])
def test_monte_carlo_matches_the_model_api_and_the_oracle(D, L, M, H, sigma):
  from cnf_ot_b200.flows import FlowModel, ParamTree
  shape, spec, params, W = _flow(D, L, M, H, sigma)
  model = FlowModel(shape, "cuda")
  P = ParamTree(shape, W)
  key, n, cond = random.PRNGKey(7), 50003, 0.7
  v0, v1 = utils._fp_reference_variances(1.0, 0.5)
  smp, dens, sq = ops.density_mc(shape, W, cond, key.value, n, ref=(cond, v0, v1), want_samples=True, want_density=True)
  assert _lib.last_launch_info()["engine"] == "wide"
  y, lp = model.apply.sample_and_log_prob(P, cond=torch.full((n, 1), cond, device="cuda"), seed=key, sample_shape=(n, ))
  assert float((smp - y).abs().max()) <= 1e-6 and float((dens - torch.exp(lp)).abs().max()) <= 1e-6
  # the error sum against the oracle on the exported latent rows
  lat = ops.philox_rows(key.value, 0, _lib.ROWS_NORMAL, n, D, "cuda").double().cpu()
  with torch.no_grad():
    want = float(odens.rmse_mc(spec, params, cond, lat, 1.0, 0.5))
  got = float(torch.sqrt(sq / n))
  assert abs(got - want) < 2e-5 * want
  # another step of the same key draws other rows
  smp2, _, _ = ops.density_mc(shape, W, cond, key.value, n, want_samples=True, step=1)
  assert float((smp2 - smp).abs().max()) > 0.1


def test_edges_of_the_c_abi():
  lib = _lib.load()
  shape, _, _, W = _flow(2, 2, 2, 128, 0.02)
  desc = _lib.flow_desc(shape)
  nbytes = lib.cnfot_density_workspace_bytes(desc, 1)
  assert nbytes >= 0 and lib.cnfot_density_workspace_bytes(desc, 0) >= 0
  ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
  stream = torch.cuda.current_stream().cuda_stream
  # n = 0: nothing to evaluate, the error sum is zero
  sq = torch.full((1, ), float("nan"), dtype=torch.float64, device="cuda")
  _lib.check(lib.cnfot_density_mc(stream, desc, W.data_ptr(), 1.0, 3, 0, 0, None, None, 1, 0.5, 1.0, 2.0, sq.data_ptr(),
                                  ws.data_ptr(), nbytes))
  torch.cuda.synchronize()
  assert float(sq[0]) == 0.0
  # a workspace one byte short
  t = torch.tensor([0.5], dtype=torch.float32)
  dens = torch.empty(4, 4, device="cuda")
  args = lambda nb: (stream, desc, W.data_ptr(), t.data_ptr(), 1, -1.0, 1.0, -1.0, 1.0, 4, 4, dens.data_ptr(), 0, 0.0, 1.0,
                     1.0, None, ws.data_ptr(), nb)
  with pytest.raises(CnfotError):
    _lib.check(lib.cnfot_density_grid(*args(nbytes - 1)))
  _lib.check(lib.cnfot_density_grid(*args(nbytes)))
  assert _lib.last_launch_info()["engine"] == "wide"
  assert bool(torch.isfinite(dens).all())
  # grids are two-dimensional
  shape3, _, _, W3 = _flow(3, 2, 2, 128, 0.02)
  with pytest.raises(CnfotError):
    ops.density_grid(shape3, W3, [0.5], [-1, 1, -1, 1], 8, 8)


@pytest.mark.parametrize("typ,sub", [("fp", "gradient"), ("rwpo", "double_well")])
def test_solver_evaluate_on_a_hidden_128_flow(typ, sub, monkeypatch):
  """config/mfc.yaml with cnf.hidden_size = 128: solvers.evaluate runs its whole tail on the wide engine."""
  from cnf_ot_b200 import solvers
  from cnf_ot_b200.flows import ParamTree
  monkeypatch.delenv("CNFOT_ENGINE")   # hidden 128 is wide-only: no override needed
  cfg = make_cfg(typ, sub, dim=2, H=128)
  model, _, _ = solvers.build(cfg)
  _, params = make_params(cfg, 0.02)
  P = ParamTree(model.shape, pack(model.shape, params).cuda())
  out = solvers.evaluate(cfg, model, P, random.PRNGKey(5), batch_size=512, t_size=4, verbose=False)
  assert _lib.last_launch_info()["engine"] == "wide"
  if typ == "fp":
    assert np.isfinite(out["rmse_mc"]) and np.isfinite(out["rmse_grid"])
    assert out["rmse_mc"] > 0 and out["rmse_grid"] > 0
  else:
    assert tuple(out["density_T"].shape) == (100, 100) and bool(torch.isfinite(out["density_T"]).all())
    assert float(out["density_T"].min()) >= 0 and float(out["density_T"].max()) > 0
