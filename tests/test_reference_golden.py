"""Reference-generated golden vectors (tests/golden/ref_*.npz).

They are outputs of the reference's OWN source files (`cnf_ot/models/{flows,autoregressive,conditional}.py`,
`cnf_ot/mfc/applications.py`, imported unmodified from /root/reference by tests/golden/make_reference_golden.py and
executed on torch-float64 stand-ins for jax / haiku / distrax, tests/golden/refshim.py): model built as
`solvers.py:41-54`, loss functions as `solvers.py:58-88`, called as `update` calls them (`solvers.py:94`).

CPU: the oracle (oracle/flow.py, oracle/losses.py) reproduces the reference's samples, log-probs, losses and
gradients to float64 rounding (values 1e-10, losses / gradients / energies 1e-12; the float32 `first` leaf 2e-6) -- this pins the restatement to the reference's code.
GPU (-m gpu): the CUDA path through the C ABI matches them at the float32 tolerances of the other parity tests
(values: 99 % within 2e-5, all within 2e-4; loss 2e-5 relative; gradient 5e-5 of the largest entry)."""
import os

import numpy as np
import pytest
import torch

from cnf_ot_b200.layout import FlowShape, pack, unpack
from oracle import flow as oflow
from oracle import losses as olosses
from util import make_cfg

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

STEPS = {
  "ref_step_ot_free_d2": ("ot", "free", {}),
  "ref_step_ot_obstacle_d2": ("ot", "obstacle", {}),
  "ref_step_rwpo_double_well_d2": ("rwpo", "double_well", {}),
  "ref_step_rwpo_quadratic_d3": ("rwpo", "quadratic", dict(dim=3)),
  "ref_step_fp_gradient_d2": ("fp", "gradient", {}),
  "ref_step_fp_nongradient_d2": ("fp", "nongradient", {}),
  "ref_step_fp_lorenz_d3": ("fp", "lorenz", dict(dim=3)),
  # other network shapes (taken from the fixture): hidden 64, 3 hidden layers, 3 flow layers, 8 bins x hidden 32
  "ref_step_ot_obstacle_d2_h64": ("ot", "obstacle", {}),
  "ref_step_rwpo_double_well_d2_m3": ("rwpo", "double_well", {}),
  "ref_step_fp_nongradient_d2_l3": ("fp", "nongradient", {}),
  "ref_step_ot_free_d2_k8_h32": ("ot", "free", {}),
}
FLOWS = ["ref_flow_d2", "ref_flow_d3_h8"]
ENERGIES = ["ref_energy_d2", "ref_energy_d3"]
DR = {"ref_dr_enc_dec_d4": "enc_dec", "ref_dr_dec_only_d4": "dec_only"}


def load(name):
  z = np.load(os.path.join(GOLD, name + ".npz"))
  return {k: torch.from_numpy(np.asarray(z[k])) for k in z.files}


def parts(g):
  D, L, M, H, K = (int(v) for v in g["shape"])
  shape = FlowShape(D, L, M, H, K)
  spec = olosses.spec_from_config(make_cfg(dim=D, L=L, M=M, H=H, K=K))
  params = unpack(shape, g["blob"])
  params["~"]["first"] = params["~"]["first"].float()   # float32 leaf in the reference (flows.py:47-55)
  return shape, spec, params


def step_cfg(name, g):
  typ, sub, kw = STEPS[name]
  D, L, M, H, K = (int(v) for v in g["shape"])
  return make_cfg(typ, sub, Tn=int(g["t_batch"].numel()), lam=float(g["lam"]), B=int(g["latent"].shape[0]),
                  L=L, M=M, H=H, K=K, **kw)


def close(a, b, tol=2e-5, tol_max=2e-4):
  a = a.detach().cpu().double().reshape(-1)
  b = b.detach().cpu().double().reshape(-1)
  e = (a - b).abs() / (b.abs() + 1.0)
  ok = float(e.quantile(0.99)) < tol and float(e.max()) < tol_max
  if not ok:
    print("reference golden mismatch: q99 %.3e max %.3e" % (float(e.quantile(0.99)), float(e.max())))
  return ok


# ------------------------------------------------------------------ CPU: oracle vs the reference's outputs
@pytest.mark.parametrize("name", FLOWS)
def test_oracle_flow_matches_reference(name):
  g = load(name)
  shape, spec, params = parts(g)
  n = g["latent"].shape[0]
  y, lp = oflow.sample_and_log_prob(spec, params, g["latent"], g["t"].reshape(-1, 1))
  assert float((y - g["sample_y"]).abs().max()) < 1e-10
  assert float((lp - g["sample_log_prob"]).abs().max()) < 1e-10
  c0 = torch.full((1, ), float(g["t0"]), dtype=torch.float64)
  assert float((oflow.log_prob(spec, params, g["x"], c0) - g["log_prob_x"]).abs().max()) < 1e-10
  cn = torch.full((n, 1), float(g["t0"]), dtype=torch.float64)
  # model.apply.forward = latent -> sample direction, model.apply.inverse = sample -> latent (flows.py:151,219-221)
  assert float((oflow.sample(spec, params, g["x"], cn) - g["forward_x"]).abs().max()) < 1e-10
  xi, _ = oflow.flow_inverse_and_log_det(spec, params, g["x"], cn)
  fw, _ = oflow.flow_forward_and_log_det(spec, params, g["x"], cn)
  lat = xi if float((xi - g["inverse_x"]).abs().max()) < float((fw - g["inverse_x"]).abs().max()) else fw
  assert float((lat - g["inverse_x"]).abs().max()) < 1e-10


def _ot_reverse_kl_oracle(spec, params, latent):
  """applications.py:91-126 restated on the oracle flow (targets N(3, I) at t = 0 and N(0, I) at t = 1)."""
  n, d = latent.shape
  tot = 0.0
  for cond, mean in ((0.0, 3.0), (1.0, 0.0)):
    y, lp = oflow.sample_and_log_prob(spec, params, latent, torch.full((n, 1), cond, dtype=torch.float64))
    tot = tot + (lp - (-0.5 * ((y - mean)**2).sum(-1) - 0.5 * d * np.log(2 * np.pi))).mean()
  return tot


@pytest.mark.parametrize("name", FLOWS)
def test_oracle_ot_reverse_kl_matches_reference(name):
  g = load(name)
  shape, spec, params = parts(g)
  got = _ot_reverse_kl_oracle(spec, params, g["latent"])
  assert abs(float(got) - float(g["ot_reverse_kl"])) <= 1e-12 * abs(float(g["ot_reverse_kl"]))


# a checkout of the original project (github.com/jiaxi98/cnf_ot); the two tests that read its source skip without one
REF_ROOT = os.environ.get("CNF_OT_REFERENCE", "")
REF = os.path.join(REF_ROOT, "cnf_ot")
NO_REF = "needs a checkout of the original cnf_ot project in CNF_OT_REFERENCE"


def _check_signatures(mod, sigs, only=None):
  """Each function of `sigs` (name -> parameter names) exists in `mod` with those parameters first, in that order;
  any further parameters are optional."""
  import inspect
  for name, args in sigs.items():
    if only is not None and name not in only:
      continue
    params = list(inspect.signature(getattr(mod, name)).parameters.values())
    assert [p.name for p in params[:len(args)]] == args, (mod.__name__, name, args, params)
    assert all(p.default is not inspect.Parameter.empty for p in params[len(args):]), (name, params[len(args):])


@pytest.mark.skipif(not REF_ROOT or not os.path.isdir(REF), reason=NO_REF)
def test_mirror_signatures_match_the_reference():
  """Every function of the reference's applications.py, the two energies of utils.py, RQSFlow and solvers.main exist in
  the mirror with the same parameter names in the same order (extra trailing optional parameters allowed)."""
  import ast
  import cnf_ot_b200.applications as A
  import cnf_ot_b200.flows as F
  import cnf_ot_b200.solvers as S
  import cnf_ot_b200.utils as U

  def ref_sigs(path):
    tree = ast.parse(open(path).read())
    return {n.name: [a.arg for a in n.args.args + n.args.kwonlyargs] for n in tree.body if isinstance(n, ast.FunctionDef)}
  _check_signatures(A, ref_sigs(REF + "/mfc/applications.py"))
  _check_signatures(U, ref_sigs(REF + "/utils.py"), {"calc_kinetic_energy", "calc_score_kinetic_energy"})
  _check_signatures(F, ref_sigs(REF + "/models/flows.py"), {"RQSFlow"})
  _check_signatures(S, ref_sigs(REF + "/mfc/solvers.py"), {"main"})


def test_mirror_signatures_match_the_stored_record():
  """The same API -- every public function of applications.py, the two energies of utils.py, RQSFlow, solvers.main --
  against tests/golden/mirror_signatures.json (tests/golden/make_golden.py), under the same rule.  The record holds
  the mirror's own signatures, not data read from the original project; it keeps the API from drifting where no checkout
  of the original is at hand."""
  import importlib
  import json
  with open(os.path.join(GOLD, "mirror_signatures.json")) as f:
    record = json.load(f)
  assert set(record) == {"cnf_ot_b200.applications", "cnf_ot_b200.utils", "cnf_ot_b200.flows", "cnf_ot_b200.solvers"}
  for mod_name, sigs in record.items():
    _check_signatures(importlib.import_module(mod_name), sigs)


@pytest.mark.skipif(not REF_ROOT or not os.path.isdir(REF), reason=NO_REF)
def test_reference_own_spline_test_passes_on_the_restated_spline():
  """The original project's tests/test_rqs_accuracy.py, executed UNMODIFIED against oracle/rqs.py behind the
  `distrax.RationalQuadraticSpline` interface (tests/golden/run_reference_tests.py; own process because the stand-ins
  register fake jax / distrax modules): round trips, log-det vs autodiff Jacobian, boundaries, all < 1e-12."""
  import subprocess
  import sys
  here = os.path.dirname(os.path.abspath(__file__))
  r = subprocess.run([sys.executable, os.path.join(here, "golden", "run_reference_tests.py")], capture_output=True,
                     text=True, timeout=600)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
  assert "PASSED " + os.path.join(REF_ROOT, "tests", "test_rqs_accuracy.py") + "::TestRQSAccuracy::test_rqs_comprehensive" in r.stdout


@pytest.mark.parametrize("name", list(STEPS))
def test_oracle_step_matches_reference(name):
  g = load(name)
  shape, spec, params = parts(g)
  assert int(g["n_params"]) == shape.param_count() == spec.param_count()   # leaves model.init created (solvers.py:54)
  cfg = step_cfg(name, g)
  inputs = {k: g[k] for k in ("latent", "src", "tgt", "t_batch")}
  loss, grads = olosses.value_and_grad(cfg, spec, params, inputs)
  assert abs(float(loss) - float(g["loss"])) <= 1e-12 * abs(float(g["loss"]))
  err = (pack(shape, grads, torch.float64) - g["grad"]).abs() / float(g["grad"].abs().max())
  # `first` is a float32 leaf in the reference (flows.py:47-55): its gradient is accumulated in float32 on both sides
  assert float(err[:shape.Pp].max()) <= 2e-6 and float(err[shape.Pp:].max()) <= 1e-12


@pytest.mark.parametrize("name", ENERGIES)
def test_oracle_energies_match_reference(name):
  """utils.calc_kinetic_energy / calc_score_kinetic_energy (cnf_ot/utils.py:311-389) run from the reference."""
  from oracle import energies as oen
  g = load(name)
  shape, spec, params = parts(g)
  n_t = int(g["t_size"])
  ts = np.linspace(0.0, 1.0, n_t).tolist()
  lat = g["latent"].unsqueeze(0).expand(n_t, *g["latent"].shape)
  e = oen.kinetic_energy(spec, params, lat, ts)
  assert abs(float(e) - float(g["e_kin"])) <= 1e-12 * abs(float(g["e_kin"]))
  ts = np.linspace(0.0, float(g["T"]), n_t).tolist()
  es = oen.score_kinetic_energy(spec, params, lat, ts, beta=float(g["beta"]))
  assert abs(float(es) - float(g["e_score"])) <= 1e-12 * abs(float(g["e_score"]))


@pytest.mark.parametrize("name", ["ref_rqs_symbolic_k5", "ref_rqs_symbolic_k8"])
def test_oracle_spline_matches_reference_symbolic_form(name):
  """In-bin map and derivative of the restated spline vs the reference's own symbolic statement
  (cnf_ot/models/nsf_symbol.py:3-10, lambdified with sympy by the generator)."""
  from oracle import rqs as orqs
  g = load(name)
  y, ld, b = orqs.rqs_forward(g["x"], g["theta"])
  assert torch.equal(b, g["bin"])
  assert float((y - g["y"]).abs().max()) < 1e-12 and float((ld - g["logdet"]).abs().max()) < 1e-11
  xi, ldi, _ = orqs.rqs_inverse(g["y"], g["theta"])
  assert float((xi - g["x"]).abs().max()) < 1e-11 and float((ldi + g["logdet"]).abs().max()) < 1e-10


def _dr_parts(g):
  D, L, M, H, K = (int(v) for v in g["shape"])
  shape = FlowShape(D, L, M, H, K, conditional=False)
  spec = oflow.FlowSpec(D, L, [H] * M, K, conditional=False)

  def tree(blob):
    p = unpack(shape, blob)
    p["~"]["first"] = p["~"]["first"].float()
    return p
  return shape, spec, tree


@pytest.mark.parametrize("name", list(DR))
def test_oracle_dr_matches_reference(name):
  """cnf_ot/dr/trainers.py:train's own loss_fn and value_and_grad (:91-117), run for one epoch from the reference."""
  from oracle import dr as odr
  g = load(name)
  shape, spec, tree = _dr_parts(g)
  model = DR[name]
  dec = tree(g["blob_decoder"])
  params = {"encoder": tree(g["blob_encoder"]), "decoder": dec} if model == "enc_dec" else dec
  loss, grads = odr.value_and_grad(model, spec, params, g["x"], int(g["sub_dim"]))
  assert abs(float(loss) - float(g["loss"])) <= 1e-12 * abs(float(g["loss"]))
  for key, gr in (("decoder", grads["decoder"] if model == "enc_dec" else grads),
                  ("encoder", grads.get("encoder") if model == "enc_dec" else None)):
    if gr is None:
      continue
    err = (pack(shape, gr, torch.float64) - g["grad_" + key]).abs() / float(g["grad_" + key].abs().max())
    assert float(err[:shape.Pp].max()) <= 2e-6 and float(err[shape.Pp:].max()) <= 1e-12, key


# ------------------------------------------------------------------ GPU: kernels vs the reference's outputs
@pytest.fixture(params=["mma", "cuda", "wide"])
def engine(request, monkeypatch):
  """All three conditioner engines: warp-level tensor-core (default at hidden 16), CUDA-core, and the wide-
  conditioner engine (batched tcgen05 GEMMs, csrc/wide.cu) forced onto these small flows."""
  monkeypatch.setenv("CNFOT_ENGINE", request.param)
  return request.param


@pytest.mark.gpu
@pytest.mark.parametrize("name", FLOWS)
def test_gpu_flow_matches_reference(name, engine):
  from cnf_ot_b200 import ops
  g = load(name)
  shape, _, _ = parts(g)
  f = lambda t: t.float().cuda()
  W = f(g["blob"])
  n = g["latent"].shape[0]
  # sample_and_log_prob: latent -> y = sample direction; log p(y | t) = N(latent) - log-det
  y, ld = ops.flow_eval(shape, W, f(g["latent"]), f(g["t"]), inverse=False)
  base = -0.5 * (g["latent"]**2).sum(-1) - 0.5 * shape.dim * np.log(2 * np.pi)
  assert close(y, g["sample_y"]) and close(base - ld.cpu().double(), g["sample_log_prob"])
  t0 = torch.full((n, ), float(g["t0"]))
  _, lp = ops.flow_eval(shape, W, f(g["x"]), f(t0), inverse=True, add_base=True)
  assert close(lp, g["log_prob_x"])
  yf, _ = ops.flow_eval(shape, W, f(g["x"]), f(t0), inverse=False)
  xi, _ = ops.flow_eval(shape, W, f(g["x"]), f(t0), inverse=True)
  assert close(yf, g["forward_x"]) and close(xi, g["inverse_x"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(STEPS))
def test_gpu_step_matches_reference(name, engine):
  from cnf_ot_b200 import ops
  g = load(name)
  shape, _, _ = parts(g)
  cfg = step_cfg(name, g)
  B = int(g["latent"].shape[0])
  b = B // 32
  typ = cfg["general"]["type"]
  f = lambda t: t.float().cuda()
  out = ops.mfc_step(shape, ops.problem_desc(cfg), f(g["blob"]), None if typ == "ot" else f(g["latent"]),
                     f(g["latent"][:b]), f(g["src"]) if typ == "ot" else None,
                     f(g["tgt"]) if typ == "ot" else None, g["t_batch"].tolist(), float(g["lam"]), B, b)
  out = out.cpu().double()
  G, loss = out[:shape.blob_size], float(out[shape.blob_size])
  assert abs(loss - float(g["loss"])) <= 2e-5 * abs(float(g["loss"]))
  # score terms: central differences of the float32 log-prob with 1 / dx = 100 and only b = 4-8 rows per term, so a
  # single row within rounding of a spline knot shows at the 1e-4 level (tests/test_golden.py, tools/diag_noise.py)
  assert float((G - g["grad"]).abs().max() / g["grad"].abs().max()) <= (5e-5 if typ == "ot" else 2e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ENERGIES)
def test_gpu_energies_match_reference(name, engine):
  from cnf_ot_b200 import ops
  g = load(name)
  shape, _, _ = parts(g)
  n_t = int(g["t_size"])
  W, lat = g["blob"].float().cuda(), g["latent"].float().cuda()
  e = ops.kinetic_energy(shape, W, lat, np.linspace(0.0, 1.0, n_t).tolist(), latent_blocks=1)
  # finite differences with 1/dt = 1/dx = 100 amplify float32 rounding: stated tolerance 2e-4 relative
  assert abs(float(e) - float(g["e_kin"])) <= 2e-4 * abs(float(g["e_kin"]))
  es = ops.kinetic_energy(shape, W, lat, np.linspace(0.0, float(g["T"]), n_t).tolist(), with_score=True,
                          kappa=1.0 / float(g["beta"]), latent_blocks=1)
  assert abs(float(es) - float(g["e_score"])) <= 1e-3 * abs(float(g["e_score"]))   # see tests/test_gpu_energies.py


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DR))
def test_gpu_dr_matches_reference(name):
  from cnf_ot_b200 import dr
  from cnf_ot_b200.flows import ParamTree
  g = load(name)
  shape, _, _ = _dr_parts(g)
  model = DR[name]
  cfg = {"cnf": {"flow_num_layers": shape.num_layers, "mlp_num_layers": shape.mlp_layers, "hidden_size": shape.hidden,
                 "num_bins": shape.num_bins}}
  enc, dec = dr.build(shape.dim, cfg, model)
  td = ParamTree(shape, g["blob_decoder"].float().cuda())
  params = {"encoder": ParamTree(shape, g["blob_encoder"].float().cuda()), "decoder": td} if model == "enc_dec" else td
  loss, grads = dr.value_and_grad(model, enc, dec, int(g["sub_dim"]))(params, g["x"].float().cuda())
  assert abs(float(loss) - float(g["loss"])) <= 2e-5 * abs(float(g["loss"]))
  G = (grads["decoder"] if model == "enc_dec" else grads).blob.cpu().double()
  err = (G - g["grad_decoder"]).abs() / g["grad_decoder"].abs().max()
  assert float(err.quantile(0.99)) <= 5e-5 and float(err.max()) <= 1e-3   # tie rows: see tests/test_gpu_dr.py


@pytest.mark.gpu
def test_gpu_ot_reverse_kl_mirror():
  """applications.ot_reverse_kl_loss_fn of the mirror vs the restatement pinned above, on the mirror's own draws."""
  from cnf_ot_b200 import applications, random
  from cnf_ot_b200.flows import ParamTree, RQSFlow
  g = load("ref_flow_d2")
  shape, spec, params = parts(g)
  model = RQSFlow((shape.dim, ), shape.num_layers, [shape.hidden] * shape.mlp_layers, shape.num_bins)
  tree = ParamTree(model.shape, g["blob"].float().cuda())
  rng = random.PRNGKey(3)
  n = 1024
  got = applications.ot_reverse_kl_loss_fn(model, shape.dim, 1, tree, rng, n)
  latent = random.normal(rng, (n, shape.dim)).double().cpu()
  want = _ot_reverse_kl_oracle(spec, params, latent)
  assert abs(float(got) - float(want)) <= 2e-5 * abs(float(want))
