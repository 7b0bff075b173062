"""Generate the golden fixtures under tests/golden/ from the CPU oracle (torch float64).

  python tests/golden/make_golden.py
  python -c "import make_golden; make_golden.save_mirror_signatures()"   (from tests/golden: the API record alone)

PROVENANCE: these vectors are outputs of oracle/ (the restatement of the reference), NOT of the reference itself; the
fixtures produced by the reference's own code are tests/golden/ref_*.npz (make_reference_golden.py), which also pin
oracle/.  The files made here cover shapes the reference's code does not run (3- and 4-dimensional mixtures, the hidden-64
flow of the wide engine), pin the oracle against silent change (tests/test_golden.py, CPU) and give the GPU parity
tests fixed vectors that do not depend on torch's RNG stream (tests/test_golden.py, -m gpu).
Every input is float32-representable so the kernels see exactly the same numbers.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "tests")):
  if p not in sys.path:
    sys.path.insert(0, p)

from cnf_ot_b200.layout import pack  # noqa: E402
from oracle import flow as oflow  # noqa: E402
from oracle import losses as olosses  # noqa: E402
from oracle import rqs as orqs  # noqa: E402
from util import make_cfg, make_inputs, make_params, shape_of  # noqa: E402

f32 = lambda t: t.to(torch.float32).to(torch.float64)


def spline_case(K, n, seed):
  """Raw parameters as the reference test draws them (tests/test_rqs_accuracy.py:60-69: N(0,1) * 0.5),
  inputs spread over the range and both tails, plus inputs sitting exactly on interior knots."""
  g = torch.Generator().manual_seed(seed)
  P = 3 * K + 1
  theta = f32(torch.randn(n, P, generator=g, dtype=torch.float64) * 0.5)
  x = f32((torch.rand(n, generator=g, dtype=torch.float64) - 0.5) * 26.0)  # [-13, 13]: tails included
  y, ld, bins = orqs.rqs_forward(x, theta)
  xi, ldi, bins_i = orqs.rqs_inverse(x, theta)
  return {"theta": theta, "x": x, "fwd_y": y, "fwd_logdet": ld, "fwd_bin": bins,
          "inv_x": xi, "inv_logdet": ldi, "inv_bin": bins_i}


def flow_case(D, L, M, H, K, sigma, n, seed):
  cfg = make_cfg(dim=D, L=L, M=M, H=H, K=K)
  shape = shape_of(cfg)
  spec, params = make_params(cfg, sigma)
  g = torch.Generator().manual_seed(seed)
  x = f32(torch.randn(n, D, generator=g, dtype=torch.float64))
  t = f32(torch.rand(n, generator=g, dtype=torch.float64))
  y, fld = oflow.flow_forward_and_log_det(spec, params, x, t.reshape(-1, 1))
  xi, ild = oflow.flow_inverse_and_log_det(spec, params, x, t.reshape(-1, 1))
  return {"shape": np.array([D, L, M, H, K]), "blob": pack(shape, params, torch.float64), "x": x, "t": t,
          "fwd_y": y, "fwd_logdet": fld, "inv_x": xi, "inv_logdet": ild,
          "log_prob": oflow.base_log_prob(xi) + ild}


def step_case(typ, sub, B, lam, Tn, **kw):
  sigma = kw.pop("sigma", 0.3)
  cfg = make_cfg(typ, sub, Tn=Tn, lam=lam, B=B, **kw)
  shape = shape_of(cfg)
  spec, params = make_params(cfg, sigma)
  inputs = make_inputs(cfg)
  loss, grads = olosses.value_and_grad(cfg, spec, params, inputs)
  c = cfg["cnf"]
  return {"shape": np.array([cfg["general"]["dim"], c["flow_num_layers"], c["mlp_num_layers"], c["hidden_size"],
                             c["num_bins"]]),
          "blob": pack(shape, params, torch.float64), "latent": inputs["latent"], "src": inputs["src"],
          "tgt": inputs["tgt"], "t_batch": inputs["t_batch"], "lam": np.array(lam), "loss": loss.detach(),
          "grad": pack(shape, grads, torch.float64)}


def dr_case(model, D, L, H, sub_dim, sigma, n, seed):
  """Dimension-reduction loss (cnf_ot/dr/trainers.py:91-111) on unconditional flows (oracle/dr.py)."""
  from cnf_ot_b200.layout import FlowShape
  from oracle import dr as odr
  spec = oflow.FlowSpec(D, L, [H, H], 5, conditional=False)
  shape = FlowShape(D, L, 2, H, 5, conditional=False)

  def mk(s):
    p = oflow.perturb_params(oflow.init_params(spec, s), sigma, seed=s + 10)
    return {m: {k: v.to(torch.float32).to(v.dtype) for k, v in lv.items()} for m, lv in p.items()}
  g = torch.Generator().manual_seed(seed)
  x = f32(torch.randn(n, D, generator=g, dtype=torch.float64) * 1.5)
  dec = mk(2)
  params = {"encoder": mk(1), "decoder": dec} if model == "enc_dec" else dec
  loss, grads = odr.value_and_grad(model, spec, params, x, sub_dim)
  out = {"shape": np.array([D, L, 2, H, 5]), "sub_dim": np.array(sub_dim), "x": x, "loss": loss,
         "blob_decoder": pack(shape, dec, torch.float64),
         "grad_decoder": pack(shape, grads["decoder"] if model == "enc_dec" else grads, torch.float64)}
  if model == "enc_dec":
    out["blob_encoder"] = pack(shape, params["encoder"], torch.float64)
    out["grad_encoder"] = pack(shape, grads["encoder"], torch.float64)
  return out


def save(name, d):
  out = {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in d.items()}
  np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
  print(name, {k: v.shape for k, v in out.items()})


# the mirror's API that tests/test_reference_golden.py compares with the original project's source
# (None: every public function of the module)
SIGNATURES = {"cnf_ot_b200.applications": None,
              "cnf_ot_b200.utils": ["calc_kinetic_energy", "calc_score_kinetic_energy"],
              "cnf_ot_b200.flows": ["RQSFlow"], "cnf_ot_b200.solvers": ["main"]}


def save_mirror_signatures():
  """mirror_signatures.json: parameter names of the mirror's API as this repository defines it (NOT read from the
  original project), so that the mirror cannot drift without a test failing where the original is not at hand."""
  import importlib
  import inspect
  import json
  out = {}
  for mod_name, names in SIGNATURES.items():
    mod = importlib.import_module(mod_name)
    if names is None:
      names = sorted(n for n, f in inspect.getmembers(mod, inspect.isfunction)
                     if f.__module__ == mod_name and not n.startswith("_"))
    out[mod_name] = {n: list(inspect.signature(getattr(mod, n)).parameters) for n in names}
  with open(os.path.join(HERE, "mirror_signatures.json"), "w") as f:
    json.dump(out, f, indent=1)
    f.write("\n")


STEP_CASES = {
  # hidden 64: outside the fused kernels, runs on the wide-conditioner engine (csrc/wide.cu)
  "step_ot_free_d3_h64": ("ot", "free", 256, 500.0, 2, dict(dim=3, H=64, sigma=0.05)),
  "step_ot_obstacle": ("ot", "obstacle", 256, 500.0, 2, {}),
  "step_rwpo_double_well": ("rwpo", "double_well", 256, 500.0, 2, {}),
  "step_fp_nongradient_d4": ("fp", "nongradient", 128, 100.0, 1, dict(dim=4, sigma=0.1)),
}

if __name__ == "__main__":
  save("rqs_k5", spline_case(5, 512, 7))
  save("rqs_k8", spline_case(8, 256, 8))
  save("flow_d2", flow_case(2, 2, 2, 16, 5, 0.3, 384, 9))
  save("flow_d3_h8", flow_case(3, 3, 1, 8, 3, 0.1, 256, 10))
  save("flow_d3_h64", flow_case(3, 2, 2, 64, 5, 0.05, 256, 11))
  save("dr_enc_dec_d4", dr_case("enc_dec", 4, 2, 16, 2, 0.08, 320, 12))
  save("dr_dec_only_d4", dr_case("dec_only", 4, 2, 16, 2, 0.08, 320, 13))
  for name, (typ, sub, B, lam, Tn, kw) in STEP_CASES.items():
    save(name, step_case(typ, sub, B, lam, Tn, **dict(kw)))
  save_mirror_signatures()
