"""Float32 conditioning of the train step at B = 2^17 (dev tool; the sigma choices of tests/test_gpu_scale.py rest on it):
  python tools/diag_scale.py

For two flows of the step matrix -- the mfc.yaml flow on rwpo/double_well and the M = 1 flow on ot/free -- and a few
parameter perturbations sigma, prints each engine's gradient error against the float64 oracle (max |G - G_oracle| over
the largest oracle entry, one-thread-per-row kinetic form), and, at the largest sigma, how far 32 shards of 4 096 rows
(one tile per CTA) are from the same engine's whole-batch result (multi-tile grid, several tiles per CTA).  Errors that
differ between engines, grow with the batch and sigma, and come with shards that add up to the whole batch are the
case's float32 conditioning, not a fault of the persistent kernels."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
from cnf_ot_b200 import _lib, ops
from cnf_ot_b200.layout import pack
from oracle import losses as olosses
from util import make_cfg, make_inputs, make_params, shape_of

B, LAM, SHARD = 1 << 17, 500.0, 4096
CASES = [("rwpo", "double_well", dict(M=2), (0.3, 0.2)), ("ot", "free", dict(M=1), (0.3, 0.1))]


def step(cfg, shape, params, inputs, rows, sub_rows):
  b = B // 32
  f = lambda t: t.float().cuda()
  ot = cfg["general"]["type"] == "ot"
  out = ops.mfc_step(shape, ops.problem_desc(cfg), pack(shape, params).cuda(),
                     None if ot else f(inputs["latent"][rows]), f(inputs["latent"][:b][sub_rows]),
                     f(inputs["src"][rows]) if ot else None, f(inputs["tgt"][rows]) if ot else None,
                     inputs["t_batch"].tolist(), LAM, B, b)
  return out.cpu().double()[:shape.blob_size]


def main():
  os.environ["CNFOT_KINETIC_SPLIT"] = "0"
  print(json.dumps({"gpu": torch.cuda.get_device_name(0)}))
  for typ, sub, kw, sigmas in CASES:
    cfg = make_cfg(typ, sub, B=B, Tn=2, lam=LAM, **kw)
    shape = shape_of(cfg)
    inputs = make_inputs(cfg)
    for sigma in sigmas:
      spec, params = make_params(cfg, sigma)
      _, grads = olosses.value_and_grad(cfg, spec, params, inputs)
      Gor = pack(shape, grads, torch.float64)
      for eng in ("mma", "cuda", "tc"):
        os.environ["CNFOT_ENGINE"] = eng
        whole = step(cfg, shape, params, inputs, slice(0, B), slice(0, B // 32))
        r = {"case": f"{typ}/{sub}", "M": kw["M"], "sigma": sigma, "engine": eng, "grid": _lib.last_launch_info()["grid"],
             "grad_rel": float((whole - Gor).abs().max() / Gor.abs().max())}
        if sigma == sigmas[0]:
          s = SHARD // 32
          parts = [step(cfg, shape, params, inputs, slice(i * SHARD, (i + 1) * SHARD), slice(i * s, (i + 1) * s))
                   for i in range(B // SHARD)]
          r["shard_grid"] = _lib.last_launch_info()["grid"]
          r["shards_vs_whole"] = float((sum(parts) - whole).abs().max() / Gor.abs().max())
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
  main()
