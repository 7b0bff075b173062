"""ctypes binding of libcnfot.so (the C ABI declared in include/cnfot.h).

The library is built in-tree by `__graft_entry__.build()` /
`make -C cnf_ot_b200/csrc`.  There is no fallback of any kind: a missing
library or a failing call raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, os.environ.get("CNFOT_LIB", "libcnfot.so"))   # CNFOT_LIB: an alternative build (A/B timing)

ABI_VERSION = 2
NUM_LOSS_SLOTS = 8

OT, RWPO, FP = 0, 1, 2
SUBTYPES = {
  "ot": {"free": 0, "obstacle": 1},
  "rwpo": {"quadratic": 0, "double_well": 1},
  "fp": {"gradient": 0, "nongradient": 1, "lorenz": 2},
}
TYPES = {"ot": OT, "rwpo": RWPO, "fp": FP}


class CnfotError(RuntimeError):
  pass


class FlowDesc(Structure):
  _fields_ = [
    ("dim", c_int32), ("num_layers", c_int32), ("mlp_layers", c_int32), ("hidden", c_int32),
    ("num_bins", c_int32), ("range_min", c_float), ("range_max", c_float),
    ("min_bin_size", c_float), ("min_knot_slope", c_float),
  ]


class ProblemDesc(Structure):
  _fields_ = [
    ("type", c_int32), ("subtype", c_int32), ("T", c_float), ("beta", c_float), ("a", c_float),
    ("sigma", c_float), ("dt", c_float), ("dx", c_float),
  ]


class PeerDesc(Structure):
  """cnfot_peer_desc: peer-mapped exchange buffers of the fused step + all-reduce."""
  _fields_ = [("rank", c_int32), ("world", c_int32), ("epoch", ctypes.c_uint32),
              ("xbuf", c_void_p * 8), ("flags", c_void_p * 8)]


class AdamDesc(Structure):
  """cnfot_adam_desc: optax.adam hyper-parameters (solvers.py:55)."""
  _fields_ = [("lr", c_float), ("b1", c_float), ("b2", c_float), ("eps", c_float)]


# cnfot_philox_rows sources (include/cnfot.h)
ROWS_NORMAL, ROWS_OT_SOURCE = 1, 3
STATUS_WORD = 4

_F = POINTER(FlowDesc)
_P = POINTER(ProblemDesc)
_RQS = [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_float, c_float, c_float, c_float,
        c_void_p, c_void_p, c_void_p]
_RQS_VJP = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_float, c_float,
            c_float, c_float, c_void_p, c_void_p]
_FLOW = [c_void_p, _F, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int32]
_FLOW_VJP = [c_void_p, _F, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
             c_int32, c_void_p, c_void_p, c_void_p, c_int64]
_STEP = [c_void_p, _F, _P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
         c_int64, c_int64, c_int64, c_int64, c_float, c_void_p, c_void_p, c_int64]

# every symbol include/cnfot.h declares: name -> (restype, argtypes)
SIGNATURES = {
  "cnfot_abi_version": (c_int32, []),
  "cnfot_last_error": (c_char_p, []),
  "cnfot_last_launch_info": (None, [POINTER(c_int32)] * 4),
  "cnfot_last_launch_variant": (None, [POINTER(c_int32)] * 4),
  "cnfot_debug_step_timeline": (None, [c_void_p]),
  "cnfot_workspace_register": (c_int32, [c_void_p, _F, c_void_p, c_int64]),
  "cnfot_workspace_release": (c_int32, [c_void_p]),
  "cnfot_param_count": (c_int64, [_F]),
  "cnfot_spline_param_stride": (c_int64, [_F]),
  "cnfot_offset_first": (c_int64, [_F]),
  "cnfot_offset_linear": (c_int64, [_F, c_int32, c_int32, c_int32, c_int32]),
  "cnfot_flow_supported": (c_int32, [_F]),
  "cnfot_rqs_forward": (c_int32, _RQS),
  "cnfot_rqs_inverse": (c_int32, _RQS),
  "cnfot_rqs_forward_vjp": (c_int32, _RQS_VJP),
  "cnfot_rqs_inverse_vjp": (c_int32, _RQS_VJP),
  "cnfot_flow_forward": (c_int32, _FLOW),
  "cnfot_flow_inverse": (c_int32, _FLOW),
  "cnfot_flow_workspace_bytes": (c_int64, [_F, c_int64]),
  "cnfot_flow_forward_ws": (c_int32, _FLOW + [c_void_p, c_int64]),
  "cnfot_flow_inverse_ws": (c_int32, _FLOW + [c_void_p, c_int64]),
  "cnfot_flow_vjp_workspace_bytes": (c_int64, [_F, c_int64]),
  "cnfot_flow_forward_vjp": (c_int32, _FLOW_VJP),
  "cnfot_flow_inverse_vjp": (c_int32, _FLOW_VJP),
  "cnfot_mfc_step_workspace_bytes": (c_int64, [_F, c_int64, c_int64, c_int32]),
  "cnfot_mfc_step": (c_int32, _STEP),
  "cnfot_mfc_step_host_workspace_bytes": (c_int64, [_F, c_int64, c_int64, c_int32]),
  "cnfot_mfc_step_host": (c_int32, _STEP),
  "cnfot_kinetic_energy_workspace_bytes": (c_int64, [_F, c_int32]),
  "cnfot_kinetic_energy": (c_int32, [c_void_p, _F, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int32,
                                     c_float, c_int32, c_float, c_float, c_void_p, c_void_p, c_int64]),
  "cnfot_dp_exchange_stride": (c_int64, [_F]),
  "cnfot_dp_exchange_floats": (c_int64, [_F, c_int32]),
  "cnfot_dp_flag_count": (c_int64, [_F, c_int32]),
  "cnfot_mfc_step_dp": (c_int32, _STEP + [POINTER(PeerDesc)]),
  "cnfot_philox_rows": (c_int32, [c_void_p, ctypes.c_uint64, ctypes.c_uint32, c_int32, c_int64, c_int64, c_int64, c_int32,
                                  c_void_p]),
  "cnfot_philox_times_host": (c_int32, [ctypes.c_uint64, ctypes.c_uint32, c_int32, c_float, c_void_p]),
  "cnfot_mfc_step_rng": (c_int32, [c_void_p, _F, _P, c_void_p, ctypes.c_uint64, ctypes.c_uint32, c_int32, c_int64, c_int64,
                                   c_int64, c_int64, c_int64, c_int64, c_float, c_void_p, c_void_p, c_int64,
                                   POINTER(PeerDesc)]),
  "cnfot_mfc_step_rng_host_workspace_bytes": (c_int64, [_F]),
  "cnfot_mfc_step_rng_host": (c_int32, [c_void_p, _F, _P, c_void_p, ctypes.c_uint64, ctypes.c_uint32, c_int32, c_int64,
                                        c_int64, c_int64, c_int64, c_int64, c_int64, c_float, c_void_p, c_void_p, c_int64]),
  "cnfot_train_state_bytes": (c_int64, [_F]),
  "cnfot_train_state_init": (c_int32, [c_void_p, _F, c_void_p, c_int64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32]),
  "cnfot_mfc_update": (c_int32, [c_void_p, _F, _P, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, POINTER(AdamDesc),
                                 c_int32, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_float, c_void_p,
                                 c_void_p, c_int64, POINTER(PeerDesc)]),
  "cnfot_density_workspace_bytes": (c_int64, [_F, c_int32]),
  "cnfot_density_grid": (c_int32, [c_void_p, _F, c_void_p, c_void_p, c_int32, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                   ctypes.c_double, c_int32, c_int32, c_void_p, c_int32, c_float, c_float, c_float, c_void_p,
                                   c_void_p, c_int64]),
  "cnfot_density_mc": (c_int32, [c_void_p, _F, c_void_p, c_float, ctypes.c_uint64, ctypes.c_uint32, c_int64, c_void_p, c_void_p,
                                 c_int32, c_float, c_float, c_float, c_void_p, c_void_p, c_int64]),
  "cnfot_dense_prepared_floats": (c_int64, [c_int32, c_int32]),
  "cnfot_dense_prepare": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]),
  "cnfot_dense_forward": (c_int32, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_void_p, c_int32, c_void_p,
                                    c_void_p, c_int32, c_int32, c_void_p, c_int32]),
  "cnfot_dense_wgrad": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int64, c_int32, c_int32,
                                  c_void_p, c_int32, c_void_p]),
  "cnfot_mask_tail": (c_int32, [c_void_p, c_void_p, c_int64, c_int32, c_int32]),
  "cnfot_recon_head": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_float, c_void_p, c_void_p]),
  "cnfot_adam_update": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                  c_float, c_float, c_float, c_float, c_int64]),
}

_lib = None


def load() -> ctypes.CDLL:
  """Load libcnfot.so and bind every declared symbol; raises if anything is missing."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise CnfotError(
      f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
      "or `make -C cnf_ot_b200/csrc` (nvcc, sm_100a). cnf_ot_b200 has no CPU fallback."
    )
  lib = ctypes.CDLL(LIB_PATH)
  for name, (res, args) in SIGNATURES.items():
    fn = getattr(lib, name)  # AttributeError if the symbol is not exported
    fn.restype = res
    fn.argtypes = args
  if lib.cnfot_abi_version() != ABI_VERSION:
    raise CnfotError("libcnfot.so ABI version mismatch; rebuild")
  _lib = lib
  return lib


def last_launch_info() -> dict:
  vals = [c_int32(0) for _ in range(4)]
  load().cnfot_last_launch_info(*[ctypes.byref(v) for v in vals])
  eng = vals[3].value  # 0 CUDA cores, 1 tcgen05 engine, 2 warp-level MMA engine, 4 wide-conditioner engine
  return {"grid": vals[0].value, "smem_bytes": vals[1].value, "ctas_per_sm": vals[2].value,
          "tensor_cores": bool(eng), "engine": {0: "cuda", 1: "tc", 2: "mma", 4: "wide"}.get(eng, "?")}


def last_launch_variant() -> dict:
  """Kernel instantiation of the calling thread's most recent fused step / VJP launch (cnfot_last_launch_variant)."""
  vals = [c_int32(0) for _ in range(4)]
  load().cnfot_last_launch_variant(*[ctypes.byref(v) for v in vals])
  plan = {0: "cuda", 1: "tc", 2: "mma", 3: "mma_stream", 4: "wide"}.get(vals[0].value, None)
  return {"plan": plan, "stash_tmem_cols": vals[1].value, "kinetic_group": vals[2].value, "latency": bool(vals[3].value)}


def check(rc: int) -> None:
  if rc != 0:
    msg = load().cnfot_last_error()
    raise CnfotError(f"libcnfot error {rc}: {msg.decode() if msg else '?'}")


def flow_desc(shape) -> FlowDesc:
  return FlowDesc(shape.dim, shape.num_layers, shape.mlp_layers, shape.hidden, shape.num_bins,
                  shape.range_min, shape.range_max, shape.min_bin_size, shape.min_knot_slope)
