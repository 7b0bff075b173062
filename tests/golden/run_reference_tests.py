"""Execute the reference's OWN unit test of the spline, unmodified, against the stand-in spline (oracle/rqs.py behind the
`distrax.RationalQuadraticSpline` interface of tests/golden/refshim.py):

  CNF_OT_REFERENCE=<checkout of the original cnf_ot project> python tests/golden/run_reference_tests.py
                                                     (exit code 0 = every test method passed)

The original project's tests/test_rqs_accuracy.py holds the reference's known-answer checks for this path (SURVEY.md section 8c):
forward-inverse and inverse-forward round trips, log-det against the autodiff Jacobian, boundary round trips, all < 1e-12
in float64 on three spline configurations.  Run in its own process: the stand-ins register fake `jax` / `distrax` modules.
"""
import importlib.util
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, HERE):
  if p not in sys.path:
    sys.path.insert(0, p)

import refshim  # noqa: E402

refshim.install()
refshim.Draws.set()   # nothing programmed: jax.random.uniform is a seeded stream per key

if not os.environ.get("CNF_OT_REFERENCE"):
  sys.exit("set CNF_OT_REFERENCE to a checkout of the original cnf_ot project")
path = os.path.join(os.environ["CNF_OT_REFERENCE"], "tests", "test_rqs_accuracy.py")
spec = importlib.util.spec_from_file_location("reference_test_rqs_accuracy", path)
mod = importlib.util.module_from_spec(spec)
spec.loader.exec_module(mod)
ran = 0
for cls_name in dir(mod):
  cls = getattr(mod, cls_name)
  if isinstance(cls, type) and cls_name.startswith("Test"):
    obj = cls()
    for name in dir(obj):
      if name.startswith("test_"):
        getattr(obj, name)()
        ran += 1
        print(f"PASSED {path}::{cls_name}::{name}")
assert ran >= 1
