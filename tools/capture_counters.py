"""Hardware counters of one launch of the cfg-2 step kernel (the headline workload of bench.py), read through the CUPTI
range profiler API -- the three counters profiles/traffic.json records, without Nsight Compute:

  python tools/capture_counters.py OUT.json      # then: python tools/make_traffic.py OUT.json

Builds tools/cupti_counters.cpp into a temporary directory, runs three warm-up steps and captures the next one as a
user range (one step is one kernel launch on a registered workspace); if the metric set needs several passes, the
step is repeated, one pass each.  L2 is flushed before every captured step, as Nsight Compute does by default, so the
DRAM bytes are those of a step that starts from a cold cache.  The output carries the GPU, its power limit and the
hash of the kernel sources the library was built from.  Needs access to the GPU's performance counters.
"""
import ctypes, json, os, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
METRICS = ["smsp__inst_executed.sum", "dram__bytes_read.sum", "dram__bytes_write.sum"]


def build_lib(tmp):
  cuda = os.path.dirname(os.path.dirname(subprocess.check_output(["which", "nvcc"], text=True).strip()))
  lib64 = os.path.join(cuda, "lib64")
  so = os.path.join(tmp, "libcupti_counters.so")
  subprocess.check_call(["nvcc", "-Wno-deprecated-gpu-targets", "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC,-fvisibility=hidden",
                         os.path.join(ROOT, "tools", "cupti_counters.cpp"), "-o", so, "-I", os.path.join(cuda, "include"),
                         "-L", lib64, "-L", os.path.join(lib64, "stubs"), "-lcupti", "-lcuda", f"-Xlinker=-rpath={lib64}"])
  return so


def main():
  out_path = sys.argv[1]
  import torch
  import bench
  from make_traffic import fingerprint

  class _D:
    world, rank, local = 1, 0, 0
    dev = torch.device("cuda", 0)
    td = None

  torch.cuda.set_device(0)
  w = bench.Workload("cfg2", _D())
  for i in range(3):
    w.step(i)
  torch.cuda.synchronize()
  with tempfile.TemporaryDirectory() as tmp:
    cc = ctypes.CDLL(build_lib(tmp))
  cc.cc_error.restype = ctypes.c_char_p
  # L2 flush without dirty lines: both buffers are written first, then `cold` is read, which evicts `hot`'s written-back
  # lines and leaves L2 full of clean ones
  hot, cold = (torch.ones(96 << 20, device="cuda") for _ in range(2))
  if cc.cc_begin(",".join(METRICS).encode(), 1, 1) != 0:
    sys.exit(f"capture_counters: {cc.cc_error().decode()}")
  done, i = ctypes.c_int(0), 3
  while not done.value:
    hot.add_(1.0)
    float(cold.sum())
    if cc.cc_start() != 0:
      sys.exit(f"capture_counters: {cc.cc_error().decode()}")
    w.step(i)
    torch.cuda.synchronize()
    if cc.cc_stop(ctypes.byref(done)) != 0:
      sys.exit(f"capture_counters: {cc.cc_error().decode()}")
    i += 1
  buf = ctypes.create_string_buffer(1 << 16)
  if cc.cc_end(buf, len(buf)) != 0:
    sys.exit(f"capture_counters: {cc.cc_error().decode()}")
  ranges = [l.split("\t") for l in buf.value.decode().splitlines() if not l.startswith("#")]
  if len(ranges) != 1:
    sys.exit(f"capture_counters: expected one range, got {buf.value.decode()!r}")
  smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
  res = {"metrics": {m: float(v) for m, v in zip(METRICS, ranges[0][1:])}, "passes": i - 3, "gpu": smi,
         "csrc_sha16": fingerprint(), "rows": w.B, "tool": "CUPTI range profiler, one step as a user range after an L2 flush, tools/capture_counters.py"}
  with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
  print(json.dumps(res, indent=1))


if __name__ == "__main__":
  main()
