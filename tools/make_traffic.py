"""profiles/traffic.json from a counter capture of the step kernel (run after every kernel change; bench.py refuses a
file whose source hash differs from the sources the loaded library was built from):

  python tools/make_traffic.py <step.ncu-rep | capture.json> [<dense_tc.ncu-rep>]

capture.json: written by tools/capture_counters.py (CUPTI range profiler); it must carry the hash of the sources here.

Records, per launch of mfc_step_kernel (BASELINE cfg 2): dram__bytes_read.sum + dram__bytes_write.sum and
smsp__inst_executed.sum, plus the hash of cnf_ot_b200/csrc the capture belongs to (bench.kernel_fingerprint)."""
import csv, io, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def fingerprint():
  import hashlib
  h = hashlib.sha256()
  csrc = os.path.join(ROOT, "cnf_ot_b200", "csrc")
  for fn in sorted(os.listdir(csrc)):
    if fn.endswith((".cu", ".cuh", ".h")):
      with open(os.path.join(csrc, fn), "rb") as f:
        h.update(fn.encode())
        h.update(f.read())
  return h.hexdigest()[:16]


def raw(rep):
  out = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
  rows = list(csv.reader(io.StringIO(out)))
  h, units = rows[0], rows[1]
  return [dict(zip(h, r)) for r in rows[2:]], dict(zip(h, units))


def num(v, unit):
  x = float(v.replace(",", ""))
  return x * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "inst": 1, "": 1}.get(unit, 1)


def main():
  step_rep = sys.argv[1]
  if step_rep.endswith(".json"):
    cap = json.load(open(step_rep))
    if cap["csrc_sha16"] != fingerprint():
      sys.exit(f"{step_rep} was captured from other kernel sources ({cap['csrc_sha16']} != {fingerprint()})")
    m = cap["metrics"]
    rd, wr, insts = m["dram__bytes_read.sum"], m["dram__bytes_write.sum"], m["smsp__inst_executed.sum"]
    how = f"{cap['tool']}, {cap['gpu']}"
  else:
    ks, units = raw(step_rep)
    k = next(r for r in ks if "mfc_step_kernel" in r["Kernel Name"])
    rd = num(k["dram__bytes_read.sum"], units["dram__bytes_read.sum"])
    wr = num(k["dram__bytes_write.sum"], units["dram__bytes_write.sum"])
    insts = num(k["smsp__inst_executed.sum"], units["smsp__inst_executed.sum"])
    how = "ncu --set full --clock-control none"
  tpath = os.path.join(ROOT, "profiles", "traffic.json")
  old = json.load(open(tpath)) if os.path.exists(tpath) else {}
  tj = {
    "csrc_sha16": fingerprint(),
    "mfc_step_kernel_dram_bytes_per_launch": int(rd + wr),
    "mfc_step_kernel_warp_insts_per_launch": int(insts),
    "source": f"{os.path.basename(step_rep)} ({how}, one launch of the cfg-2 step: dram__bytes_read.sum "
              f"{int(rd)} + dram__bytes_write.sum {int(wr)}; smsp__inst_executed.sum); written by tools/make_traffic.py",
  }
  for key in ("dense_tc_kernel_256_1_dram_bytes_per_launch", "dense_tc_kernel_source"):
    if key in old:
      tj[key] = old[key]
  if len(sys.argv) > 2:
    ks, units = raw(sys.argv[2])
    k = next(r for r in ks if "dense_tc_kernel" in r["Kernel Name"])
    tj["dense_tc_kernel_256_1_dram_bytes_per_launch"] = int(num(k["dram__bytes_read.sum"], units["dram__bytes_read.sum"]) +
                                                            num(k["dram__bytes_write.sum"], units["dram__bytes_write.sum"]))
    tj["dense_tc_kernel_source"] = f"{os.path.basename(sys.argv[2])} (ncu --set full, one launch)"
  with open(tpath, "w") as f:
    json.dump(tj, f, indent=1)
  print(json.dumps(tj, indent=1))


if __name__ == "__main__":
  main()
