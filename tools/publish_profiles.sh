#!/bin/bash
# Copy the evidence of one tools/gpu_round2.sh visit (gpurun_out/*_TAG.*) into profiles/ under the round-2 names that
# profiles/README.md lists, regenerate the ncu summaries and tie profiles/latest_traffic.json to the build the capture ran on.
# usage: tools/publish_profiles.sh TAG      (run from the repository root, after the library has been built)
set -e
TAG=$1; G=gpurun_out; P=profiles
cp $G/bench_$TAG.json $P/r02_bench.json
cp $G/bench_ref_$TAG.json $P/r02_bench_ref.json
cp $G/launches_$TAG.csv $P/r02_launches.csv
cp $G/sweep_$TAG.jsonl $P/r02_sweep.jsonl
cp $G/pytest_gpu_$TAG.log $P/r02_pytest_gpu.log
for k in r64 w big; do
  [ -f $G/prof_${k}_$TAG.ncu-rep ] && bash tools/ncu_sum.sh $G/prof_${k}_$TAG.ncu-rep > $P/r02_ncu_summary_$k.txt
done
[ -f /tmp/ncu_prof_r64_$TAG.src.csv ] && python tools/ncu_regions.py /tmp/ncu_prof_r64_$TAG.src.csv 128 > $P/r02_ncu_regions_r64.txt
python - "$TAG" <<'PY'
import json, re, sys
sys.path.insert(0, "spectroplot-js_b200")
from spectro_b200 import _lib
tag = sys.argv[1]
txt = open("profiles/r02_ncu_summary_r64.txt").read()
rd = float(re.search(r"dram__bytes_read.sum\s+([\d.]+) Mbyte", txt).group(1))
wr = float(re.search(r"dram__bytes_write.sum\s+([\d.]+) Mbyte", txt).group(1))
bench = json.loads(open("profiles/r02_bench.json").read().strip().splitlines()[-1])
bid = bench["roofline"]["kernel_build"]
assert bid == _lib.build_id(), (bid, _lib.build_id(), "the library in the tree is not the build the evidence run used")
json.dump({"dram_bytes_per_launch": int(round((rd + wr) * 1e6)), "build_id": bid,
           "kernel": "render_r64_kernel<CS16> (N=4096, 64x64 FFT, 4 FFT streams + store warpgroup)",
           "source": f"profiles/r02_ncu_summary_r64.txt: dram__bytes_read.sum {rd:.3f} MB + dram__bytes_write.sum {wr:.3f} MB, ncu --set full, "
                     f"C2 workload, build {bid} (gpurun visit {tag})"}, open("profiles/latest_traffic.json", "w"))
print(open("profiles/latest_traffic.json").read())
PY
