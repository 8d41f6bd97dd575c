#!/bin/bash
# Overlap of back-to-back N = 4096 renders (render_r64_kernel / finalize_kernel, programmatic dependent launch), on one B200:
# GPU suite + smoke, then `bench.py --kernel-only` (the timed C2 leg) alternating three arms REPS times - the parent build in
# spectroplot-js_b200/lib_base (make OUT=../lib_base at the parent commit), this build, this build with SP_NO_PDL=1 - and
# the full bench line of both builds with --dump-outputs, compared output for output.
# usage: bash tools/gpu_pdl_ab.sh OUT_DIR [REPS]      (logs, bench lines and summary.txt go to OUT_DIR)
OUT=${1:?usage: bash tools/gpu_pdl_ab.sh OUT_DIR [REPS]}; REPS=${2:-3}; mkdir -p $OUT
BASE=$(realpath spectroplot-js_b200/lib_base/libspectro_b200.so)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/gpu.txt
timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider > $OUT/pytest_gpu.log 2>&1; echo "pytest rc=$?" >> $OUT/pytest_gpu.log
tail -2 $OUT/pytest_gpu.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/smoke.log
tail -1 $OUT/smoke.log
: > $OUT/ab.jsonl
for rep in $(seq $REPS); do
  for arm in base new nopdl; do
    case $arm in
      base) line=$(SP_LIB=$BASE timeout 300 python bench.py --steps 1000 --warmup 20 --kernel-only 2>> $OUT/ab.err) ;;
      new) line=$(timeout 300 python bench.py --steps 1000 --warmup 20 --kernel-only 2>> $OUT/ab.err) ;;
      nopdl) line=$(SP_NO_PDL=1 timeout 300 python bench.py --steps 1000 --warmup 20 --kernel-only 2>> $OUT/ab.err) ;;
    esac
    echo "{\"arm\": \"$arm\", \"rep\": $rep, \"bench\": ${line:-null}}" >> $OUT/ab.jsonl
  done
done
SP_LIB=$BASE timeout 900 python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs $OUT/dump_base > $OUT/bench_base.json 2>> $OUT/bench.err
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs $OUT/dump_new > $OUT/bench_new.json 2>> $OUT/bench.err
python - <<PY | tee $OUT/summary.txt
import glob, json, os
import numpy as np
out = "$OUT"
print(open(out + "/gpu.txt").read().strip())
rows = [json.loads(l) for l in open(out + "/ab.jsonl")]
for arm in ("base", "new", "nopdl"):
    r = [x["bench"] for x in rows if x["arm"] == arm and x["bench"]]
    v = sorted(x["value"] for x in r); k = [x["kernel_ms"] for x in r]; s = [x["ms_per_step"] for x in r]
    print(f"{arm:6s} value median {np.median(v):.0f} range {min(v):.0f}..{max(v):.0f}  ms_per_step {np.median(s):.5f}  "
          f"kernel_ms median {np.median(k):.5f} range {min(k):.5f}..{max(k):.5f}  hist_ok {all(x['hist_ok'] for x in r)}")
same = True
for f in sorted(glob.glob(out + "/dump_base/*.npy")):
    a, b = np.load(f), np.load(f.replace("dump_base", "dump_new"))
    eq = a.shape == b.shape and np.array_equal(a, b)
    same &= eq
    print("dump", os.path.basename(f), "identical" if eq else "DIFFERENT")
print("dump-outputs identical:", same)
for arm in ("base", "new"):
    try:
        d = json.loads(open(f"{out}/bench_{arm}.json").read().strip().splitlines()[-1])
        print(arm, "value", round(d["value"]), "ms_per_step", round(d["ms_per_step"], 5), "kernel_ms", round(d["roofline"]["kernel_ms"], 5),
              "parity_check", json.dumps(d["parity_check"]))
    except Exception as ex:
        print(arm, "bench line missing:", ex)
PY
rm -rf $OUT/dump_base $OUT/dump_new
