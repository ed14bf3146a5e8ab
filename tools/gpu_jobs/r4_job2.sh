#!/bin/bash
# round 4, job 2: the headline A/B of r4_job1.sh once more (parent / new alternating, three rounds of mfcc_exten and
# fwss_burg; r4_job1.sh's third new mfcc_exten run was 0.08 ms slower than its first two), then the default bench line,
# which r4_job1.sh ran out of time for
OUT=${1:?usage: r4_job2.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
B="python bench.py --steps 20 --warmup 3 --no-cpu-baseline --e2e-steps 0 --others none --no-selfcheck --cli-utts 0"
L=ctucopy_b200/libctucopy_b200.so
cp $L /tmp/new.so
show() { python - "$1" <<'P'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
print(sys.argv[1].split("/")[-1], round(d["ms_per_step"], 3), {k: round(v, 3) for k, v in d["kernel_ms_per_step"].items()}, "clock samples", d["clocks"]["samples"])
P
}
lib() { case $1 in parent) echo ctucopy_b200/lib_parent.so ;; new) echo /tmp/new.so ;; esac; }
use() { cp "$(lib $1)" $L; }
for r in 1 2 3; do
  for v in parent new; do
    use $v
    for w in mfcc_exten fwss_burg; do
      $B --workload $w > $OUT/r4b_${v}${r}_$w.json 2> $OUT/r4b_${v}${r}_$w.err; show $OUT/r4b_${v}${r}_$w.json
    done
  done
done
use new
python bench.py > $OUT/r4_bench_default.json 2> $OUT/r4_bench_default.err; echo "bench rc=$?"
python - "$OUT" <<'P'
import json, sys
d = json.loads(open(sys.argv[1] + "/r4_bench_default.json").read().strip().splitlines()[-1])
print("default bench", d.get("value"), d.get("ms_per_step"), "selfcheck", d.get("selfcheck"))
for k, v in (d.get("workloads") or {}).items():
    print("  ", k, v.get("ms_per_step"), v.get("selfcheck"))
P
