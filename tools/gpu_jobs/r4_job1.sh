#!/bin/bash
# round 4, job 1: k_bank with the fused noise-reduction scan on bin pairs (nr_step2, packed FP32, LDS.64 / STS.64) and the
# DCT two cepstral rows per pass over the band vector (new), against the parent build (ctucopy_b200/lib_parent.so, built
# from the parent commit) and the bin-pair scan alone (ctucopy_b200/lib_pairs.so, this tree with the parent's DCT loop):
# alternating device-resident step times (three rounds of the MFCC chains, one of the other 512-point chains), output
# equality on all eight bench.py workloads, then the GPU suite, smoke() and the default bench
OUT=${1:?usage: r4_job1.sh OUTPUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
B="python bench.py --steps 20 --warmup 3 --no-cpu-baseline --e2e-steps 0 --others none --no-selfcheck --cli-utts 0"
L=ctucopy_b200/libctucopy_b200.so
cp $L /tmp/new.so
show() { python - "$1" <<'P'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
print(sys.argv[1].split("/")[-1], round(d["ms_per_step"], 3), {k: round(v, 3) for k, v in d["kernel_ms_per_step"].items()})
P
}
lib() { case $1 in parent) echo ctucopy_b200/lib_parent.so ;; pairs) echo ctucopy_b200/lib_pairs.so ;; new) echo /tmp/new.so ;; esac; }
use() { cp "$(lib $1)" $L; }
for r in 1 2 3; do
  for v in parent pairs new; do
    use $v
    ws="mfcc_exten mfcc_d_a"; [ $r = 1 ] && ws="mfcc_exten mfcc_d_a plp trapdct exten fwss_burg"
    for w in $ws; do
      $B --workload $w > $OUT/r4_${v}${r}_$w.json 2> $OUT/r4_${v}${r}_$w.err; show $OUT/r4_${v}${r}_$w.json
    done
  done
done
for v in parent new; do
  use $v
  for w in mfcc_exten mfcc_d_a plp trapdct exten fwss_burg tdiir mfcc_trap5; do
    python bench.py --workload $w --steps 2 --warmup 1 --no-cpu-baseline --e2e-steps 0 --others none --no-selfcheck --cli-utts 0 \
      --dump-outputs /tmp/dump_$v/$w > /dev/null 2> $OUT/r4_dump_${v}_$w.err || echo "dump $v $w failed"
  done
done
python - <<'P'
import glob, os, numpy as np
for d in sorted(glob.glob("/tmp/dump_parent/*")):
    w = os.path.basename(d)
    for f in sorted(glob.glob(d + "/*.npy")):
        a = np.load(f); b = np.load(f.replace("dump_parent", "dump_new"))
        print("dump", w, os.path.basename(f), a.shape, "array_equal" if np.array_equal(a, b) else "DIFFERENT")
P
use new
python -m pytest tests -m gpu -q > $OUT/r4_pytest_gpu.log 2>&1; echo "pytest gpu rc=$?"; tail -3 $OUT/r4_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
python bench.py > $OUT/r4_bench_default.json 2> $OUT/r4_bench_default.err; echo "bench rc=$?"
python - "$OUT" <<'P'
import json, sys
d = json.loads(open(sys.argv[1] + "/r4_bench_default.json").read().strip().splitlines()[-1])
print("default bench", d.get("value"), d.get("ms_per_step"), "selfcheck", d.get("selfcheck"))
for k, v in (d.get("workloads") or {}).items():
    print("  ", k, v.get("ms_per_step"), v.get("selfcheck"))
P
