#!/bin/bash
# round 3, job 1: k_frames2 / k_frames256 with the tile descriptors fetched ahead (cp.async into shared memory) and four
# samples per thread in the PCM staging, against the parent build (ctucopy_b200/lib_parent.so): alternating device-resident
# step times (three rounds for the headline, one for the other 512-point chains), the 8 kHz front end, output equality on all eight bench.py workloads, then the GPU suite and the default bench
OUT=${1:?usage: r3_job1.sh OUTPUT_DIR}
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
use() { cp $1 $L; }
for r in 1 2 3; do
  for v in parent new; do
    if [ $v = parent ]; then use ctucopy_b200/lib_parent.so; else use /tmp/new.so; fi
    ws=mfcc_exten; [ $r = 1 ] && ws="mfcc_exten mfcc_d_a plp trapdct exten fwss_burg"
    for w in $ws; do
      $B --workload $w > $OUT/r3_${v}${r}_$w.json 2> $OUT/r3_${v}${r}_$w.err; show $OUT/r3_${v}${r}_$w.json
    done
  done
done
T="python tools/time_args.py 4000 --"
for v in parent new; do
  if [ $v = parent ]; then use ctucopy_b200/lib_parent.so; else use /tmp/new.so; fi
  echo "== 8 kHz mfcc d_a ($v)"; $T -fs 8000 -format_in raw -preset mfcc -preem 0.97 -fea_delta d_a -format_out htk 2>&1 | grep -E "k_frames<pcm|total|frames/s" | head -4
done
for v in parent new; do
  if [ $v = parent ]; then use ctucopy_b200/lib_parent.so; else use /tmp/new.so; fi
  for w in mfcc_exten mfcc_d_a plp trapdct exten fwss_burg tdiir mfcc_trap5; do
    python bench.py --workload $w --steps 2 --warmup 1 --no-cpu-baseline --e2e-steps 0 --others none --no-selfcheck --cli-utts 0 \
      --dump-outputs /tmp/dump_$v/$w > /dev/null 2> $OUT/r3_dump_${v}_$w.err || echo "dump $v $w failed"
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
use /tmp/new.so
python -m pytest tests -m gpu -q > $OUT/r3_pytest_gpu.log 2>&1; echo "pytest gpu rc=$?"; tail -3 $OUT/r3_pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
python bench.py > $OUT/r3_bench_default.json 2> $OUT/r3_bench_default.err; echo "bench rc=$?"
python - "$OUT" <<'P'
import json, sys
d = json.loads(open(sys.argv[1] + "/r3_bench_default.json").read().strip().splitlines()[-1])
print("default bench", d.get("value"), d.get("ms_per_step"), "selfcheck", d.get("selfcheck"))
for k, v in (d.get("workloads") or {}).items():
    print("  ", k, v.get("ms_per_step"), v.get("selfcheck"))
P
