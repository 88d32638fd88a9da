#!/bin/bash
# Fused transition kernel on one box: card + power limit, its GPU tests, per-launch times (tools/ff_times.py), then the C2
# forward alternating the fused kernel on / off (AF2_FF_FUSED) for PAIRS pairs, and C3 / C4 once per path.
# usage: [OUT=dir] tools/gpu_ff_ab.sh [tag] [pairs]      (results under $OUT, default ab_out/)
TAG=${1:-ff}; PAIRS=${2:-5}; OUT=${OUT:-ab_out}
mkdir -p $OUT
L=$OUT/ab_${TAG}.log
: > $L
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader >> $L
timeout 300 python -m pytest -q -m gpu -s tests/test_gpu_ff_fused.py > $OUT/test_ff_fused.txt 2>&1
rc=$?
echo "test_gpu_ff_fused exit $rc" >> $L
grep -E "fused vs two-launch" $OUT/test_ff_fused.txt >> $L
tail -3 $OUT/test_ff_fused.txt >> $L
[ $rc -eq 0 ] || { tail -40 $OUT/test_ff_fused.txt; cat $L; exit 1; }
timeout 300 python tools/ff_times.py >> $L 2>&1
run_bench() {
  local label=$1; shift
  env "$@" timeout 300 python bench.py --steps 20 --warmup 5 --no-cpu-baseline ${WL:+--workload $WL} ${DUMP:+--dump-outputs $DUMP} > $OUT/ab_tmp.json 2> $OUT/ab_tmp.err
  python - "$label" "$OUT" <<'PY' >> $L
import json, sys
try:
    d = json.loads([l for l in open(sys.argv[2] + '/ab_tmp.json') if l.startswith('{')][-1])
    print(sys.argv[1], 'ms_per_step', round(d['ms_per_step'], 3), 'e2e_ms', round(d['e2e']['ms_per_step'], 3),
          [(k['name'][:10], round(k['ms_per_step'], 3)) for k in d['kernel_classes']])
except Exception as e:
    print(sys.argv[1], 'FAILED', e, open(sys.argv[2] + '/ab_tmp.err').read()[-600:])
PY
}
DUMP=$OUT/dump_fused run_bench C2_fused_0 AF2_FF_FUSED=1
DUMP=$OUT/dump_two_launch run_bench C2_two_launch_0 AF2_FF_FUSED=0
python - "$OUT" <<'PY' >> $L
import sys
import numpy as np
for n in ("pair", "msa", "distogram"):
    a = np.load(f"{sys.argv[1]}/dump_fused/{n}.npy").astype(np.float64)
    b = np.load(f"{sys.argv[1]}/dump_two_launch/{n}.npy").astype(np.float64)
    print(f"dump {n}: max |fused - two_launch| {np.abs(a - b).max():.3e}, rms {np.sqrt((b ** 2).mean()):.3e}")
PY
rm -rf $OUT/dump_fused $OUT/dump_two_launch
for i in $(seq 1 $PAIRS); do
  run_bench C2_fused_$i AF2_FF_FUSED=1
  run_bench C2_two_launch_$i AF2_FF_FUSED=0
done
for wl in C3 C4; do
  WL=$wl run_bench ${wl}_fused AF2_FF_FUSED=1
  WL=$wl run_bench ${wl}_two_launch AF2_FF_FUSED=0
done
cat $L
