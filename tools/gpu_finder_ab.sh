#!/bin/bash
# One GPU visit for a compress-finder change: the finder cycle account of two stats builds, compress_kernel A/B of two
# product builds, bench.py alternated (three runs each), output parity (bench.py --dump-outputs), the GPU suite (plain,
# and with the compact kernel forced) and smoke, all with the second build.
# usage: tools/gpu_finder_ab.sh A.so B.so A_stats.so B_stats.so [OUT]
#   B = the build under test, installed as the package's; logs and dumps go to OUT (default build/finder_ab)
A=$1; B=$2; AS=$3; BS=$4; OUT=${5:-build/finder_ab}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/card.txt" 2>&1; cat "$OUT/card.txt"
timeout 900 python -m pytest -q -m gpu tests/test_gpu_retest_exits.py > "$OUT/pytest_exits.log" 2>&1; echo "new tests rc=$?"; tail -3 "$OUT/pytest_exits.log"
timeout 600 python tools/finder_stats.py "$AS" "$BS" > "$OUT/finder_exits.txt" 2>&1; echo "finder_stats rc=$?"
timeout 900 python tools/compress_ab.py "$A" "$B" > "$OUT/compress_ab.txt" 2>&1; echo "compress_ab rc=$?"; cat "$OUT/compress_ab.txt"
BENCH="python bench.py --gpus 1 --steps 20 --warmup 3 --no-cpu --no-extras"
for r in 1 2 3; do
  for who in parent new; do
    lib=$A; [ $who = new ] && lib=$B
    extra=""; [ $r = 1 ] && extra="--dump-outputs $OUT/dump_$who"
    B200LZ4_LIB=$lib timeout 600 $BENCH $extra > "$OUT/bench_${who}_$r.json" 2> "$OUT/bench_${who}_$r.err"
    echo "bench $who $r rc=$? $(BENCH_JSON="$OUT/bench_${who}_$r.json" python -c "import json, os; d = json.loads(open(os.environ['BENCH_JSON']).read().strip().splitlines()[-1]); r = d.get('roofline', {}); print(d.get('value'), r.get('kernel_ms'), r.get('compact_ms'))" 2>&1)"
  done
done
OUT="$OUT" python - <<'EOF'
import glob, os, numpy as np
out = os.environ["OUT"]
a = sorted(os.path.basename(p) for p in glob.glob(f"{out}/dump_parent/*.npy"))
b = sorted(os.path.basename(p) for p in glob.glob(f"{out}/dump_new/*.npy"))
same = a == b and all(np.array_equal(np.load(f"{out}/dump_parent/{f}"), np.load(f"{out}/dump_new/{f}")) for f in a)
print(f"dump-outputs: {len(a)} / {len(b)} files, {'identical' if same else 'DIFFER'}")
EOF
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "suite rc=$?"; tail -3 "$OUT/pytest_gpu.log"
B200LZ4_NO_WIDE=1 B200LZ4_COMPACT=1 timeout 1500 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu_compact.log" 2>&1; echo "suite (NO_WIDE COMPACT) rc=$?"; tail -3 "$OUT/pytest_gpu_compact.log"
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?"; tail -1 "$OUT/smoke.log"
