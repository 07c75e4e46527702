#!/usr/bin/env bash
# Pair lists: the new GPU tests first, smoke(), tools/pair_lists.py, then the whole GPU suite. Evidence r07a_* under
# the output directory given as the first argument. (bench.py against the parent commit: tools/gpu_r7b.sh.)
cd "$(dirname "$0")/.."
OUT=$(realpath -m "${1:?usage: tools/gpu_r7a.sh OUT_DIR}")
mkdir -p "$OUT"
t0=$(date +%s)
el() { echo "[t+$(( $(date +%s) - t0 ))s] $*"; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r07a_smi.txt

timeout 900 python -m pytest tests/test_gpu_pair_lists.py -q -rs -p no:cacheprovider > $OUT/r07a_pytest_pair_lists.log 2>&1
rc=$?; el "new tests rc=$rc"; tail -4 $OUT/r07a_pytest_pair_lists.log | cut -c1-300
if [ $rc -ne 0 ]; then grep -E "^E |assert|Error|FAILED" $OUT/r07a_pytest_pair_lists.log | head -30 | cut -c1-300; fi

timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/r07a_smoke.txt 2>&1
el "smoke rc=$?"; tail -2 $OUT/r07a_smoke.txt | cut -c1-300

timeout 1200 python tools/pair_lists.py $OUT > $OUT/r07a_pair_lists.log 2>&1
el "pair_lists rc=$?"; tail -6 $OUT/r07a_pair_lists.log | cut -c1-700

timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_pair_lists.py > $OUT/r07a_pytest_gpu.log 2>&1
rc=$?; el "gpu suite rc=$rc"; tail -3 $OUT/r07a_pytest_gpu.log | cut -c1-300
if [ $rc -ne 0 ]; then grep -E "^E |FAILED" $OUT/r07a_pytest_gpu.log | head -30 | cut -c1-300; fi
