#!/usr/bin/env bash
# uint8 fragment grid + column-state windows: the new GPU tests first, smoke(), the whole GPU suite, bench.py against
# the parent commit's library (alternating, puzzle and Hisfrag20 128 fragments, with --dump-outputs compared), then
# tools/fragment_scale.py. Evidence r06a_* under the output directory given as the first argument; the parent library
# is the second argument (built from the parent commit with VITED_OUT_DIR).
cd "$(dirname "$0")/.."
OUT=$(realpath -m "${1:?usage: tools/gpu_r6a.sh OUT_DIR PARENT_LIB}")
OLD=$(realpath "${2:?usage: tools/gpu_r6a.sh OUT_DIR PARENT_LIB}")
NEW=$PWD/vit-ed_b200/lib/libvited_b200.so
mkdir -p "$OUT"
t0=$(date +%s)
el() { echo "[t+$(( $(date +%s) - t0 ))s] $*"; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r06a_smi.txt

timeout 900 python -m pytest tests/test_gpu_fragment_scale.py -q -rs -p no:cacheprovider > $OUT/r06a_pytest_fragment_scale.log 2>&1
rc=$?; el "new tests rc=$rc"; tail -4 $OUT/r06a_pytest_fragment_scale.log | cut -c1-300
if [ $rc -ne 0 ]; then grep -E "^E |assert|Error|FAILED" $OUT/r06a_pytest_fragment_scale.log | head -30 | cut -c1-300; fi

timeout 300 python -c 'import __graft_entry__ as g; g.smoke()' > $OUT/r06a_smoke.txt 2>&1
el "smoke rc=$?"; tail -2 $OUT/r06a_smoke.txt | cut -c1-300

timeout 1500 python -m pytest tests -q -m gpu -p no:cacheprovider --deselect tests/test_gpu_fragment_scale.py > $OUT/r06a_pytest_gpu.log 2>&1
rc=$?; el "gpu suite rc=$rc"; tail -3 $OUT/r06a_pytest_gpu.log | cut -c1-300
if [ $rc -ne 0 ]; then grep -E "^E |FAILED" $OUT/r06a_pytest_gpu.log | head -30 | cut -c1-300; fi

b() {   # b <tag> <lib> [extra args]
  local tag=$1 lib=$2; shift 2
  mkdir -p $OUT/dump_$tag
  VITED_LIB=$lib timeout 400 python bench.py --gpus 1 --dump-outputs $OUT/dump_$tag "$@" > $OUT/r06a_bench_$tag.json 2> $OUT/r06a_bench_$tag.err
  echo "[$tag] rc=$? $(cut -c1-200 $OUT/r06a_bench_$tag.json)"
}
b pz_new_1 $NEW --steps 10 --warmup 3; b pz_old_1 $OLD --steps 10 --warmup 3
b pz_new_2 $NEW --steps 10 --warmup 3; b pz_old_2 $OLD --steps 10 --warmup 3
b hf_new_1 $NEW --workload hisfrag --items 128 --steps 2 --warmup 1; b hf_old_1 $OLD --workload hisfrag --items 128 --steps 2 --warmup 1
b hf_new_2 $NEW --workload hisfrag --items 128 --steps 2 --warmup 1; b hf_old_2 $OLD --workload hisfrag --items 128 --steps 2 --warmup 1
python - > $OUT/r06a_dump_compare.txt <<PY
import glob, os
import numpy as np
for w in ('pz', 'hf'):
    for f in sorted(glob.glob('$OUT/dump_%s_new_1/*.npy' % w)):
        a = np.load(f); b = np.load(f.replace('_new_1', '_old_1'))
        print(w, os.path.basename(f), a.shape, 'bit-identical' if np.array_equal(a, b) else 'max abs diff %g' % np.abs(a - b).max())
PY
cat $OUT/r06a_dump_compare.txt; rm -rf $OUT/dump_*
el "bench done"

timeout 1200 python tools/fragment_scale.py $OUT > $OUT/r06a_fragment_scale.log 2>&1
el "fragment_scale rc=$?"; tail -6 $OUT/r06a_fragment_scale.log | cut -c1-600
