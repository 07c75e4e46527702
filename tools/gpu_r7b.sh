#!/usr/bin/env bash
# bench.py of this tree against the parent commit's tree (its own Python binding and library, since the binding of
# this tree also binds vited_score_pairs), alternating, puzzle and Hisfrag20 128 fragments, with --dump-outputs
# compared. Evidence r07b_* under the output directory given as the first argument; the parent commit's tree, with its
# library built, is the second argument.
cd "$(dirname "$0")/.."
OUT=$(realpath -m "${1:?usage: tools/gpu_r7b.sh OUT_DIR PARENT_TREE}")
OLD=$(realpath "${2:?usage: tools/gpu_r7b.sh OUT_DIR PARENT_TREE}")
NEW=$PWD
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r07b_smi.txt
b() {   # b <tag> <tree> [extra args]
  local tag=$1 tree=$2; shift 2
  mkdir -p $OUT/dump_$tag
  (cd $tree && timeout 400 python bench.py --gpus 1 --dump-outputs $OUT/dump_$tag "$@" > $OUT/r07b_bench_$tag.json 2> $OUT/r07b_bench_$tag.err)
  echo "[$tag] rc=$? $(cut -c1-200 $OUT/r07b_bench_$tag.json)"
}
b pz_new_1 $NEW --steps 10 --warmup 3; b pz_old_1 $OLD --steps 10 --warmup 3
b pz_new_2 $NEW --steps 10 --warmup 3; b pz_old_2 $OLD --steps 10 --warmup 3
b pz_new_3 $NEW --steps 10 --warmup 3; b pz_old_3 $OLD --steps 10 --warmup 3
b hf_new_1 $NEW --workload hisfrag --items 128 --steps 2 --warmup 1; b hf_old_1 $OLD --workload hisfrag --items 128 --steps 2 --warmup 1
python - > $OUT/r07b_dump_compare.txt <<PY
import glob, os
import numpy as np
for w in ('pz', 'hf'):
    for f in sorted(glob.glob('$OUT/dump_%s_new_1/*.npy' % w)):
        a = np.load(f); b = np.load(f.replace('_new_1', '_old_1'))
        print(w, os.path.basename(f), a.shape, 'bit-identical' if np.array_equal(a, b) else 'max abs diff %g' % np.abs(a - b).max())
PY
cat $OUT/r07b_dump_compare.txt; rm -rf $OUT/dump_*
