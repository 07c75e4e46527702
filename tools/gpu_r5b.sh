#!/usr/bin/env bash
# A/B of the cross projection folded into the fused MLP kernel against the parent commit: the parent runs from its own
# tree (tools/bin/parent_tree/: the parent's sources and its library, built separately; its C-ABI lacks the new entry
# point, so it cannot be loaded through this tree's bindings). bench.py alternating, four runs each, the output dumps
# of both, the Hisfrag20 model alternating, three runs each. Evidence r03b_* under the output directory given as the
# first argument.
cd "$(dirname "$0")/.."
ROOT=$PWD
OUT=$(realpath -m "${1:?usage: tools/gpu_r5b.sh OUT_DIR}")
mkdir -p "$OUT"
t0=$(date +%s)
el() { echo "[t+$(( $(date +%s) - t0 ))s] $*"; }
OLD=$ROOT/tools/bin/parent_tree
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03b_smi.txt
show() {
  python - "$@" <<'PY'
import json, sys
tag, rc, f = sys.argv[1:4]
try:
    d = json.load(open(f))
    print(f'[{tag}] rc={rc} value', round(d['value']), 'clocks', d['clocks'])
except Exception as ex:
    print(f'[{tag}] rc={rc} no bench line', ex)
PY
}
pz() {   # pz <tag> <tree> [extra args]
  local tag=$1 tree=$2; shift 2
  (cd $tree && timeout 200 python bench.py --no-cpu --no-extras "$@" > $OUT/r03b_bench_$tag.json 2> $OUT/r03b_bench_$tag.err)
  show puzzle_$tag $? $OUT/r03b_bench_$tag.json
}
pz new_1 $ROOT; pz old_1 $OLD; pz new_2 $ROOT; pz old_2 $OLD
pz new_3 $ROOT --dump-outputs $OUT/r03b_dump_new; pz old_3 $OLD --dump-outputs $OUT/r03b_dump_old
pz new_4 $ROOT; pz old_4 $OLD
el "puzzle A/B done"
python - "$OUT" <<'PY' | tee $OUT/r03b_dump_compare.txt
import glob, os, sys
import numpy as np
for f in sorted(glob.glob(os.path.join(sys.argv[1], 'r03b_dump_new', '*.npy'))):
    a = np.load(f).astype(np.float64); b = np.load(f.replace('dump_new', 'dump_old')).astype(np.float64)
    d = np.abs(a - b)
    print(os.path.basename(f), a.shape, 'max |dlogit|', d.max(), 'mean', d.mean(),
          'argmax agreement (last axis)', (a.argmax(-1) == b.argmax(-1)).mean(),
          'argmax agreement (axis 1)', (a.argmax(1) == b.argmax(1)).mean())
PY
hf() {
  local tag=$1 tree=$2
  (cd $tree && timeout 200 python bench.py --workload hisfrag --items 128 --steps 1 --warmup 1 > $OUT/r03b_hisfrag128_$tag.json 2> $OUT/r03b_hisfrag128_$tag.err)
  show hisfrag_$tag $? $OUT/r03b_hisfrag128_$tag.json
}
hf new_1 $ROOT; hf old_1 $OLD; hf new_2 $ROOT; hf old_2 $OLD; hf new_3 $ROOT; hf old_3 $OLD
el "hisfrag A/B done"
