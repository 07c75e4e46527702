#!/usr/bin/env bash
# After the removal of the experimental kernel variants and the kernel-selecting environment switches: the GPU test
# suite and smoke() on this tree, then bench.py of this tree against the parent commit's tree, alternating (puzzle 3x,
# Hisfrag20 128 fragments 2x, training 2x), with --dump-outputs compared bit for bit. Evidence r08a_* under the output
# directory given as the first argument; the parent commit's tree, with its library built, is the second argument.
cd "$(dirname "$0")/.."
OUT=$(realpath -m "${1:?usage: tools/gpu_r8a.sh OUT_DIR PARENT_TREE}")
OLD=$(realpath "${2:?usage: tools/gpu_r8a.sh OUT_DIR PARENT_TREE}")
NEW=$PWD
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r08a_smi.txt
timeout 1500 python -m pytest -q -p no:cacheprovider tests > $OUT/r08a_pytest.txt 2>&1
echo "pytest rc=$? $(tail -1 $OUT/r08a_pytest.txt)"
timeout 300 python -m pytest -q -s -p no:cacheprovider tests/test_gpu_score_kernels.py -k attention_cls \
  > $OUT/r08a_pytest_cls.txt 2>&1
echo "pytest attention_cls rc=$? $(tail -1 $OUT/r08a_pytest_cls.txt)"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r08a_smoke.txt 2>&1
echo "smoke rc=$? $(tail -1 $OUT/r08a_smoke.txt)"
b() {   # b <tag> <tree> [extra args]
  local tag=$1 tree=$2; shift 2
  mkdir -p $OUT/dump_$tag
  (cd $tree && timeout 400 python bench.py --gpus 1 --dump-outputs $OUT/dump_$tag "$@" > $OUT/r08a_bench_$tag.json 2> $OUT/r08a_bench_$tag.err)
  echo "[$tag] rc=$? $(cut -c1-200 $OUT/r08a_bench_$tag.json)"
}
PZ="--steps 10 --warmup 3"; HF="--workload hisfrag --items 128 --steps 2 --warmup 1"; TR="--workload train --steps 3 --warmup 2"
b pz_new_1 $NEW $PZ; b pz_old_1 $OLD $PZ
b pz_new_2 $NEW $PZ; b pz_old_2 $OLD $PZ
b pz_new_3 $NEW $PZ; b pz_old_3 $OLD $PZ
b hf_new_1 $NEW $HF; b hf_old_1 $OLD $HF
b hf_new_2 $NEW $HF; b hf_old_2 $OLD $HF
b tr_new_1 $NEW $TR; b tr_old_1 $OLD $TR
b tr_new_2 $NEW $TR; b tr_old_2 $OLD $TR
python - > $OUT/r08a_dump_compare.txt <<PY
import glob, os
import numpy as np
for w in ('pz', 'hf', 'tr'):
    runs = sorted(glob.glob('$OUT/dump_%s_*' % w))
    ref = '$OUT/dump_%s_old_1' % w
    for f in sorted(glob.glob(ref + '/*.npy')):
        a = np.load(f)
        for r in runs:
            if r == ref:
                continue
            g = os.path.join(r, os.path.basename(f))
            b = np.load(g) if os.path.exists(g) else None
            same = b is not None and a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()
            print(w, os.path.basename(r), os.path.basename(f), a.shape,
                  'bit-identical' if same else ('missing' if b is None else 'max abs diff %g' % np.nanmax(np.abs(a.astype(np.float64) - b.astype(np.float64)))))
PY
cat $OUT/r08a_dump_compare.txt; rm -rf $OUT/dump_*
