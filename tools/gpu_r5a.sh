#!/usr/bin/env bash
# Cross projection folded into the fused MLP kernel (mlp_ln_cproj): kernel tests first, then bench.py and the Hisfrag20
# model three times each, the op-level timing, the parity / retrieval numbers, the whole GPU suite, the timing-fuzz and
# bf16 suites and smoke(). Evidence r03a_* under the output directory given as the first argument; the A/B against
# the parent commit is tools/gpu_r5b.sh.
cd "$(dirname "$0")/.."
OUT=$(realpath -m "${1:?usage: tools/gpu_r5a.sh OUT_DIR}")
mkdir -p "$OUT"
t0=$(date +%s)
el() { echo "[t+$(( $(date +%s) - t0 ))s] $*"; }
NEW=$PWD/vit-ed_b200/lib/libvited_b200.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03a_smi.txt

timeout 400 python -m pytest tests/test_gpu_cproj_mlp.py -q -p no:cacheprovider > $OUT/r03a_pytest_cproj_mlp.log 2>&1
rc=$?; el "new kernel tests rc=$rc"; tail -3 $OUT/r03a_pytest_cproj_mlp.log | cut -c1-300
if [ $rc -ne 0 ]; then grep -E "^E |assert|Error" $OUT/r03a_pytest_cproj_mlp.log | head -20 | cut -c1-300; exit 1; fi

pz() {   # pz <tag> <lib> [extra args]
  local tag=$1 lib=$2; shift 2
  VITED_LIB=$lib timeout 200 python bench.py --no-cpu --no-extras "$@" > $OUT/r03a_bench_$tag.json 2> $OUT/r03a_bench_$tag.err
  local rc=$?
  python - <<PY
import json
try:
    d = json.load(open('$OUT/r03a_bench_$tag.json'))
    print('[puzzle $tag] rc=$rc value', round(d['value']), 'ms/step', round(d['ms_per_step'], 1), 'clocks', d['clocks'])
except Exception as ex:
    print('[puzzle $tag] rc=$rc no bench line', ex)
PY
}
pz new_1 $NEW; pz new_2 $NEW; pz new_3 $NEW
el "puzzle runs done"
hf() {
  local tag=$1 lib=$2
  VITED_LIB=$lib timeout 200 python bench.py --workload hisfrag --items 128 --steps 1 --warmup 1 > $OUT/r03a_hisfrag128_$tag.json 2> $OUT/r03a_hisfrag128_$tag.err
  local rc=$?
  python - <<PY
import json
try:
    d = json.load(open('$OUT/r03a_hisfrag128_$tag.json'))
    print('[hisfrag $tag] rc=$rc value', round(d['value']), 'clocks', d['clocks'])
except Exception as ex:
    print('[hisfrag $tag] rc=$rc no bench line', ex)
PY
}
hf new_1 $NEW; hf new_2 $NEW; hf new_3 $NEW
el "hisfrag runs done"

OPS=fused timeout 300 python tools/bench_ops.py > $OUT/r03a_bench_ops_fused.jsonl 2> $OUT/r03a_bench_ops_fused.err
el "bench_ops fused rc=$?"; cut -c1-200 $OUT/r03a_bench_ops_fused.jsonl

timeout 400 python -m pytest "tests/test_gpu_parity.py::test_sharp_attention_matches_oracle_on_the_production_shape" \
  "tests/test_gpu_retrieval.py::test_retrieval_top1_and_map_identical_to_three_decimals" -q -s -p no:cacheprovider \
  > $OUT/r03a_pytest_parity_retrieval.log 2>&1
el "parity + retrieval rc=$?"; grep -E "sharp attention|operand rounding|mAP|max \|logit|passed|failed" $OUT/r03a_pytest_parity_retrieval.log | cut -c1-300

timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider > $OUT/r03a_pytest_gpu.log 2>&1
el "pytest gpu rc=$?"; tail -3 $OUT/r03a_pytest_gpu.log | cut -c1-300
VITED_LIB=$PWD/tools/bin/jitter/libvited_b200.so timeout 600 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_cproj_mlp.py tests/test_gpu_parity.py tests/test_gpu_train.py -q -x -p no:cacheprovider > $OUT/r03a_pytest_jitter.log 2>&1
el "jitter rc=$?"; tail -2 $OUT/r03a_pytest_jitter.log | cut -c1-300
VITED_LIB=$PWD/tools/bin/bf16/libvited_b200.so timeout 600 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_cproj_mlp.py tests/test_gpu_parity.py tests/test_gpu_train.py -q -p no:cacheprovider > $OUT/r03a_pytest_bf16.log 2>&1
el "bf16 rc=$?"; tail -3 $OUT/r03a_pytest_bf16.log | cut -c1-300
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r03a_smoke.txt 2>&1
el "smoke rc=$?"; tail -2 $OUT/r03a_smoke.txt | cut -c1-300
