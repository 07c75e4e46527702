#!/usr/bin/env bash
# Builds the C-ABI shared library for sm_100a (cross-compiles without a GPU).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${VITED_OUT_DIR:-$HERE/../lib}"   # VITED_OUT_DIR / VITED_EXTRA_FLAGS: variant builds (trace points, bf16 operands)
mkdir -p "$OUT"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
"$NVCC" -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --threads 4 \
  -Xcompiler -fPIC -Xcompiler -fvisibility=hidden -shared -cudart static \
  ${VITED_PTXAS_V:+-Xptxas -v} ${VITED_EXTRA_FLAGS:-} \
  -o "$OUT/libvited_b200.so" \
  "$HERE/engine.cu" "$HERE/gemm_tc.cu" "$HERE/gemm_ln.cu" "$HERE/mlp_ln.cu" "$HERE/attention.cu" "$HERE/attention_tc.cu" "$HERE/attention_pair.cu" "$HERE/rowops.cu" "$HERE/pair_lists.cu" "$HERE/train_ops.cu" "$HERE/train_attn.cu" "$HERE/train_optim.cu" "$HERE/solver_tables.cu" "$HERE/piece_prep.cu" "$HERE/retrieval_metrics.cu"
echo "built $OUT/libvited_b200.so"
