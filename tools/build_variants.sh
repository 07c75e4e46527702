#!/usr/bin/env bash
# Variant builds of the C-ABI library used by the A/B and robustness runs (git-ignored, under tools/bin/<variant>/):
#   bf16    -DVITED_ACT_BF16=1                      bf16 operands instead of fp16 (tools/gpu_fp16.sh, tests/analysis/*)
#   jitter  -DVITED_JITTER                          random 0..4 us sleeps in front of mbarrier waits (timing fuzzer)
#   trace   -DVITED_LN_TRACE -DVITED_ATTN_TRACE     clock64 trace points (tools/trace_*.py)
# Select one with VITED_LIB=$PWD/tools/bin/<variant>/libvited_b200.so
set -euo pipefail
cd "$(dirname "$0")/.."
VITED_OUT_DIR=$PWD/tools/bin/bf16 VITED_EXTRA_FLAGS="-DVITED_ACT_BF16=1" bash vit-ed_b200/csrc/build.sh
VITED_OUT_DIR=$PWD/tools/bin/jitter VITED_EXTRA_FLAGS="-DVITED_JITTER" bash vit-ed_b200/csrc/build.sh
VITED_OUT_DIR=$PWD/tools/bin/trace VITED_EXTRA_FLAGS="-DVITED_LN_TRACE -DVITED_ATTN_TRACE -DVITED_MLP_TRACE" bash vit-ed_b200/csrc/build.sh
