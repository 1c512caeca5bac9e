#!/bin/bash
# Builds lib variants/libbounds.so with -DQLB_BOUNDS_CHECK (every kernel tests the indices it is about to use and traps on the
# first one out of range) and runs the cross-kernel agreement script and the streaming / parity tests against it.
# compute-sanitizer is closed on the B200 pool (profiles/r02_compute_sanitizer_closed.log); this is its stand-in.
#   here (CPU box):  bash scripts/bounds_check_build.sh build
#   on the GPU box:  bash scripts/bounds_check_build.sh run > gpurun_out/bounds.log
set -e
cd "$(dirname "$0")/.."
if [ "$1" = build ]; then
  python -c 'from qkd_ldpc_b200 import build as b
b.build_library(force=True, verbose_ptxas=False, out=b.LIB_DIR / "variants" / "libbounds.so", extra_flags=["-DQLB_BOUNDS_CHECK", "-DQLB_STREAM_LEAN"])'
  ls -la qkd_ldpc_b200/lib/variants/libbounds.so
else
  export QLB_LIBRARY=$PWD/qkd_ldpc_b200/lib/variants/libbounds.so
  python scripts/sanitize_case.py
  python -m pytest tests/test_gpu_codes.py tests/test_gpu_parity.py -m gpu -q -x -k "(streaming and not other_bit_weights) or golden or waterfall_fp64 or edge_cases or no_clamp or multi_rate or storage_tiers or block_length"
fi
