#!/bin/bash
# Builds the whole library with extra nvcc flags into qkd_ldpc_b200/lib/variants/lib<tag>.so (select with QLB_LIBRARY=<path>).
#   bash scripts/build_flag_variant.sh libm "-DQLB_F64_LIBM_FORMS -DQLB_STREAM_LEAN -DQLB_R64_LEAN"
set -e
cd "$(dirname "$0")/.."
TAG=$1; FLAGS=$2
python -c 'import sys
from qkd_ldpc_b200 import build as b
b.build_library(force=True, verbose_ptxas=False, out=b.LIB_DIR / "variants" / f"lib{sys.argv[1]}.so", extra_flags=sys.argv[2].split())' "$TAG" "$FLAGS"
ls -la qkd_ldpc_b200/lib/variants/lib$TAG.so
