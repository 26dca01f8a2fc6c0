#!/bin/bash
# Build instrumented variants of liblirec_b200.so into variants/<name>.so (git-ignored), then restore the default
# build.  The one such variant is the in-kernel GEMM trace that tools/gemm_trace.py reads:
#   bash tools/build_variants.sh "trace:-DLIREC_GEMM_TRACE=1"
set -e
cd "$(dirname "$0")/.."
rm -rf variants
mkdir -p variants
build() {   # name, defines
  LIREC_NVCC_DEFINES="$2" python -m lirec_b200.build --force > /dev/null
  cp lirec_b200/liblirec_b200.so variants/$1.so
  echo "built variants/$1.so  [$2]"
}
build default ""
for spec in "$@"; do
  build "${spec%%:*}" "${spec#*:}"
done
python -m lirec_b200.build --force > /dev/null    # the default build is what ships
