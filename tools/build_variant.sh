#!/bin/bash
# build_variant.sh NAME [GIT_REV] [extra nvcc flags]: compile the CUDA library of the working tree (GIT_REV = "-") or of a
# commit into variants/libsnk_NAME.so for A/B timing on one box (SNK_LIB=variants/libsnk_NAME.so python tools/ab.py ...).
# Either way the working tree's __graft_entry__.build_library compiles it.
set -e
cd "$(dirname "$0")/.."
name=$1; rev=${2:--}; shift; shift || true
src=$PWD
if [ "$rev" != "-" ]; then
  src=$(mktemp -d /tmp/snk_variant_XXXX)
  trap 'rm -rf "$src"' EXIT
  git archive "$rev" snakes_b200/csrc include | tar -x -C "$src"
fi
mkdir -p variants
python3 -c 'import sys, __graft_entry__ as g; g.build_library(sys.argv[1], sys.argv[2], sys.argv[3:])' "$src" "variants/libsnk_$name.so" "$@"
echo built variants/libsnk_$name.so
