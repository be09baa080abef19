#!/bin/sh
# Builds the reference's UNMODIFIED KITTI scorer (src/dataset/kitti-eval/cpp/evaluate_object.cpp,
# recipe = its own one-line Makefile: `g++ -Wall -Wno-sign-compare`) from the sources where they
# lie in the reference checkout, into OUT_DIR (default oracle/_ref, where __graft_entry__.build()
# puts it and squeezedet_b200/eval.py shells out to it, mirroring src/dataset/kitti.py:129-136).
# No reference source is copied into this repo; the binary is git-ignored.
# Usage: oracle/build_kitti_eval.sh [/path/to/reference [OUT_DIR]]
set -e
REF="${1:-$SQDET_REFERENCE}"
SRC="$REF/src/dataset/kitti-eval/cpp/evaluate_object.cpp"
HERE="$(cd "$(dirname "$0")/.." && pwd)"
OUT="${2:-$HERE/oracle/_ref}"
if [ ! -f "$SRC" ]; then
  echo "build_kitti_eval: $SRC not found (pass the reference checkout as the first argument)" >&2
  exit 2
fi
mkdir -p "$OUT"
g++ -O2 -Wall -Wno-sign-compare -Wno-unused-variable -Wno-unused-result \
    -I "$REF/src/dataset/kitti-eval/cpp" -o "$OUT/evaluate_object" "$SRC"
echo "built $OUT/evaluate_object"
