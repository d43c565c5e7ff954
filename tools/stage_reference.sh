#!/usr/bin/env bash
# Stage the UNMODIFIED reference checkout next to the repo so that it travels to the GPU box with the gpurun
# snapshot (baseline/_ref/ is git-ignored but NOT gpurun-ignored: nothing of the reference enters the history).
#
#   tools/stage_reference.sh [/root/reference]
#
# Result: baseline/_ref/HairFastGAN/   byte-for-byte copy of the checkout (no edits; verified with diff -r)
#         baseline/_ref/ext/           the reference's two JIT extensions (op/fused_act.py:10-16,
#                                      op/upfirdn2d.py:10-16) prebuilt for sm_100a by baseline/build_ref_ext.py so the
#                                      GPU box does not spend 2.5 min of nvcc per process on them
# The staged tree is what `bench.py --impl reference`, `bench.py`'s `reference_gpu` leg and baseline/run_swap.py run.
set -euo pipefail
SRC="${1:-/root/reference}"
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
DST="$ROOT/baseline/_ref/HairFastGAN"
if [ ! -d "$SRC/models" ]; then echo "no reference checkout at $SRC" >&2; exit 1; fi
mkdir -p "$ROOT/baseline/_ref"
rm -rf "$DST.tmp"
cp -r "$SRC" "$DST.tmp"
find "$DST.tmp" -name '__pycache__' -type d -prune -exec rm -rf {} +
rm -rf "$DST"
mv "$DST.tmp" "$DST"
diff -r -q "$SRC" "$DST" -x __pycache__ >/dev/null && echo "staged $SRC -> $DST (identical)"
python "$ROOT/baseline/build_ref_ext.py"
