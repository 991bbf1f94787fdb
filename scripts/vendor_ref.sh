#!/bin/bash
# Copies the UNMODIFIED reference (its Python sources and configs; 0.8 MB) into baseline/_ref/, where the tests and the
# benchmark find it:  scripts/vendor_ref.sh /path/to/DANBO-pytorch.  baseline/_ref/ is git-ignored (never committed).
# Used only as the measured baseline (bench.py --impl reference, cpu_baseline kind "reference") and as the caller in
# the drop-in tests (tests/test_gpu_dropin.py); nothing in the product imports it.
set -eu
SRC=${1:?usage: scripts/vendor_ref.sh /path/to/DANBO-pytorch}
ROOT=$(cd "$(dirname "$0")/.." && pwd)
DST=$ROOT/baseline/_ref
[ -d "$SRC/core" ] || { echo "no reference at $SRC"; exit 0; }
mkdir -p "$DST"
rm -rf "$DST/core" "$DST/configs"
cp -r "$SRC/core" "$SRC/configs" "$DST/"
cp "$SRC/run_nerf.py" "$SRC/run_render.py" "$DST/"
find "$DST" -name __pycache__ -type d -prune -exec rm -rf {} +
(cd "$SRC" && find core configs run_nerf.py run_render.py -type f ! -path '*/__pycache__/*' -exec sha256sum {} + | sort -k2) > "$DST/SHA256SUMS"
echo "vendored $(find "$DST" -type f | wc -l) files into $DST"
