#!/usr/bin/env bash
# Installs the UNMODIFIED reference into baseline/_ref/ (git-ignored; it travels to the GPU
# box with the gpurun snapshot, like a `pip install --target baseline/_ref` would):
#   baseline/_ref/gsplatcu*.so   the reference's CUDA extension (gsplatcu/setup.py:4-14) built
#                                for sm_100a -- benchmarks/compare_ref_gpu.py times it next to
#                                ours on the same B200 ("B-REF-GPU" in BASELINE.md)
#   baseline/_ref/py/            the reference's pure-Python package gsplat/, train.py and its
#                                forward_gpu.py / backward_gpu.py / backward_cpu.py / forward_cpu.py, so
#                                benchmarks/train_reference.py and run_reference_scripts.py can run the
#                                reference's own scripts (BASELINE config 3, the 19-line [OK] parity
#                                script) on either gsplatcu
# The reference tree is read-only, so the build runs from a scratch copy under /tmp.  No
# reference source enters this repository's history.  Only runs where /root/reference exists
# (the dev container).   usage: build_ref_gpu.sh [py]   ("py": only refresh baseline/_ref/py)
set -euo pipefail
REF=${REF:-/root/reference}
OUT="$(cd "$(dirname "$0")" && pwd)/_ref"
[ -d "$REF/gsplatcu" ] || { echo "no reference tree at $REF - skipping"; exit 0; }
mkdir -p "$OUT/py"
rm -rf "$OUT/py/gsplat"
cp -r "$REF/gsplat" "$OUT/py/gsplat"
cp "$REF/train.py" "$OUT/py/train.py"
# the reference's own parity / inference scripts (benchmarks/run_reference_scripts.py runs them unmodified)
for f in forward_gpu.py backward_gpu.py backward_cpu.py forward_cpu.py; do cp "$REF/$f" "$OUT/py/$f"; done
find "$OUT/py" -name __pycache__ -prune -exec rm -rf {} +
if [ "${1:-}" = "py" ]; then ls "$OUT" "$OUT/py"; exit 0; fi
TMP=$(mktemp -d)
# the copied sources keep the reference tree's read-only modes: make them removable on exit
trap 'chmod -R u+w "$TMP"; rm -rf "$TMP"' EXIT
cp -r "$REF/gsplatcu" "$TMP/src"
cd "$TMP/src"
TORCH_CUDA_ARCH_LIST="10.0a" MAX_JOBS=4 python setup.py build_ext --build-lib "$OUT" --build-temp "$TMP/build" > "$TMP/build.log" 2>&1 \
  || { tail -30 "$TMP/build.log"; exit 1; }
ls -la "$OUT"
