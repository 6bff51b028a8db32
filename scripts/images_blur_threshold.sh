#!/bin/bash
# Evidence for the fused-blur threshold of lccrf_images (kFusedBlurMaxN = 32768 pixels, csrc/engine.cuh): the workloads
# on each side of it (640x480 x 16 and 160x120 x 64, scripts/images_bench.py) with two variant builds of the library,
# one that takes k_blur_fused for every image size and one that never does.  The variants live in a temporary
# directory (or in VARIANT_DIR when given; builds found there are reused) and are never installed.
# Usage: bash scripts/images_blur_threshold.sh OUTDIR [VARIANT_DIR]
set -e
OUT=${1:?usage: images_blur_threshold.sh OUTDIR [VARIANT_DIR]}
ROOT=$(cd "$(dirname "$0")/.." && pwd)
VDIR=${2:-}
if [ -z "$VDIR" ]; then
    VDIR=$(mktemp -d)
    trap 'rm -rf "$VDIR"' EXIT
fi
for v in fused_always:2147483647 fused_never:0; do
    name=${v%%:*}
    thr=${v##*:}
    tree=$VDIR/$name
    if [ ! -f "$tree/lc-crf-slam_b200/liblccrf.so" ]; then
        mkdir -p "$tree/lc-crf-slam_b200"
        cp -r "$ROOT/include" "$tree/"
        cp -r "$ROOT/lc-crf-slam_b200/csrc" "$ROOT/lc-crf-slam_b200/densecrf" "$ROOT"/lc-crf-slam_b200/*.py "$tree/lc-crf-slam_b200/"
        rm -rf "$tree/lc-crf-slam_b200/csrc/build"
        sed -i "s/constexpr int kFusedBlurMaxN = 32768;/constexpr int kFusedBlurMaxN = $thr;/" "$tree/lc-crf-slam_b200/csrc/engine.cuh"
        grep -q "kFusedBlurMaxN = $thr;" "$tree/lc-crf-slam_b200/csrc/engine.cuh"
        make -C "$tree/lc-crf-slam_b200/csrc" -j16 > /dev/null
    fi
    python "$ROOT/scripts/images_bench.py" --out "$OUT" --workloads c2_b16,small_b64 --pkg-root "$tree" --tag "$name"
done
