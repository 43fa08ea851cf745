#!/bin/bash
# The frame parity tests against a build with -DVX_DEBUG_CHECKS (index checks inside the frame kernels, the step bound of
# the ray cast kernel; stands in for compute-sanitizer memcheck, which is closed on the GPU pool).  usage: bash tools/debug_checks.sh <tag>
# -> $VX_LOG_DIR/debug_checks_<tag>.log (VX_LOG_DIR defaults to logs/)
TAG=${1:-x}
OUT=${VX_LOG_DIR:-logs}
mkdir -p "$OUT"
LOG=$OUT/debug_checks_${TAG}.log
bash tools/build_variant.sh dbg "-DVX_DEBUG_CHECKS" > /dev/null 2>&1 || true
VX_B200_LIB=$PWD/variants/libvx_dbg.so python -m pytest tests/test_frame_gpu.py tests/test_golden.py tests/test_frame_capacity_gpu.py tests/test_atlas_shading_gpu.py tests/test_world_gpu.py tests/test_block_edit_gpu.py tests/test_multi_gpu.py -m gpu -x -q > $LOG 2>&1
echo "debug-checks build: rc=$? $(tail -1 $LOG)"
VX_B200_LIB=$PWD/variants/libvx_dbg.so python tools/sanitize_target.py >> $LOG 2>&1; echo "target rc=$?"
