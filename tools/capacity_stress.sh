#!/bin/bash
# The frame parity tests against a build whose frame scratch starts tiny (16 entries per tile bin, no spare triangle slots,
# no spare raster work items) and whose big-triangle list takes every triangle over more than 8 tiles: every frame then
# overflows and takes the grow-and-retry paths (bins, triangle slots without repeated ids, work items), and the raster
# kernel's big-list path is used by every frame with large triangles.  usage: bash tools/capacity_stress.sh <tag>
# -> $VX_LOG_DIR/capacity_stress_<tag>.log (VX_LOG_DIR defaults to logs/)
TAG=${1:-x}
FLAGS="-DVX_BIN_CAP0=16 -DVX_TRI_SLACK=0 -DVX_ITEM_SLACK=0 -DVX_BIG_TILES=8"
OUT=${VX_LOG_DIR:-logs}
mkdir -p "$OUT"
LOG=$OUT/capacity_stress_${TAG}.log
bash tools/build_variant.sh stress "$FLAGS" > $LOG 2>&1 || { echo "capacity-stress build failed"; tail -5 $LOG; exit 1; }
export VX_B200_LIB=$PWD/variants/libvx_stress.so
python - >> $LOG 2>&1 <<'PY'
# how much of each capacity path a 1280x720 and a 3840x2160 terrain frame use in this build (first frame on a new context)
import ctypes as C, sys
sys.path.insert(0, "tests")
import vx_scenes
from differential_projection_voxel_renderer_b200 import api
for vd, w, h in ((12, 1280, 720), (32, 3840, 2160)):
    ctx = api.Context(0)
    pos, world, p, v, nb = vx_scenes.terrain_scene(vd)
    batch = api.BinaryGreedyMesher.mesh_batch(v, p, nb, None, ctx)
    cam = vx_scenes.main_camera(w, h)
    api.render_frame(batch, cam.view_projection(), cam.position, api.default_frame_config(w, h), mesh_ids=None, view_distance=vd, ctx=ctx)
    cnt = (C.c_uint32 * 32)()
    ctx.check(ctx.lib.vx_frame_counters(ctx.handle, cnt))
    print(f"{w}x{h} vd{vd}: big triangles {cnt[6]}, fullest bin {cnt[5]}, triangles {cnt[2]}, second near-clip pieces {cnt[13]}, "
          f"work items {cnt[9]} (plan wanted {cnt[12]})")
    batch.release()
    ctx.close()
PY
python -m pytest tests/test_frame_gpu.py tests/test_golden.py tests/test_frame_capacity_gpu.py tests/test_atlas_shading_gpu.py -m gpu -q -rA >> $LOG 2>&1
rc=$?
echo "capacity-stress build ($FLAGS): rc=$rc $(tail -1 $LOG)"
grep -E "^[0-9]+x[0-9]+ vd" $LOG
