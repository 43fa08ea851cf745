"""Region edit timings on the view-distance-12 world (World.fill_ball / fill_box, vx_world_batch_fill_regions).

    python tools/region_bench.py --out DIR [--explosions 40]

Workloads:
  explosions  seeded balls with radius_sq 64 and 576 centred on terrain surface voxels near the camera, carving solid to air
              (replace = grass, dirt, stone), one after the other.  Per explosion: the device time of the
              vx_world_batch_fill_regions call (CUDA events on the context's stream around it: op and slot upload, kernel,
              change-byte read-back), the host time of World.fill_ball (chunk set, the call, bookkeeping) and of the
              MeshCache.refresh that follows.
  replay      --replay-ops small balls recorded on the chunks around x = 300, then every chunk a fill changed is unloaded
              and generated again: the device time of the one fill_regions call that replays the fills, and the host time
              of the World.update that reloads them.
  box         a 256 x 64 x 256 fill with stone, replace = air only (128 chunks); then, for comparison, the same 4.2 M voxels
              with their resulting types through World.set_blocks (host time).
Every fill is checked against the CPU oracle (tests/region_oracle.c): the touched chunks are read back before and after the
call and must equal the oracle's result bit for bit, change bytes included; reloaded chunks must equal their state before
unloading.  The world's voxels are not flushed from L2 between calls: an interactive edit touches a world that the frame
loop keeps reading.  Writes DIR/region_bench.json with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

VD = 12
CAMERA = (0.0, 10.0, 20.0)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


class TimedDevice:
    """Wraps the world's fill_regions: CUDA events around each call, and an oracle check of what it did."""

    def __init__(self, torch, w, vro):
        self.torch, self.w, self.vro = torch, w, vro
        self.stream = torch.cuda.ExternalStream(w.device.ctx.stream, device=torch.device("cuda", w.device.ctx.device))
        self.inner = w.device.fill_regions
        self.ms, self.checked = [], 0
        w.device.fill_regions = self

    def __call__(self, ops, slots):
        at = {s: p for p, s in self.w.chunks.items()}
        vox, flags = self.w.device.read_voxels(slots)
        rows = vox.copy()
        pos = np.array([at[s] for s in slots.tolist()], dtype=np.int32).reshape(-1, 3)
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        changed = self.inner(ops, slots)
        e1.record(self.stream)
        e1.synchronize()
        self.ms.append(e0.elapsed_time(e1))
        self.last = (int(ops.size), int(slots.size))
        rc, want = self.vro.fill_regions(pos, vox, flags, ops, np.arange(slots.size, dtype=np.int32))  # vox, flags: expected
        got_vox, got_flags = self.w.device.read_voxels(slots)
        varied = flags == 0
        assert rc == 0 and np.array_equal(changed, want) and np.array_equal(got_flags, flags), "fill differs from the oracle"
        assert np.array_equal(got_vox[varied], vox[varied]) and np.array_equal(got_vox[~varied], rows[~varied]), "voxels differ"
        self.checked += int(slots.size)
        return changed


def surface_voxels(rng, worldgen, n, spread):
    x0, z0 = int(CAMERA[0]) - spread, int(CAMERA[2]) - spread
    h = worldgen.terrain_heights(x0, z0, 2 * spread, 2 * spread)
    xz = rng.integers(0, 2 * spread, (n, 2))
    return [(x0 + int(x), int(h[z, x]), z0 + int(z)) for x, z in xz.tolist()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--explosions", type=int, default=40)
    ap.add_argument("--replay-ops", type=int, default=200)
    a = ap.parse_args()
    import torch

    from differential_projection_voxel_renderer_b200 import api, world as vxw, worldgen
    import vx_region_oracle as vro

    info = gpu_info()
    ctx = api.Context(0)
    w = vxw.World(vxw.WorldConfig(view_distance=VD, max_chunks_per_frame=1 << 20), ctx=ctx)
    w.update(CAMERA)
    cache = vxw.MeshCache(w)
    cache.update(sorted(w.chunks))
    dev = TimedDevice(torch, w, vro)
    rng = np.random.default_rng(2026)
    result = {"gpu": info, "view_distance": VD, "chunks_loaded": w.chunk_count(), "workloads": {}}

    # explosions
    for r2 in (64, 576):
        call_ms, fill_ms, refresh_ms, dirty_n = [], [], [], []
        for c in surface_voxels(rng, worldgen, a.explosions + 2, 160):
            n0 = len(dev.ms)
            t0 = time.perf_counter()
            dirty = w.fill_ball(c, r2, 0, replace=(1, 2, 3))
            t1 = time.perf_counter()
            cache.refresh(dirty)
            t2 = time.perf_counter()
            assert len(dev.ms) == n0 + 1
            call_ms.append(dev.ms[-1])
            fill_ms.append((t1 - t0) * 1e3)
            refresh_ms.append((t2 - t1) * 1e3)
            dirty_n.append(len(dirty))
        skip = 2  # warm-up
        result["workloads"][f"explosion_r2_{r2}"] = {
            "explosions": a.explosions, "device_ms_per_call": float(np.mean(call_ms[skip:])), "device_ms_min": float(np.min(call_ms[skip:])),
            "host_ms_fill_ball": float(np.mean(fill_ms[skip:])), "host_ms_refresh": float(np.mean(refresh_ms[skip:])),
            "dirty_chunks_mean": float(np.mean(dirty_n[skip:]))}

    # replay, before the box's set_blocks comparison, whose 4.2 M edits would be replayed too
    centre = np.array([300, 0, 20])
    hc = worldgen.terrain_heights(int(centre[0]) - 32, int(centre[2]) - 32, 64, 64)
    n0 = len(dev.ms)
    for _ in range(a.replay_ops):
        dx, dz = rng.integers(0, 64, 2)
        c = (int(centre[0]) - 32 + int(dx), int(hc[dz, dx]), int(centre[2]) - 32 + int(dz))
        try:
            w.fill_ball(c, int(rng.integers(4, 50)), int(rng.integers(0, 4)))
        except KeyError:
            pass
    recorded = len(dev.ms) - n0
    held = sorted(p for p in w._fills_at if p in w.chunks)  # every chunk a fill changed, the explosions' included
    before = {p: w.chunk_voxels(p) for p in held}
    w.update((32.0 * 40, 10.0, 20.0))
    assert not any(p in w.chunks for p in held)
    n0 = len(dev.ms)
    t0 = time.perf_counter()
    w.update(CAMERA)
    t1 = time.perf_counter()
    replay = dev.ms[n0:]
    assert len(replay) == 1
    for p in held:
        f, v = w.chunk_voxels(p)
        assert f == before[p][0] and np.array_equal(v, before[p][1]), f"{p} differs after the replay"
    result["workloads"]["replay"] = {
        "ops_recorded": recorded, "chunks_replayed": dev.last[1], "ops_replayed": dev.last[0], "device_ms_replay_call": float(replay[0]),
        "host_ms_update_reload": (t1 - t0) * 1e3, "chunks_generated": len(w.generated_last_update)}

    # box fill, air only, then the same voxels through set_blocks
    lo, hi = np.array([-128, 0, -128]), np.array([127, 63, 127])
    n0 = len(dev.ms)
    t0 = time.perf_counter()
    dirty = w.fill_box(lo, hi, 3, replace=(0,))
    t1 = time.perf_counter()
    box_call = dev.ms[n0:]
    positions = [(x, y, z) for x in range(-4, 4) for y in range(0, 2) for z in range(-4, 4)]
    final = {p: w.chunk_voxels(p)[1] for p in positions}
    g = np.stack(np.meshgrid(np.arange(lo[0], hi[0] + 1), np.arange(lo[1], hi[1] + 1), np.arange(lo[2], hi[2] + 1), indexing="ij"),
                 axis=-1).reshape(-1, 3)
    cp = g >> 5
    stacked = np.stack([final[p] for p in positions])  # positions in (x, y, z) order
    idx = (cp[:, 0] + 4) * 16 + cp[:, 1] * 8 + (cp[:, 2] + 4)
    types = stacked[idx, g[:, 2] & 31, g[:, 1] & 31, g[:, 0] & 31]
    t2 = time.perf_counter()
    w.set_blocks(g, types)
    t3 = time.perf_counter()
    assert all(np.array_equal(w.chunk_voxels(p)[1], final[p]) for p in positions), "set_blocks of the filled types changed voxels"
    result["workloads"]["box_256x64x256_air_only"] = {
        "voxels": int(g.shape[0]), "chunks": len(positions), "device_ms_per_call": float(box_call[0]), "host_ms_fill_box": (t1 - t0) * 1e3,
        "dirty_chunks": len(dirty), "host_ms_set_blocks_same_voxels": (t3 - t2) * 1e3}

    result["oracle_checked_chunk_fills"] = dev.checked
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "region_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    w.batch.release()
    ctx.close()


if __name__ == "__main__":
    main()
