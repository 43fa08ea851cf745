"""Picking and block-edit timings on the view-distance-12 world (vx_world_raycast_device, vx_world_batch_set_blocks).

    python tools/raycast_bench.py --out DIR [--iters 200] [--warmup 10]

Workloads, each timed with CUDA events on the context's stream over --iters back-to-back launches after --warmup:
  pixels   one ray per pixel of a 1280x720 frame from the bench camera ((0,10,20), looking down -Z), max_t 384
  random   1,000,000 rays from seeded random origins inside the loaded world, random unit directions, max_t 384
The world's voxels are not flushed from L2 between launches: a picking loop re-reads the same world.  DDA steps per ray
(face crossings) come from a second, counting run of the same walk on its CPU oracle (tests/ray_oracle.c), whose hits
must equal the device's.
Also timed on the host clock: one interactive edit -- set_blocks of one chunk-border voxel + MeshCache.refresh, ending in
a device synchronise.  Writes DIR/raycast_bench.json with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, VD, MAX_T, N_RANDOM = 1280, 720, 12, 384.0, 1_000_000


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def host_slots(w, worldgen):
    """Slot-indexed world arrays for the oracle (no edits are made before the ray workloads)."""
    cap = w.capacity
    pos, flags = np.zeros((cap, 3), np.int32), np.ones(cap, np.uint8)
    nbr, vox = np.full((cap, 6), -1, np.int32), np.zeros((cap, 32768), np.uint8)
    allp = sorted(w.chunks)
    g = worldgen.generate_world(np.array(allp, dtype=np.int32))
    for i, p in enumerate(allp):
        s = w.chunks[p]
        pos[s], flags[s], nbr[s] = p, g.uniform_flags[i], w._neighbor_row(p)
        if flags[s] == 0:
            vox[s] = g.voxels[i]
    return pos, vox, flags, nbr


def time_rays(torch, ctx, w, o, d, iters, warmup):
    dev = torch.device("cuda", ctx.device)
    to, td = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    ts = torch.from_numpy(w.start_slots(o)).to(dev)
    th = torch.empty((o.shape[0], 32), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    args = (ctx.handle, w.batch.handle, to.data_ptr(), td.data_ptr(), ts.data_ptr(), o.shape[0], MAX_T, th.data_ptr())
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    for _ in range(warmup):
        ctx.check(ctx.lib.vx_world_raycast_device(*args))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        ctx.check(ctx.lib.vx_world_raycast_device(*args))
    e1.record(stream)
    e1.synchronize()
    ms = e0.elapsed_time(e1) / iters
    return ms, th.cpu().numpy().reshape(-1).view(np.dtype((np.void, 32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    a = ap.parse_args()
    import torch

    from differential_projection_voxel_renderer_b200 import api, camera, world as vxw, worldgen
    import vx_ray_oracle

    info = gpu_info()
    ctx = api.Context(0)
    cam = camera.Camera((0.0, 10.0, 20.0), W / H)
    vp = cam.view_projection()
    w = vxw.World(vxw.WorldConfig(view_distance=VD, max_chunks_per_frame=1 << 20), ctx=ctx)
    cache = vxw.MeshCache(w)
    vxw.frame(w, cache, cam.position, vp, api.default_frame_config(W, H), ctx)
    host = host_slots(w, worldgen)

    px = np.stack(np.meshgrid(np.arange(W), np.arange(H)), axis=-1).reshape(-1, 2)
    rng = np.random.default_rng(2024)
    c = np.array(sorted(w.chunks), dtype=np.float64)
    ro = ((c[rng.integers(0, c.shape[0], N_RANDOM)] + rng.random((N_RANDOM, 3))) * 32.0).astype(np.float32)
    rd = rng.normal(size=(N_RANDOM, 3))
    rd = (rd / np.linalg.norm(rd, axis=1, keepdims=True)).astype(np.float32)
    workloads = {"pixels_1280x720": api.pixel_rays(vp, cam.position, px, W, H), "random_1M": (ro, rd)}

    result = {"gpu": info, "view_distance": VD, "chunks_loaded": w.chunk_count(),
              "varied_chunks": int(sum(1 for f in w.uniform_flags.values() if f == 0)), "max_t": MAX_T,
              "iters": a.iters, "warmup": a.warmup, "workloads": {}}
    for name, (o, d) in workloads.items():
        ms, dev_hits = time_rays(torch, ctx, w, o, d, a.iters, a.warmup)
        want, steps = vx_ray_oracle.raycast(*host, o, d, w.start_slots(o), MAX_T, want_steps=True)
        assert dev_hits.tobytes() == want.tobytes(), f"{name}: device hits differ from the oracle"
        status = np.bincount(want["status"], minlength=4)
        result["workloads"][name] = {
            "rays": int(o.shape[0]), "ms_per_launch": ms, "rays_per_s": o.shape[0] / (ms * 1e-3),
            "dda_steps_per_ray": float(steps.mean()), "dda_steps_max": int(steps.max()),
            "status_counts": {"hit": int(status[0]), "miss": int(status[1]), "left_world": int(status[2]), "invalid": int(status[3])}}

    # one interactive edit: a border voxel of a meshed Varied chunk, alternately stone and air
    p = next(q for q in sorted(cache.cached) if w.uniform_flags[q] == 0 and (q[0] + 1, q[1], q[2]) in cache.cached)
    voxel = (p[0] * 32 + 31, p[1] * 32 + 16, p[2] * 32 + 16)
    times, dirty = [], []
    for k in range(60):
        ctx.synchronize()
        t0 = time.perf_counter()
        dirty = w.set_blocks([voxel], [3 if k % 2 == 0 else 0])
        cache.refresh(dirty)
        ctx.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    times = times[10:]
    result["edit"] = {"what": "World.set_blocks of one chunk-border voxel + MeshCache.refresh (2 chunks re-meshed) + synchronise, "
                              "host clock, 50 edits after 10 warm-up", "chunks_refreshed": len(dirty),
                      "ms_median": statistics.median(times), "ms_p90": sorted(times)[int(0.9 * len(times))], "ms_min": min(times)}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "raycast_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    w.batch.release()
    ctx.close()


if __name__ == "__main__":
    main()
