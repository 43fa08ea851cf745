"""Swept-box collision timings on the view-distance-12 world (vx_world_move_boxes_device).

    python tools/move_bench.py --out DIR [--iters 100] [--warmup 10]

Workloads, 1,000,000 seeded boxes each, dropped around the terrain surface (corner 0 .. 4 voxels above the column's top
block, where entities are and where moves collide; only corners in loaded chunks, so every box is valid):
  player   0.6 x 1.8 x 0.6 boxes, deltas up to 1 on each axis
  large    boxes of up to 16 on each side, deltas up to 16 on each axis
Every launch starts from the same inputs: before each, the positions and slots are restored from a pristine device copy
(the kernel updates them in place) outside the timed window; each launch is timed with CUDA events on the context's
stream, and the result is the mean over --iters launches after --warmup.  The world's voxels are not flushed from L2
between launches: a physics loop re-reads the same world every tick.  The voxel bytes each move reads come from a counting
run of the same moves on the CPU oracle (tests/move_oracle.c), whose results must equal the device's bit for bit.  Writes
DIR/move_bench.json with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

VD, N = 12, 1_000_000


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def host_slots(w, worldgen):
    """Slot-indexed world arrays for the oracle (the world is not edited)."""
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


def surface_boxes(rng, w, worldgen, size, max_delta):
    """N boxes with corners on random columns of the loaded world, 0 .. 4 voxels above the column's top block, in loaded
    chunks."""
    c = np.array(sorted(w.chunks), dtype=np.int64)
    x0, z0 = int(c[:, 0].min()) * 32, int(c[:, 2].min()) * 32
    nx, nz = (int(c[:, 0].max()) + 1) * 32 - x0, (int(c[:, 2].max()) + 1) * 32 - z0
    heights = worldgen.terrain_heights(x0, z0, nx, nz)
    m = 2 * N  # the columns of the bounding square outside the loaded sphere are dropped
    xz = rng.random((m, 2)) * [nx, nz] + [x0, z0]
    p = np.stack([xz[:, 0], np.zeros(m), xz[:, 1]], axis=1)
    p[:, 1] = heights[np.floor(xz[:, 1]).astype(np.int64) - z0, np.floor(xz[:, 0]).astype(np.int64) - x0] + 1.0 + 4.0 * rng.random(m)
    p = p.astype(np.float32)
    p = p[w.start_slots(p) >= 0][:N]
    assert p.shape[0] == N
    return p, np.ascontiguousarray(np.broadcast_to(size, (N, 3)), dtype=np.float32), \
        rng.uniform(-max_delta, max_delta, (N, 3)).astype(np.float32)


def time_moves(torch, ctx, w, pos, size, delta, iters, warmup):
    dev = torch.device("cuda", ctx.device)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    n = pos.shape[0]
    with torch.cuda.stream(stream):
        p0, s0 = torch.from_numpy(pos).to(dev), torch.from_numpy(w.start_slots(pos)).to(dev)
        tp, ts = p0.clone(), s0.clone()
        tsz, td = torch.from_numpy(size).to(dev), torch.from_numpy(delta).to(dev)
        tf = torch.empty(n, dtype=torch.int32, device=dev)
        args = (ctx.handle, w.batch.handle, tp.data_ptr(), tsz.data_ptr(), td.data_ptr(), ts.data_ptr(), n, tf.data_ptr())
        events = []
        for k in range(warmup + iters):
            tp.copy_(p0)
            ts.copy_(s0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.check(ctx.lib.vx_world_move_boxes_device(*args))
            e1.record(stream)
            if k >= warmup:
                events.append((e0, e1))
    stream.synchronize()
    ms = [a.elapsed_time(b) for a, b in events]
    return float(np.mean(ms)), float(np.min(ms)), tp.cpu().numpy(), ts.cpu().numpy(), tf.cpu().numpy().view(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    a = ap.parse_args()
    import torch

    from differential_projection_voxel_renderer_b200 import api, world as vxw, worldgen
    import vx_move_oracle

    info = gpu_info()
    ctx = api.Context(0)
    w = vxw.World(vxw.WorldConfig(view_distance=VD, max_chunks_per_frame=1 << 20), ctx=ctx)
    w.update((0.0, 10.0, 20.0))
    host = host_slots(w, worldgen)
    rng = np.random.default_rng(2025)
    workloads = {"player_1M": surface_boxes(rng, w, worldgen, (0.6, 1.8, 0.6), 1.0)}
    pos, _, delta = surface_boxes(rng, w, worldgen, (1.0, 1.0, 1.0), 16.0)
    workloads["large_1M"] = (pos, (16.0 * (1.0 - rng.random((N, 3)))).astype(np.float32), delta)

    result = {"gpu": info, "view_distance": VD, "chunks_loaded": w.chunk_count(),
              "varied_chunks": int(sum(1 for f in w.uniform_flags.values() if f == 0)), "iters": a.iters, "warmup": a.warmup,
              "workloads": {}}
    for name, (pos, size, delta) in workloads.items():
        ms, ms_min, dpos, dslots, dflags = time_moves(torch, ctx, w, pos, size, delta, a.iters, a.warmup)
        wpos, wslots, wflags, reads = vx_move_oracle.move_boxes(*host, pos, size, delta, w.start_slots(pos), want_reads=True)
        assert np.array_equal(dpos.view(np.uint32), wpos.view(np.uint32)) and np.array_equal(dslots, wslots) \
            and np.array_equal(dflags, wflags), f"{name}: device moves differ from the oracle"
        result["workloads"][name] = {
            "boxes": N, "ms_per_launch": ms, "ms_min": ms_min, "boxes_per_s": N / (ms * 1e-3),
            "voxels_read_per_box": float(reads.mean()), "voxels_read_max": int(reads.max()),
            "on_ground": int(((wflags >> 3) & 1).sum()), "blocked_any": int(((wflags & 63) != 0).sum()),
            "touched_unloaded": int(((wflags >> 6) & 1).sum()), "invalid": int(((wflags >> 7) & 1).sum())}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "move_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    w.batch.release()
    ctx.close()


if __name__ == "__main__":
    main()
