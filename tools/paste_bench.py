"""Copy and paste timings on the view-distance-12 world (World.copy_region / World.paste, vx_world_batch_copy_region and
vx_world_batch_paste).

    python tools/paste_bench.py --out DIR [--stamps 40]

Workloads:
  stamp       seeded 16^3 and 64^3 structures (random solid types in a blob, transparent air around it) centred on terrain
              surface voxels near the camera, one after the other.  Per stamp: the device time of the vx_world_batch_paste
              call (CUDA events on the context's stream around it: op, slot and template upload, kernel, change-byte
              read-back) and the host time of World.paste (template checks, chunk set, the call, bookkeeping).
  copy        the 256 x 64 x 256 box -128..127, 0..63, -128..127 (4.2 M voxels, 128 chunks): the device time of the
              vx_world_batch_copy_region call (table upload, gather kernel, stale-table check, the copy of the box back)
              and the host time of World.copy_region.
  clone       that copy pasted 64 voxels higher (128 chunks): device and host time of the paste.
  replay      every chunk a paste changed is unloaded and generated again: the device time of the replay calls and the
              host time of the World.update that reloads them.
Every paste is checked against the CPU oracle (tests/paste_oracle.c): the listed chunks are read back before and after the
call and must equal the oracle's result bit for bit, change bytes included; the copy must equal the oracle's copy of the
same chunks; reloaded chunks must equal their state before unloading.  The host time of these checks is taken out of
the host timings.  Writes DIR/paste_bench.json with the card's name
and power limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import CAMERA, VD, gpu_info, surface_voxels  # noqa: E402


class Timed:
    """CUDA events around each call of the world's paste and copy_region, and an oracle check of what they did."""

    def __init__(self, torch, w, vpo):
        self.torch, self.w, self.vpo = torch, w, vpo
        self.stream = torch.cuda.ExternalStream(w.device.ctx.stream, device=torch.device("cuda", w.device.ctx.device))
        self.inner_paste, self.inner_copy = w.device.paste, w.device.copy_region
        self.ms, self.copy_ms, self.checked = [], [], 0
        self.check_s = 0.0  # host time spent in the checks, taken out of the host timings
        w.device.paste, w.device.copy_region = self.paste, self.copy_region

    def _time(self, fn, *args):
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        out = fn(*args)
        e1.record(self.stream)
        e1.synchronize()
        return out, e0.elapsed_time(e1)

    def paste(self, ops, templates, slots):
        t0 = time.perf_counter()
        at = {s: p for p, s in self.w.chunks.items()}
        vox, flags = self.w.device.read_voxels(slots)
        rows = vox.copy()
        pos = np.array([at[s] for s in slots.tolist()], dtype=np.int32).reshape(-1, 3)
        t1 = time.perf_counter()
        changed, ms = self._time(self.inner_paste, ops, templates, slots)
        t2 = time.perf_counter()
        self.ms.append(ms)
        self.last = (int(ops.size), int(slots.size))
        rc, want = self.vpo.paste(pos, vox, flags, ops, templates, np.arange(slots.size, dtype=np.int32))  # vox, flags: expected
        got_vox, got_flags = self.w.device.read_voxels(slots)
        varied = flags == 0
        assert rc == 0 and np.array_equal(changed, want) and np.array_equal(got_flags, flags), "paste differs from the oracle"
        assert np.array_equal(got_vox[varied], vox[varied]) and np.array_equal(got_vox[~varied], rows[~varied]), "voxels differ"
        self.checked += int(slots.size)
        self.check_s += (t1 - t0) + (time.perf_counter() - t2)
        return changed

    def copy_region(self, lo, dims, chunk_slots):
        box, ms = self._time(self.inner_copy, lo, dims, chunk_slots)
        t2 = time.perf_counter()
        self.copy_ms.append(ms)
        listed = np.unique(chunk_slots[chunk_slots >= 0]).astype(np.int32)  # the oracle sees the listed slots only, renumbered
        vox, flags = self.w.device.read_voxels(listed)
        at = {s: p for p, s in self.w.chunks.items()}
        pos = np.array([at[s] for s in listed.tolist()], np.int32).reshape(-1, 3)
        table = np.where(chunk_slots >= 0, np.searchsorted(listed, chunk_slots), -1).astype(np.int32)
        rc, want = self.vpo.copy_region(pos, vox, flags, lo, dims, table)
        assert rc == 0 and np.array_equal(box, want), "copy differs from the oracle"
        self.check_s += time.perf_counter() - t2
        return box


def structure(rng, size):
    t = rng.integers(1, 4, (size, size, size)).astype(np.uint8)
    g = np.indices((size, size, size)) - (size - 1) / 2
    keep = (g ** 2).sum(axis=0) <= (size / 2) ** 2 * rng.uniform(0.4, 1.0)
    return np.where(keep & (rng.random(t.shape) < 0.8), t, 0xFF).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--stamps", type=int, default=40)
    a = ap.parse_args()
    import torch

    from differential_projection_voxel_renderer_b200 import api, world as vxw, worldgen
    import vx_paste_oracle as vpo

    info = gpu_info()
    ctx = api.Context(0)
    w = vxw.World(vxw.WorldConfig(view_distance=VD, max_chunks_per_frame=1 << 20), ctx=ctx)
    w.update(CAMERA)
    cache = vxw.MeshCache(w)
    cache.update(sorted(w.chunks))
    dev = Timed(torch, w, vpo)
    rng = np.random.default_rng(2026)
    result = {"gpu": info, "view_distance": VD, "chunks_loaded": w.chunk_count(), "workloads": {}}

    # stamps
    for size in (16, 64):
        call_ms, host_ms, chunks = [], [], []
        for c in surface_voxels(rng, worldgen, a.stamps + 2, 160):
            t = structure(rng, size)
            n0 = len(dev.ms)
            t0, c0 = time.perf_counter(), dev.check_s
            w.paste(t, np.array(c) - size // 2)
            t1 = time.perf_counter() - (dev.check_s - c0)
            assert len(dev.ms) == n0 + 1
            call_ms.append(dev.ms[-1])
            host_ms.append((t1 - t0) * 1e3)
            chunks.append(dev.last[1])
        skip = 2  # warm-up
        result["workloads"][f"stamp_{size}"] = {
            "stamps": a.stamps, "device_ms_per_call": float(np.mean(call_ms[skip:])), "device_ms_min": float(np.min(call_ms[skip:])),
            "host_ms_paste": float(np.mean(host_ms[skip:])), "chunks_per_stamp": float(np.mean(chunks[skip:]))}

    # replay, before the large clone, which would be replayed too
    held = sorted(p for p in w._pastes_at if p in w.chunks)
    before = {p: w.chunk_voxels(p) for p in held}
    w.update((32.0 * 40, 10.0, 20.0))
    assert not any(p in w.chunks for p in held)
    n0 = len(dev.ms)
    t0, c0 = time.perf_counter(), dev.check_s
    w.update(CAMERA)
    t1 = time.perf_counter() - (dev.check_s - c0)
    replay = dev.ms[n0:]
    for p in held:
        f, v = w.chunk_voxels(p)
        assert f == before[p][0] and np.array_equal(v, before[p][1]), f"{p} differs after the replay"
    result["workloads"]["replay"] = {
        "pastes_recorded": len(w.pastes), "chunks_replayed": len(held), "paste_calls": len(replay),
        "device_ms_replay_calls": float(np.sum(replay)), "host_ms_update_reload": (t1 - t0) * 1e3,
        "chunks_generated": len(w.generated_last_update)}

    # the 256 x 64 x 256 copy: 4 warm-up, then 20 timed
    lo, hi = np.array([-128, 0, -128]), np.array([127, 63, 127])
    host = []
    for _ in range(24):
        t0, c0 = time.perf_counter(), dev.check_s
        box = w.copy_region(lo, hi)
        host.append((time.perf_counter() - t0 - (dev.check_s - c0)) * 1e3)
    assert (box != 0xFF).all()
    result["workloads"]["copy_256x64x256"] = {
        "voxels": int(box.size), "chunks": 128, "device_ms_per_call": float(np.mean(dev.copy_ms[4:])),
        "device_ms_min": float(np.min(dev.copy_ms[4:])), "host_ms_copy_region": float(np.mean(host[4:]))}

    # clone it 64 voxels higher
    n0 = len(dev.ms)
    t0, c0 = time.perf_counter(), dev.check_s
    dirty = w.paste(box, lo + [0, 64, 0])
    t1 = time.perf_counter() - (dev.check_s - c0)
    assert len(dev.ms) == n0 + 1 and np.array_equal(w.copy_region(lo + [0, 64, 0], hi + [0, 64, 0]), box)
    result["workloads"]["clone_256x64x256"] = {
        "voxels": int(box.size), "chunks": dev.last[1], "device_ms_per_call": float(dev.ms[-1]), "host_ms_paste": (t1 - t0) * 1e3,
        "dirty_chunks": len(dirty)}

    result["oracle_checked_chunk_pastes"] = dev.checked
    result["oracle_checked_copies"] = len(dev.copy_ms)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "paste_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    w.batch.release()
    ctx.close()


if __name__ == "__main__":
    main()
