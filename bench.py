#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 voxel frame path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): one full 1280x720 frame at view
distance 12 -- chunk cull (filter A) + AABB reject / draw order (filter B) + project / near-clip / backface cull of every
quad + span rasterization with depth buffer and textured shading -- of the seeded synthetic terrain world (7,153
lattice chunks, the Varied ones meshed with their neighbours), camera (0,10,20) looking down -Z, meshes cached on the
device exactly as the reference caches them between frames (main.rs:225-280).  A "step" is one frame.

One JSON line on stdout (rank 0).  `value` = device-resident frames/s with `--lanes` frames in flight (api.FrameLanes: one
context -- stream + frame scratch -- per lane; the timed frames go out in groups of one frame per lane, every group starts
behind an L2 flush and is timed with CUDA events from the end of the flush to the last lane's end); `e2e` = the same frame through the public host API (VP + camera uploaded, ARGB frame read back
into pinned host memory, every step); `roofline` describes the dominant kernel; `cpu_baseline` is the C restatement of
the reference CPU path timed on this box's host cores; `extra` carries the second metric of BASELINE.json (chunks
meshed per second) and the per-kernel split.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, VD = 1280, 720, 12
METRIC = "frames_per_sec_1280x720_vd12"
UNIT = "frames/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of `kernel` per launch from the newest committed ncu capture
    (profiles/*_traffic.json, written from an `ncu --set full` run of tools/ncu_target.py), or None."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None
    try:
        return float(json.load(open(files[-1]))[kernel]["traffic"])
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_scene():
    """The seeded world of BASELINE configs[2]: every lattice chunk within VD of chunk (0,0,0) (7,153 of them, Uniform
    ones included -- the reference's get_visible_chunks_frustum walks all loaded chunks, world.rs:118-146), camera of
    main.rs:51."""
    import vx_scenes
    pos, world, p, v, nb = vx_scenes.terrain_scene(VD)
    cam = vx_scenes.main_camera(W, H)
    return {"pos": pos, "world": world, "p": p, "v": v, "nb": nb, "cam": cam,
            "flags": world.uniform_flags, "nb_full": world.neighbor_table(), "v_full": world.voxels}


def workload_config(n_gpus: int, sc, total_quads: int):
    """`config` of the JSON line -- one function for both arms, so the driver sees the same dict."""
    return {
        "workload": "full frame 1280x720 view distance 12: filter A over every loaded chunk + filter B / draw order + project / near-clip / "
                    "backface-cull every quad + span raster with depth buffer and textured shading; meshes cached (main.rs:225-280); "
                    "BASELINE.json configs[2]",
        "resolution": [W, H], "view_distance": VD,
        "chunks": int(sc["pos"].shape[0]), "varied_chunks": int(sc["p"].shape[0]), "total_quads": int(total_quads),
        "camera": "(0,10,20) yaw 0 pitch 0 fov 70",
        "l2": "CUDA arm: L2 flushed (256 MiB device write, outside the timed events) before every timed group of frames -- one frame per "
              "lane, all of them start cold; CPU arm: not applicable",
        "parallelism": "1 GPU" if n_gpus == 1 else f"{n_gpus} GPUs: work-balanced screen stripes, each rank's raster kernel stores its rows into the "
                                                   "composed frame in GPU0's memory over NVLink (CUDA IPC peer mapping, no collective)",
    }


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path (C restatement, see oracle/vx_oracle.h), all host threads
# ------------------------------------------------------------------------------------------------------------------
def cpu_frame_baseline(sc, min_seconds: float, threads: int, steps=None, warmup=1):
    from oracle import binding as ob
    pos, cam = sc["pos"], sc["cam"]
    ref = ob.mesh_chunks(sc["v_full"], sc["nb_full"], sc["flags"], pos)
    vp = cam.view_projection()
    cfg = ob.default_frame_config(W, H, n_threads=threads)
    atlas = ob.default_atlas()
    has = ref.has_mesh != 0

    def one_frame():
        vis = ob.cull_chunks(pos, vp, cam.position, VD)           # filter A over all loaded chunks (world.rs:118-146)
        ids = np.flatnonzero((vis != 0) & has).astype(np.int32)
        return ob.render_frame(ref, ids, vp, cam.position, cfg, atlas)  # filter B + sort + raster

    for _ in range(max(1, warmup)):
        one_frame()
    n, t0 = 0, time.perf_counter()
    while True:
        color, depth, _ = one_frame()
        n += 1
        el = time.perf_counter() - t0
        if steps is not None:
            if n >= steps:
                break
        elif el >= min_seconds:
            break
    return n / el, n, el, int(ref.quads.size // 3), (color, depth)


def cpu_mesh_baseline(v, nb, min_seconds: float):
    from oracle import binding as ob
    n, t0 = 0, time.perf_counter()
    while True:
        ob.mesh_chunks(v, nb)
        n += v.shape[0]
        el = time.perf_counter() - t0
        if el >= min_seconds:
            break
    return n / el, n, el


def dump_outputs(out_dir: str, color, depth):
    """--dump-outputs: the frame of the last timed step, as the caller of the path receives it, in float32 (exact):
    color_argb.npy (H, W, 4) channels A, R, G, B in 0..255 of the ARGB pixels; covered.npy (H, W) 1 where a fragment was
    drawn, else 0; depth.npy (H, W) the depth of drawn pixels, 0 elsewhere (the frame clears depth to +inf, and every
    stored value is finite so that outputs compare with a plain tolerance)."""
    os.makedirs(out_dir, exist_ok=True)
    argb = (np.asarray(color, dtype=np.uint32)[..., None] >> np.array([24, 16, 8, 0], dtype=np.uint32)) & 0xFF
    np.save(os.path.join(out_dir, "color_argb.npy"), argb.astype(np.float32))
    depth = np.asarray(depth, dtype=np.float32)
    covered = np.isfinite(depth)
    if not np.all(np.isposinf(depth[~covered])):
        raise RuntimeError("--dump-outputs: the frame's depth holds NaN or -inf")
    np.save(os.path.join(out_dir, "covered.npy"), covered.astype(np.float32))
    np.save(os.path.join(out_dir, "depth.npy"), np.where(covered, depth, np.float32(0.0)))
    log(f"outputs of the last timed step written to {out_dir}")


def cargo_note():
    import shutil
    return "cargo found on this box but the crate's dependencies are not vendored (no network)" if shutil.which("cargo") else \
        "no cargo/rustc on this box: the Rust crate cannot be built"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sc = build_scene()
    threads = os.cpu_count() or 1
    fps, n, el, tq, last_frame = cpu_frame_baseline(sc, 0.0, threads, steps=max(1, args.steps), warmup=max(1, args.warmup))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last_frame)
    out = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": n, "warmup": args.warmup,
        "ms_per_step": 1000.0 * el / n, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args.gpus, sc, tq),
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n} full frames; C restatement of the reference CPU path (oracle/), stripe-parallel over all {threads} host threads; "
                                   + cargo_note()},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_json_line(out)
    return 0


# ------------------------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------------------------
def event_pair(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def run_cuda(args):
    import torch
    from differential_projection_voxel_renderer_b200 import api, multigpu, sharding

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world_size > 1:
        import datetime
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=300))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    sc = build_scene()
    pos, p, v, nb, cam = sc["pos"], sc["p"], sc["v"], sc["nb"], sc["cam"]
    vp = cam.view_projection()
    ctx = api.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    L = max(1, args.lanes)
    lanes = api.FrameLanes(local_rank, L, first=ctx)  # lane 0 is ctx
    lane_streams = [torch.cuda.ExternalStream(c.stream, device=dev) for c in lanes.ctxs]
    n_lattice, n_varied = int(pos.shape[0]), int(p.shape[0])
    extra = {"lanes": L}

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs resident in HBM: the whole lattice (Uniform chunks carry a flag and no voxel data that is ever read) ------
    d_voxf = torch.from_numpy(sc["v_full"]).to(dev)
    d_posf = torch.from_numpy(pos).to(dev)
    d_nbf = torch.from_numpy(sc["nb_full"]).to(dev)
    d_flf = torch.from_numpy(sc["flags"]).to(dev)

    def mesh_full_locally():
        hh = C.c_void_p()
        ctx.check(ctx.lib.vx_mesh_chunks_device(ctx.handle, C.c_void_p(d_voxf.data_ptr()), C.c_void_p(d_posf.data_ptr()),
                                                C.c_void_p(d_nbf.data_ptr()), C.c_void_p(d_flf.data_ptr()), n_lattice, C.byref(hh)))
        return api.MeshBatch(ctx, hh)

    exchange = None
    if world_size == 1:
        batch = mesh_full_locally()
    else:
        # chunk-sharded meshing (chunk id modulo N) + device exchange: the frame below is rendered from the ASSEMBLED batch
        exchange = multigpu.MeshShardExchange(ctx, n_lattice, rank, world_size, dev)
        batch = exchange.sweep(d_voxf.data_ptr(), d_posf.data_ptr(), d_nbf.data_ptr(), d_flf.data_ptr())
    info = batch.info()
    total_quads = int(info.total_quads)

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def flush_l2():
        with torch.cuda.stream(stream):
            flush.fill_(1)

    cfg = api.default_frame_config(W, H)
    cfg_async = api.VxFrameConfig.from_buffer_copy(cfg)
    cfg_async.async_submit = 1
    cfg_lanes = api.VxFrameConfig.from_buffer_copy(cfg_async)  # frames that share the GPU: coarser raster work items
    cfg_lanes.frames_in_flight = L

    # ---- one synchronous full frame on every rank and lane: sizes the scratch, gives the per-tile-row work for the stripe split ----
    for c in lanes.ctxs:
        api.render_frame_device(batch, vp, cam.position, cfg, VD, c)
    st_full = api.frame_stats(ctx)
    comp = None
    comps = None
    stripes = [(0, H)]
    lane_frame_no = [0] * L
    if world_size > 1:
        # cost of every 8-row band of the full frame: bin entries + the tasks they expand to (sharding.stripe_band_cost)
        band = sharding.stripe_band_cost(api.frame_bin_counts(ctx), api.frame_bin_tasks(ctx))
        holder = [sharding.balanced_stripes(band, H, world_size, band=8, row_cost=float(band.sum()) / (20.0 * H))] if rank == 0 else [None]
        dist.broadcast_object_list(holder, src=0)
        stripes = [tuple(x) for x in holder[0]]
        # one compositor (composite buffers + flag words) per lane: a lane is an in-order sequence of frames of its own
        # (colour only unless --composite-depth: the depth plane is frame-internal on every GPU -- the reference presents
        # color_buffer, main.rs:320-322 -- and leaving it out halves what crosses NVLink; the guard below composes both planes)
        comps = [multigpu.StripeCompositor(c, W, H, rank, world_size, want_depth=bool(args.composite_depth), n_buffers=args.composite_buffers,
                                           fused_signal=bool(args.fused_signal)) for c in lanes.ctxs]
        for cp in comps:
            cp.set_stripes(stripes)
        comp = comps[0]

    cfg_stripe_lanes = api.VxFrameConfig.from_buffer_copy(cfg)
    cfg_stripe_lanes.frames_in_flight = L

    # the same camera every step: passed as tuples, which the host API recognises by identity (no per-call conversion)
    vp_t, cam_t = tuple(float(x) for x in np.asarray(vp, dtype=np.float32).reshape(16)), tuple(float(x) for x in cam.position)

    def step_device(l: int = 0, in_flight: int = 1):
        if comps is None:
            api.render_frame_device(batch, vp_t, cam_t, cfg_lanes if in_flight > 1 else cfg_async, VD, lanes[l])
        else:
            # the hand-off rides in the frame's own launch graph: the setup kernel waits for the acknowledgement, a 1-thread node
            # behind the raster kernel publishes the stripe, GPU0's raster kernel waits for all of them and hands the buffer back
            k = lane_frame_no[l]
            fused = comps[l].render(batch, vp_t, cam_t, cfg_stripe_lanes if in_flight > 1 else cfg, VD, k,
                                    compose_release=k if rank == 0 else None)
            if rank == 0 and not fused:
                comps[l].complete_and_release(k)
        lane_frame_no[l] += 1

    def check_lanes():
        lanes.synchronize()
        for cp in comps or []:
            cp.check()
        for c in lanes.ctxs:
            api.frame_stats(c)  # surfaces an overflow of an async frame, if any

    host_submit = [0.0, 0]  # seconds spent inside the submitting call, calls

    ev_pool = []  # timing events are created ahead of the timed loops: creating one costs the host ~2 us

    def take_event():
        return ev_pool.pop() if ev_pool else torch.cuda.Event(enable_timing=True)

    def timed_groups(n_frames: int, n_lanes: int):
        """n_frames frames in groups of one frame per lane; every group starts behind an L2 flush.  Device ms, summed over the
        groups: from the end of the flush to the end of the group's last frame."""
        n_groups = (n_frames + n_lanes - 1) // n_lanes
        while len(ev_pool) < n_groups * (n_lanes + 1):
            ev_pool.append(torch.cuda.Event(enable_timing=True))
        groups = []
        done = 0
        perf = time.perf_counter
        while done < n_frames:
            g = min(n_lanes, n_frames - done)
            flush_l2()
            f_ev = take_event()
            f_ev.record(lane_streams[0])
            ends = []
            for l in range(1, g):
                lane_streams[l].wait_event(f_ev)
            t_h = perf()
            for l in range(g):
                step_device(l, n_lanes)
            host_submit[0] += perf() - t_h
            host_submit[1] += g
            for l in range(g):
                e = take_event()
                e.record(lane_streams[l])
                ends.append(e)
            for l in range(1, g):
                lane_streams[0].wait_event(ends[l])  # the next flush starts when every lane is done
            groups.append((f_ev, ends))
            done += g
        torch.cuda.synchronize()
        total = sum(max(f_ev.elapsed_time(e) for e in ends) for f_ev, ends in groups)
        for f_ev, ends in groups:
            ev_pool.append(f_ev)
            ev_pool.extend(ends)
        return total

    # ---- warm-up ---------------------------------------------------------------------------------------------------
    Wm = max(3, args.warmup)
    for _ in range(Wm):
        for l in range(L):
            step_device(l, L)
    check_lanes()
    launches_per_frame = None

    # ---- timed region: exactly K frames, L in flight; CUDA events on the launching streams, L2 flushed before every group ----
    sampler = ClockSampler(local_rank)
    barrier()
    torch.cuda.synchronize()
    sampler.start()
    K = max(1, args.steps)
    l0 = lanes.launch_count
    total_ms = timed_groups(K, L)
    l1 = lanes.launch_count
    launches_per_frame = (l1 - l0) / K
    extra["host_submit_us_per_frame"] = host_submit[0] / max(1, host_submit[1]) * 1e6  # rank 0's; the device path is asynchronous
    if world_size > 1:
        log(f"rank {rank}: host submit {host_submit[0] / max(1, host_submit[1]) * 1e6:.1f} us per frame")
        extra["host_submit_us_per_frame_max_over_ranks"] = max_over_ranks(host_submit[0] / max(1, host_submit[1]) * 1e6)
    for cp in comps or []:
        cp.check()
    last_frame = None
    if args.dump_outputs:
        # the last timed frame, read back from the lane that rendered it (timed_groups has synchronised the device)
        dc, dd, rows_, width_ = api.framebuffer_device(lanes[(K - 1) % L])
        assert (rows_, width_) == (H, W)
        last_frame = (multigpu.device_bytes_as_tensor(dc, W * H * 4, dev).cpu().numpy().view(np.uint32).reshape(H, W),
                      multigpu.device_bytes_as_tensor(dd, W * H * 4, dev).cpu().numpy().view(np.float32).reshape(H, W))
    # keep the same load running until the sampler has seen >= 1.5 s of it (the timed frames are ~tens of microseconds)
    t_probe = time.perf_counter()
    while time.perf_counter() - t_probe < 1.5:
        for i in range(60):  # this rank's frames only: a time-based loop must not contain cross-rank waits
            api.render_frame_device(batch, vp, cam.position, cfg_lanes, VD, lanes[i % L])
        lanes.synchronize()
    clocks = sampler.stop()
    barrier()
    torch.cuda.synchronize()
    ms_per_step = max_over_ranks(total_ms) / K
    fps = 1000.0 / ms_per_step
    check_lanes()
    # the same frames one at a time (one lane, L2 flushed before each): the latency of a frame
    if L > 1:
        n_alone = min(K, 100)
        barrier()
        alone_ms = max_over_ranks(timed_groups(n_alone, 1)) / n_alone
        check_lanes()
    else:
        alone_ms = ms_per_step
    if comps is not None:
        # what the hand-off costs: the same stripes, same lanes, rendered into this GPU's own buffers with no flags
        cfg_local = api.VxFrameConfig.from_buffer_copy(cfg_lanes)
        cfg_local.stripe_y0, cfg_local.stripe_rows = stripes[rank]
        saved_comps, comps = comps, None
        saved_cfg, cfg_lanes = cfg_lanes, cfg_local
        try:
            if stripes[rank][1] > 0:
                for c in lanes.ctxs:
                    api.render_frame_device(batch, vp, cam.position, cfg_local, VD, c)
                lanes.synchronize()
                own_ms = timed_groups(K, L) / K
            else:
                own_ms = 0.0
            # ... and the same with the stripe stored into GPU0's frame (peer stores over NVLink), still without flags
            peer_ms = 0.0
            if stripes[rank][1] > 0:
                off = stripes[rank][0] * W * 4
                step_saved = step_device

                def step_peer(l: int = 0, in_flight: int = 1):
                    api.render_frame_into(batch, vp, cam.position, cfg_local, VD, saved_comps[l].color_ptr(0) + off, 0, lanes[l])

                step_device = step_peer
                try:
                    for l in range(L):
                        step_peer(l)
                    lanes.synchronize()
                    peer_ms = timed_groups(K, L) / K
                finally:
                    step_device = step_saved
        finally:
            comps, cfg_lanes = saved_comps, saved_cfg
        log(f"rank {rank}: stripe into GPU0's frame without flags {peer_ms * 1e3:.1f} us per frame")
        extra["stripe_ms_peer_stores_no_flags_this_rank"] = peer_ms
        log(f"rank {rank}: composited frames {total_ms / K * 1e3:.1f} us per frame on this rank, own stripe without hand-off {own_ms * 1e3:.1f} us")
        barrier()
        extra["stripe_ms_without_handoff_max_over_ranks"] = max_over_ranks(own_ms)
        extra["stripe_ms_composited_this_rank"] = total_ms / K
    extra["frame_alone_ms"] = alone_ms
    extra["frames_per_sec_one_frame_in_flight"] = 1000.0 / alone_ms
    frame_no = lane_frame_no[0]

    # ---- N > 1 guards (outside the timed region): the composed frame equals this GPU's own full frame, bit for bit;
    #      the assembled batch equals a locally meshed one ------------------------------------------------------------
    if comp is not None:
        lanes.synchronize()
        barrier()
        gcomp = multigpu.StripeCompositor(ctx, W, H, rank, world_size, want_depth=True)  # colour + depth, same stripes
        gcomp.set_stripes(stripes)
        k = 0
        gcomp.render(batch, vp, cam.position, cfg, VD, k)
        if rank == 0:
            gcomp.complete(k)
            ctx.synchronize()
            gcomp.check()
            got_c = gcomp.frame_tensor(k, dev).cpu().numpy().view(np.uint32)
            got_d = gcomp.depth_tensor(k, dev).cpu().numpy().view(np.uint32)
            gcomp.release(k)
            local = mesh_full_locally()
            api.render_frame_device(local, vp, cam.position, cfg, VD, ctx)
            dc, dd, rows_, width_ = api.framebuffer_device(ctx)
            ref_c = multigpu.device_bytes_as_tensor(dc, W * H * 4, dev).cpu().numpy().view(np.uint32).reshape(H, W)
            ref_d = multigpu.device_bytes_as_tensor(dd, W * H * 4, dev).cpu().numpy().view(np.uint32).reshape(H, W)
            extra["composite_bit_identical"] = bool(np.array_equal(got_c, ref_c) and np.array_equal(got_d, ref_d))
            extra["composite_covered_pixels"] = int((ref_c != cfg.clear_color).sum())
            a_, b_ = batch.download(), local.download()
            same = all(np.array_equal(a_[kk], b_[kk]) for kk in ("quad_count", "slice_offsets", "face_aabb", "has_mesh"))
            for i in np.flatnonzero(b_["has_mesh"]):
                same = same and np.array_equal(a_["quads"][int(a_["quad_base"][i]):int(a_["quad_base"][i]) + int(a_["quad_count"][i])],
                                               b_["quads"][int(b_["quad_base"][i]):int(b_["quad_base"][i]) + int(b_["quad_count"][i])])
            extra["sharded_batch_bit_identical"] = bool(same)
            local.release()
        ctx.synchronize()
        barrier()
        gcomp.close()

    # ---- chunk-sharded remesh sweep (BASELINE cfg 4): rank r re-meshes the lattice chunks k with k % N == r, the packed
    #      shards are all-gathered (NCCL) and every rank rebuilds the full batch -- the exchange is inside the timed region
    sharded = None
    if exchange is not None:
        for _ in range(2):
            exchange.sweep(d_voxf.data_ptr(), d_posf.data_ptr(), d_nbf.data_ptr(), d_flf.data_ptr())
        ctx.synchronize()
        barrier()
        sh_ms = []
        for _ in range(10):
            flush_l2()
            a, b2 = event_pair(torch)
            a.record(stream)
            exchange.sweep(d_voxf.data_ptr(), d_posf.data_ptr(), d_nbf.data_ptr(), d_flf.data_ptr())
            b2.record(stream)
            torch.cuda.synchronize()
            sh_ms.append(a.elapsed_time(b2))
        shard_ms = max_over_ranks(float(np.mean(sh_ms)))
        # the same shard without the exchange (what round 1 reported)
        ne_ms = []
        for _ in range(10):
            flush_l2()
            a, b2 = event_pair(torch)
            a.record(stream)
            api.BinaryGreedyMesher.mesh_batch_subset(d_voxf.data_ptr(), d_posf.data_ptr(), d_nbf.data_ptr(), d_flf.data_ptr(), n_lattice,
                                                     exchange.d_ids.data_ptr(), int(exchange.ids.size), ctx, batch=exchange.shard)
            b2.record(stream)
            torch.cuda.synchronize()
            ne_ms.append(a.elapsed_time(b2))
        noex_ms = max_over_ranks(float(np.mean(ne_ms)))
        sharded = {"lattice_chunks": n_lattice, "varied_chunks": n_varied, "ms_with_exchange_max_over_ranks": shard_ms,
                   "varied_chunks_meshed_per_sec_with_exchange": n_varied / (shard_ms * 1e-3),
                   "ms_mesh_only_max_over_ranks": noex_ms, "exchanged_bytes_per_rank": int(exchange.exchanged_bytes),
                   "shards_fitted_their_blocks": bool(exchange.check()),
                   "how": f"chunk id modulo {world_size}; per sweep, no host round trip: mesh kernel on the shard, vx_mesh_shard_pack_async (the block "
                          "carries the shard's quad total), ONE NCCL all_gather_into_tensor of the shard blocks, vx_mesh_batch_assemble_shards_async "
                          "on every rank (the first sweep sized the blocks through the synchronous pair)"}

    # ---- alternate-frame rendering (every rank renders whole frames, no exchange): context only, not the headline ---------
    afr_fps = None
    if world_size > 1:
        for _ in range(3):
            api.render_frame_device(batch, vp, cam.position, cfg_async, VD, ctx)
        ctx.synchronize()
        barrier()
        torch.cuda.synchronize()
        tot = 0.0
        prs = [event_pair(torch) for _ in range(K)]
        for a, b2 in prs:
            flush_l2()
            a.record(stream)
            api.render_frame_device(batch, vp, cam.position, cfg_async, VD, ctx)
            b2.record(stream)
        torch.cuda.synchronize()
        tot = sum(a.elapsed_time(b2) for a, b2 in prs)
        afr_fps = world_size * K / (max_over_ranks(tot) * 1e-3)
        api.frame_stats(ctx)

    # ---- e2e at N > 1: VP + camera + config in on every rank, stripes stored into GPU0's frame, GPU0 copies the composed
    #      ARGB frame into page-locked host memory -- every step; two frames in flight; wall clock, max over ranks ----------
    e2e_multi = None
    if comps is not None:
        # per lane four composite buffers: frame k of a lane is being composed while its frame k - 1 leaves GPU0 over the copy
        # engine (second stream); a buffer is handed back two lane-steps later, when its frame is known to be in host memory
        lanes.synchronize()
        barrier()
        for cp in comps:
            cp.close()
        Lm = max(1, min(L, args.e2e_lanes))  # lanes of the e2e loop (PCIe-bound from three on)
        extra["e2e_lanes"] = Lm
        comps = [multigpu.StripeCompositor(c, W, H, rank, world_size, want_depth=False, n_buffers=4) for c in lanes.ctxs[:Lm]]
        for cp in comps:
            cp.set_stripes(stripes)
        comp = comps[0]
        host = [[ctx.host_array((H, W), np.int32) for _ in range(2)] for _ in range(Lm)] if rank == 0 else None
        host_t = [[torch.from_numpy(hh) for hh in hl] for hl in host] if rank == 0 else None
        copy_streams = [torch.cuda.Stream(device=dev) for _ in range(Lm)]
        composed = [[torch.cuda.Event() for _ in range(2)] for _ in range(Lm)]
        copied = [[torch.cuda.Event() for _ in range(2)] for _ in range(Lm)]
        submitted = [[torch.cuda.Event() for _ in range(2)] for _ in range(Lm)]
        lane_k = [0] * Lm
        D = max(1, min(2 * Lm, args.e2e_depth if args.e2e_depth > 0 else Lm))  # frames in flight on the host (at most two per lane)

        def e2e_submit(j):
            l = j % Lm
            k = lane_k[l]
            lane_k[l] += 1
            # the lane's frame k - 2 is in host memory already (the host waited for it before submitting this one), so GPU0's
            # raster kernel of frame k can hand that buffer back itself once every stripe of frame k has arrived
            fused = comps[l].render(batch, vp, cam.position, cfg_stripe_lanes, VD, k, compose_release=(k - 2 if k >= 2 else -1) if rank == 0 else None)
            if rank == 0:
                if not fused:
                    if k >= 2:
                        comps[l].complete_and_release(k, k - 2)
                    else:
                        comps[l].complete(k)
                composed[l][k & 1].record(lane_streams[l])
                with torch.cuda.stream(copy_streams[l]):
                    copy_streams[l].wait_event(composed[l][k & 1])
                    host_t[l][k & 1].copy_(comps[l].frame_tensor(k, dev), non_blocking=True)
                    copied[l][k & 1].record(copy_streams[l])
            submitted[l][k & 1].record(lane_streams[l])

        def e2e_wait(j):
            l, k = j % Lm, j // Lm
            (copied if rank == 0 else submitted)[l][k & 1].synchronize()

        def e2e_run(n):
            for j in range(n):
                e2e_submit(j)
                if j >= D - 1:
                    e2e_wait(j - (D - 1))  # rank 0: that frame is complete in host memory
            for j in range(max(0, n - (D - 1)), n):
                e2e_wait(j)

        e2e_run(4 * Lm)
        for l in range(Lm):  # e2e_wait derives a lane's frame number from the run-local index: keep both in step
            assert lane_k[l] % 2 == 0
        ne2e = max(20, min(K, 200))
        ne2e -= ne2e % (2 * Lm)
        base_k = list(lane_k)

        def e2e_wait(j):  # noqa: F811 -- the timed run continues the lanes' frame numbers
            l, k = j % Lm, base_k[j % Lm] + j // Lm
            (copied if rank == 0 else submitted)[l][k & 1].synchronize()

        barrier()
        t0 = time.perf_counter()
        e2e_run(ne2e)
        el = time.perf_counter() - t0
        barrier()
        e2e_multi = ne2e / max_over_ranks(el)
        lanes.synchronize()
        for cp in comps:
            cp.check()
        if rank == 0:
            extra["e2e_frames_identical"] = bool(all(torch.equal(host_t[0][0], host_t[l][b]) for l in range(Lm) for b in range(2)))

    # ---- BASELINE cfg 5 (3840x2160, view distance 32): 1 GPU, and at N > 1 the stripe frame with / without the composite ---
    cfg5 = None
    try:
        cfg5 = bench_cfg5(torch, api, multigpu, sharding, ctx, stream, dev, rank, world_size, dist, flush_l2, max_over_ranks, barrier)
    except Exception as e:  # never let the context line break the headline
        cfg5 = {"error": repr(e)}
        log("cfg5 failed:", repr(e))

    if rank != 0:
        for cp in comps or []:
            cp.close()
        lanes.close()
        return teardown(torch, dist, ctx, [batch] if exchange is None else [], exchange)

    # =============================== rank 0 only from here ===============================================================
    # ---- warm-L2 back-to-back throughput (how the path is used in a render loop) --------------------------------
    e0, e1 = event_pair(torch)
    nb2b = 200
    ctx.synchronize()
    e0.record(stream)
    for _ in range(nb2b):
        api.render_frame_device(batch, vp, cam.position, cfg_async, VD, ctx)
    e1.record(stream)
    torch.cuda.synchronize()
    b2b_ms = e0.elapsed_time(e1) / nb2b

    # ---- per-kernel split (CUDA events inside the library), L2 flushed: this rank's share of the frame ---------------
    cfg_prof = api.VxFrameConfig.from_buffer_copy(cfg)
    cfg_prof.stripe_y0, cfg_prof.stripe_rows = (stripes[rank] if world_size > 1 else (0, 0))
    cfg_prof.profile_kernels = 1
    ksum = np.zeros(4)
    nprof = 20
    for _ in range(nprof):
        flush_l2()
        api.render_frame_device(batch, vp, cam.position, cfg_prof, VD, ctx)
        ksum += api.frame_kernel_times(ctx)
    kms = ksum / nprof
    knames = ["frame_cull_kernel", "frame_setup_kernel", "(unused)", "frame_raster_kernel"]
    top = int(np.argmax(kms))
    st = api.frame_stats(ctx)

    # algorithmic bytes (SURVEY.md 8d): framebuffer written once (colour u32 + depth f32, clear fused), visible quad
    # streams + mesh headers read once, chunk table read once (16 B) + visibility (4 B) per loaded chunk
    rows_mine = stripes[rank][1] if world_size > 1 else H
    b_fb = W * rows_mine * 8
    b_quads = 3 * st.n_quads + 936 * st.n_survivors
    b_cull = 20 * n_lattice
    b_frame_full = W * H * 8 + 3 * st_full.n_quads + 936 * st_full.n_survivors + b_cull
    peak, peak_src = measured_peaks()
    top_bytes = {0: b_cull, 1: b_quads, 2: 0, 3: b_fb + b_quads}[top]
    achieved = top_bytes / (kms[top] * 1e-3) / 1e9 if kms[top] > 0 else 0.0

    # ---- e2e through the host API at N = 1: api.FrameLoop, pipelined (vx_render_frame_begin / _end): VP + camera + config in,
    #      the ARGB frame + draw order land in page-locked host memory EVERY step; frame k + 1 is enqueued before the host waits
    #      for frame k (main.rs:320-336 overlaps present and the next iteration the same way) -----------------------------------
    h2d = 16 * 4 + 3 * 4 + C.sizeof(api.VxFrameConfig)
    d2h = W * H * 4 + 4 * n_lattice + 64  # frame + draw order + control block
    e2e_val, e2e_sync, e2e_note = None, None, None
    if world_size == 1:
        Le = max(1, min(L, args.e2e_lanes))  # the host loop is PCIe-bound from three lanes on; more only deepen the queue
        extra["e2e_lanes"] = Le
        loop = api.FrameLoop(batch, cfg, view_distance=VD, want_depth=False, ctx=ctx, lanes=Le)
        for _ in range(3):
            c_sync, _, s_sync = loop.render(vp, cam.position)
        ref_frame, ref_order = c_sync.copy(), s_sync.copy()
        ne2e = max(20, min(K, 200))
        ctx.synchronize()
        t0 = time.perf_counter()
        for _ in range(ne2e):
            loop.render(vp, cam.position)
        e2e_sync = ne2e / (time.perf_counter() - t0)
        D = max(1, min(2 * Le, args.e2e_depth if args.e2e_depth > 0 else Le))  # frames in flight on the host (measured: deeper queues only add latency)
        extra["e2e_frames_in_flight"] = D

        def e2e_run(n):
            ok_, pend = True, []
            for _ in range(n):
                pend.append(loop.submit(vp, cam.position))
                if len(pend) >= D:
                    c_, _, s_ = loop.wait(pend.pop(0))  # that frame is complete in host memory here
                    ok_ = bool(ok_ and c_[H // 2, W // 2] == ref_frame[H // 2, W // 2])
            while pend:
                c_, _, s_ = loop.wait(pend.pop(0))
                ok_ = ok_ and bool(np.array_equal(c_, ref_frame) and np.array_equal(s_, ref_order))  # the last D frames in full
            return bool(ok_)

        e2e_run(4 * Le)
        t0 = time.perf_counter()
        ok = e2e_run(ne2e)
        e2e_val = ne2e / (time.perf_counter() - t0)
        extra["e2e_pipelined_frames_identical_to_synchronous"] = ok
        extra["e2e_synchronous_frames_per_s"] = e2e_sync
        extra["e2e_d2h_GBps"] = e2e_val * d2h / 1e9
        if not ok:
            e2e_val = e2e_sync
        e2e_note = (f"api.FrameLoop(lanes={Le}).submit / wait -> vx_render_frame_begin / _end: VP + camera + config in; the frame is rendered into a "
                    "device buffer of its in-flight slot and leaves over the copy engine on a second stream, the ARGB frame, the draw order and "
                    f"the frame's control block land in page-locked host memory every step; {Le} lanes, {D} frames in flight on the host (the "
                    "oldest is waited for before another is enqueued); the loop is bound by the PCIe transfer of the frame "
                    "(extra.e2e_d2h_GBps); colour only -- the depth plane is frame-internal (the reference presents color_buffer only, "
                    "main.rs:320-322); extra.e2e_synchronous_frames_per_s = one blocking vx_render_frame per step")
    else:
        e2e_val = e2e_multi
        extra["e2e_d2h_GBps"] = e2e_val * d2h / 1e9
        e2e_note = ("per step every rank gets VP + camera + config and renders its stripe (vx_render_frame_stripe) straight into GPU0's frame over "
                    "NVLink; GPU0's raster kernel waits for the arrival words, the composed ARGB frame goes to page-locked host memory over the copy "
                    f"engine (second stream), a buffer is acknowledged two lane-steps later (four buffers per lane); {extra.get('e2e_lanes')} lanes, as many frames in "
                    "flight on the host; wall clock between barriers, max over ranks")

    # ---- second BASELINE metric: chunks meshed / s (whole-world remesh sweep of the Varied chunks, inputs resident) ----
    d_vox = torch.from_numpy(v).to(dev)
    d_nb = torch.from_numpy(nb).to(dev)
    d_pos = torch.from_numpy(p).to(dev)
    hv = C.c_void_p()
    ctx.check(ctx.lib.vx_mesh_chunks_device(ctx.handle, C.c_void_p(d_vox.data_ptr()), C.c_void_p(d_pos.data_ptr()), C.c_void_p(d_nb.data_ptr()),
                                            None, n_varied, C.byref(hv)))
    vbatch = api.MeshBatch(ctx, hv)

    def remesh():
        ctx.check(ctx.lib.vx_remesh_chunks_device(ctx.handle, C.c_void_p(d_vox.data_ptr()), C.c_void_p(d_nb.data_ptr()), None, vbatch.handle))

    for _ in range(3):
        remesh()
    ctx.synchronize()
    m_ms = []
    for _ in range(20):
        flush_l2()
        a, b = event_pair(torch)
        a.record(stream)
        remesh()
        b.record(stream)
        torch.cuda.synchronize()
        m_ms.append(a.elapsed_time(b))
    mesh_ms = float(np.mean(m_ms))
    chunks_per_s = n_varied / (mesh_ms * 1e-3)
    n_nbr = int((nb >= 0).sum())
    b_mesh = n_varied * (32768 + 792 + 144) + 1024 * n_nbr + 3 * total_quads
    mesh_gbs = b_mesh / (mesh_ms * 1e-3) / 1e9

    # large-batch meshing (BASELINE cfg 1 replicated: one terrain chunk, no neighbours, 16,384 copies = 512 MiB > L2), for the
    # chunk with the most quads of the world (worst case of the sweep) and for the median one
    rep = 16384
    qc_all = vbatch.download()["quad_count"]

    def big_batch(idx):
        d_big = d_vox[idx].repeat(rep, 1).contiguous()
        hb = C.c_void_p()
        ctx.check(ctx.lib.vx_mesh_chunks_device(ctx.handle, C.c_void_p(d_big.data_ptr()), None, None, None, rep, C.byref(hb)))
        big = api.MeshBatch(ctx, hb)
        quads = int(big.info().total_quads)
        bm = []
        for _ in range(5):
            a, b = event_pair(torch)
            a.record(stream)
            ctx.check(ctx.lib.vx_remesh_chunks_device(ctx.handle, C.c_void_p(d_big.data_ptr()), None, None, big.handle))
            b.record(stream)
            torch.cuda.synchronize()
            bm.append(a.elapsed_time(b))
        ms = float(np.mean(bm[1:]))
        big.release()
        del d_big
        return rep / (ms * 1e-3), (rep * (32768 + 792 + 144) + 3 * quads) / (ms * 1e-3) / 1e9, quads // rep

    big_cps, big_gbs, big_q = big_batch(int(np.argmax(qc_all)))
    med_cps, med_gbs, med_q = big_batch(int(np.argsort(qc_all)[len(qc_all) // 2]))

    # ---- meshing end to end in the steady state: the world's voxels come from page-locked host memory every sweep ----------
    mesh_e2e = None
    if world_size == 1:
        try:
            hv_t = torch.from_numpy(v).pin_memory()

            def sweep():
                with torch.cuda.stream(stream):
                    d_vox.copy_(hv_t, non_blocking=True)
                remesh()
                return vbatch.info().total_quads  # synchronises and reads the totals back

            for _ in range(3):
                sweep()
            t0 = time.perf_counter()
            reps = 20
            for _ in range(reps):
                tq_e2e = sweep()
            el = (time.perf_counter() - t0) / reps
            mesh_e2e = {"chunks_per_sec": n_varied / el, "ms_per_world": el * 1e3, "h2d_bytes_per_sweep": int(v.nbytes), "d2h_bytes_per_sweep": 32,
                        "quads": int(tq_e2e),
                        "note": f"{n_varied} x 32 KiB voxels H2D from page-locked memory + vx_remesh_chunks_device + totals read back, wall clock; PCIe-bound"}
            del hv_t
        except Exception as e:
            mesh_e2e = {"error": repr(e)}

    # ---- terrain generated on the device and meshed without ever crossing PCIe (SURVEY 8f N1): all lattice chunks --------
    gen_mesh = None
    if world_size == 1:
        try:
            d_voxg = torch.empty((n_lattice, 32768), dtype=torch.uint8, device=dev)
            tp = api.terrain_params()
            fl = api.generate_terrain(pos, d_voxg.data_ptr(), ctx, tp)
            d_flg = torch.from_numpy(fl).to(dev)
            hh = C.c_void_p()
            ctx.check(ctx.lib.vx_mesh_chunks_device(ctx.handle, C.c_void_p(d_voxg.data_ptr()), C.c_void_p(d_posf.data_ptr()),
                                                    C.c_void_p(d_nbf.data_ptr()), C.c_void_p(d_flg.data_ptr()), n_lattice, C.byref(hh)))
            bfull = api.MeshBatch(ctx, hh)
            same_world = int(bfull.info().total_quads) == total_quads
            ctx.synchronize()
            t0 = time.perf_counter()
            reps = 10
            for _ in range(reps):
                api.generate_terrain(pos, d_voxg.data_ptr(), ctx, tp)
                ctx.check(ctx.lib.vx_remesh_chunks_device(ctx.handle, C.c_void_p(d_voxg.data_ptr()), C.c_void_p(d_nbf.data_ptr()),
                                                          C.c_void_p(d_flg.data_ptr()), bfull.handle))
            ctx.synchronize()
            el = (time.perf_counter() - t0) / reps
            gen_mesh = {"chunks": n_lattice, "varied_chunks": n_varied, "ms_per_world": el * 1e3, "lattice_chunks_per_sec": n_lattice / el,
                        "same_quads_as_host_generated_world": bool(same_world),
                        "note": "vx_generate_terrain (all lattice positions -> voxels + Uniform flags on the device) + vx_remesh_chunks_device, wall clock"}
            bfull.release()
            del d_voxg
        except Exception as e:
            gen_mesh = {"error": repr(e)}

    a18 = None
    if world_size == 1:
        try:
            a18 = bench_adjacent(torch, api, ctx, stream, dev, vbatch, p, qc_all, vp, cam, cfg, loop)
        except Exception as e:  # noqa: BLE001
            a18 = {"error": repr(e)}

    # ---- CPU baseline beside it (bounded sample) -------------------------------------------------------------------
    threads = os.cpu_count() or 1
    cpu_fps, cpu_n, cpu_el, _, _ = cpu_frame_baseline(sc, 10.0, threads)
    cpu_cps, cpu_mn, cpu_mel = cpu_mesh_baseline(v, nb, 3.0)

    traffic = ncu_traffic(knames[top]) if world_size == 1 else None  # the committed capture is the 1-GPU full frame
    extra.update({
        "frame_ms_warm_l2_back_to_back": b2b_ms, "frames_per_sec_warm_l2": 1000.0 / b2b_ms,
        "kernel_ms": {k: float(x) for k, x in zip(knames, kms)},
        "kernel_ms_note": "CUDA events around each kernel (profile mode serialises them; the async path overlaps them by programmatic dependent launch)"
                          + ("" if world_size == 1 else "; rank 0's stripe"),
        "launches_per_step": launches_per_frame,
        "frame_stats": {"visible_meshes": int(st_full.n_survivors), "visible_quads": int(st_full.n_quads), "triangles": int(st_full.n_triangles),
                        "bin_entries": int(st_full.n_bin_entries)},
        "stripes": [list(s) for s in stripes],
        "frame_algorithmic_bytes": int(b_frame_full), "frame_hbm_frac": (b_frame_full / (ms_per_step * 1e-3) / 1e9) / peak,
        "chunks_meshed_per_sec": chunks_per_s, "remesh_world_ms": mesh_ms, "remesh_world_chunks": n_varied,
        "remesh_algorithmic_GBps": mesh_gbs, "remesh_hbm_frac": mesh_gbs / peak,
        "remesh_sharded": sharded,
        "chunks_meshed_per_sec_large_batch": big_cps, "large_batch": f"{rep} copies of the world's busiest terrain chunk ({big_q} quads), no neighbours (BASELINE configs[0] replicated, 512 MiB of voxels)",
        "chunks_meshed_per_sec_large_batch_median_chunk": med_cps, "median_chunk_quads": med_q,
        "large_batch_median_algorithmic_GBps": med_gbs, "large_batch_median_hbm_frac": med_gbs / peak,
        "large_batch_algorithmic_GBps": big_gbs, "large_batch_hbm_frac": big_gbs / peak,
        "cpu_chunks_meshed_per_sec_1_thread": cpu_cps,
        "cfg5_3840x2160_vd32": cfg5,
        "mesh_e2e_steady_state": mesh_e2e,
        "generate_and_mesh_on_device": gen_mesh,
        "adjacent_rasterizers_a18": a18,
        "frames_per_sec_alternate_frame_rendering": afr_fps,
        "alternate_frame_rendering": "N > 1 only: every GPU renders whole 1280x720 frames independently (no exchange), total frames / max time over ranks; context, not the headline",
        "reference_published": "162-168 fps on a 6-core i5-12400 (README.md:29-32)",
    })
    out = {
        "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": Wm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(world_size, sc, total_quads),
        "clocks": clocks,
        "gpu_launches": int(l1 - l0),
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "note": e2e_note},
        "roofline": {"bound": "hbm", "kernel": knames[top], "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(top_bytes), "kernel_ms": float(kms[top]),
                     "kernel_share_of_step": float(kms[top] / kms.sum()) if kms.sum() > 0 else None},
        "cpu_baseline": {"value": cpu_fps, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{cpu_n} full 1280x720 vd12 frames in {cpu_el:.1f} s; C restatement of the reference CPU path "
                                   f"(oracle/), stripe-parallel over all {threads} host threads; " + cargo_note()},
        "extra": extra,
    }
    if last_frame is not None:
        dump_outputs(args.dump_outputs, *last_frame)
    emit_json_line(out)
    if world_size == 1:
        del loop
    vbatch.release()
    for cp in comps or []:
        cp.close()
    lanes.close()
    return teardown(torch, dist, ctx, [batch] if exchange is None else [], exchange)


def teardown(torch, dist, ctx, batches, exchange):
    """Orderly exit: device work drained, library objects released while the context is alive, torch's cached blocks freed
    before the context's stream goes away, process group destroyed -- then main() leaves through the normal exit path."""
    rc = 0
    try:
        ctx.synchronize()
        torch.cuda.synchronize()
        for b in batches:
            b.release()
        if exchange is not None:
            exchange.close()
        if dist is not None:
            dist.barrier()
    except Exception as e:  # noqa: BLE001
        log("teardown:", repr(e))
        rc = 1
    return rc


def bench_cfg5(torch, api, multigpu, sharding, ctx, stream, dev, rank, world_size, dist, flush_l2, max_over_ranks, barrier):
    """3840x2160 view distance 32 (137,065 lattice chunks; the Varied ones are meshed on every rank): one GPU renders the whole
    frame; N GPUs render work-balanced stripes, timed with and without the peer-store composite."""
    import vx_scenes
    W5, H5, VD5 = 3840, 2160, 32
    pos5, world5, p5, v5, nb5 = vx_scenes.terrain_scene(VD5)
    batch5 = api.BinaryGreedyMesher.mesh_batch(v5, p5, nb5, None, ctx, validate=False)
    cam5 = vx_scenes.main_camera(W5, H5)
    vp5 = cam5.view_projection()
    c5 = api.default_frame_config(W5, H5)
    api.render_frame_device(batch5, vp5, cam5.position, c5, VD5, ctx)
    st5 = api.frame_stats(ctx)
    c5a = api.VxFrameConfig.from_buffer_copy(c5)
    c5a.async_submit = 1
    peak, _ = measured_peaks()
    bytes5 = W5 * H5 * 8 + 3 * st5.n_quads + 936 * st5.n_survivors + 20 * int(p5.shape[0])
    out = {"workload": "3840x2160 view distance 32 (137,065 lattice chunks, Varied ones meshed with neighbours), L2 flushed",
           "varied_chunks": int(p5.shape[0]), "visible_meshes": int(st5.n_survivors), "visible_quads": int(st5.n_quads),
           "triangles": int(st5.n_triangles), "algorithmic_bytes": int(bytes5)}

    def timed(fn, n=20):
        for _ in range(3):
            fn()
        ctx.synchronize()
        barrier()
        prs = []
        for _ in range(n):
            flush_l2()
            a, b = event_pair(torch)
            a.record(stream)
            fn()
            b.record(stream)
            prs.append((a, b))
        torch.cuda.synchronize()
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in prs)) / n

    if world_size == 1:
        ms5 = timed(lambda: api.render_frame_device(batch5, vp5, cam5.position, c5a, VD5, ctx))
        out.update({"frame_ms": ms5, "frames_per_sec": 1000.0 / ms5, "hbm_frac": bytes5 / (ms5 * 1e-3) / 1e9 / peak})
    else:
        band = api.frame_bin_counts(ctx).sum(axis=1).astype(np.float64)
        holder = [sharding.balanced_stripes(band, H5, world_size, band=8, row_cost=float(band.sum()) / (4.0 * H5))] if rank == 0 else [None]
        dist.broadcast_object_list(holder, src=0)
        stripes5 = [tuple(x) for x in holder[0]]
        # (a) every rank renders the whole frame (= the 1-GPU time on this box)
        ms_one = timed(lambda: api.render_frame_device(batch5, vp5, cam5.position, c5a, VD5, ctx))
        # (b) stripes into local memory, no composite
        cs = api.VxFrameConfig.from_buffer_copy(c5a)
        cs.stripe_y0, cs.stripe_rows = stripes5[rank]
        ms_stripe = timed(lambda: api.render_frame_device(batch5, vp5, cam5.position, cs, VD5, ctx)) if stripes5[rank][1] > 0 else timed(lambda: None)
        # (c) stripes stored into GPU0's frame over NVLink + arrival flags
        comp5 = multigpu.StripeCompositor(ctx, W5, H5, rank, world_size, want_depth=True)
        comp5.set_stripes(stripes5)
        kk = [0]

        def step():
            fused = comp5.render(batch5, vp5, cam5.position, c5, VD5, kk[0], compose_release=kk[0] if rank == 0 else None)
            if rank == 0 and not fused:
                comp5.complete_and_release(kk[0])
            kk[0] += 1

        ms_comp = timed(step)
        comp5.check()
        # guard: composed frame == this GPU's own whole frame
        k = kk[0]
        comp5.render(batch5, vp5, cam5.position, c5, VD5, k)
        same = None
        if rank == 0:
            comp5.complete(k)
            ctx.synchronize()
            got_c = comp5.frame_tensor(k, dev).cpu().numpy().view(np.uint32)
            got_d = comp5.depth_tensor(k, dev).cpu().numpy().view(np.uint32)
            comp5.release(k)
            api.render_frame_device(batch5, vp5, cam5.position, c5, VD5, ctx)
            dc, dd, _, _ = api.framebuffer_device(ctx)
            ref_c = multigpu.device_bytes_as_tensor(dc, W5 * H5 * 4, dev).cpu().numpy().view(np.uint32).reshape(H5, W5)
            ref_d = multigpu.device_bytes_as_tensor(dd, W5 * H5 * 4, dev).cpu().numpy().view(np.uint32).reshape(H5, W5)
            same = bool(np.array_equal(got_c, ref_c) and np.array_equal(got_d, ref_d))
        ctx.synchronize()
        barrier()
        comp5.close()
        out.update({"n_gpus": world_size, "stripes": [list(s) for s in stripes5],
                    "frame_ms_one_gpu_whole_frame": ms_one, "frame_ms_stripes_no_composite": ms_stripe,
                    "frame_ms": ms_comp, "frames_per_sec": 1000.0 / ms_comp, "composite_bit_identical": same,
                    "hbm_frac_per_gpu": bytes5 / world_size / (ms_comp * 1e-3) / 1e9 / peak,
                    "note": "frame_ms = work-balanced stripes, every raster kernel stores its rows (colour + depth) into GPU0's frame over NVLink, "
                            "GPU0 waits for the arrival flags; max over ranks"})
    api.frame_stats(ctx)
    # ---- BASELINE cfg 4 at this world's size: whole-world remesh sweep of the 5,877 Varied chunks (8 resident waves on one
    #      GPU), on one GPU and -- at N > 1 -- sharded by chunk id with the device exchange inside the timed region ----------
    try:
        n5 = int(p5.shape[0])
        d_v5 = torch.from_numpy(v5).to(dev)
        d_nb5 = torch.from_numpy(nb5).to(dev)
        d_p5 = torch.from_numpy(p5).to(dev)

        def remesh5():
            ctx.check(ctx.lib.vx_remesh_chunks_device(ctx.handle, C.c_void_p(d_v5.data_ptr()), C.c_void_p(d_nb5.data_ptr()), None, batch5.handle))

        ms_r1 = timed(remesh5, n=10)
        out["remesh_world_chunks"] = n5
        out["remesh_world_ms_one_gpu"] = ms_r1
        out["chunks_meshed_per_sec_one_gpu"] = n5 / (ms_r1 * 1e-3)
        if world_size > 1:
            ex5 = multigpu.MeshShardExchange(ctx, n5, rank, world_size, dev)
            ex5.sweep(d_v5.data_ptr(), d_p5.data_ptr(), d_nb5.data_ptr(), 0)
            ms_rs = timed(lambda: ex5.sweep(d_v5.data_ptr(), d_p5.data_ptr(), d_nb5.data_ptr(), 0), n=10)
            out["remesh_world_ms_sharded_with_exchange"] = ms_rs
            out["chunks_meshed_per_sec_sharded_with_exchange"] = n5 / (ms_rs * 1e-3)
            same5 = int(ex5.full.info().total_quads) == int(batch5.info().total_quads)
            out["sharded_world_same_quad_total"] = bool(same5)
            ex5.close()
        del d_v5, d_nb5, d_p5
    except Exception as e:  # noqa: BLE001 -- context numbers only
        out["remesh_error"] = repr(e)
    batch5.release()
    del v5, world5
    return out


def bench_adjacent(torch, api, ctx, stream, dev, batch, p, qc_all, vp, cam, cfg, loop):
    """Adjacent rasterizers (SURVEY 8a row a18): the reference's own span-walker bench case, the macrotile frame, the Hyper-Pipeline."""
    from oracle import binding as ob18
    sw_w, sw_h = 1920, 1080  # benches/span_walker.rs:36-77 "span_walker_full_packet_32_quads": a 4 x 8 grid of quads
    ii = np.arange(32)
    bx0 = (np.float32(-0.9) + (ii % 8).astype(np.float32) * np.float32(0.225)).astype(np.float32)
    by0 = (np.float32(-0.9) + (ii // 8).astype(np.float32) * np.float32(0.45)).astype(np.float32)
    bx1 = (bx0 + np.float32(0.2)).astype(np.float32)
    by1 = (by0 + np.float32(0.4)).astype(np.float32)
    bz = np.full(32, 0.5, dtype=np.float32)
    bt = ((ii % 4) + 1).astype(np.uint8)
    d_boxes = torch.from_numpy(np.concatenate([bx0, by0, bx1, by1, bz])).to(dev)
    d_types = torch.from_numpy(np.concatenate([bt, np.ones(32, dtype=np.uint8)])).to(dev)
    d_col = torch.zeros((sw_h, sw_w), dtype=torch.int32, device=dev)
    d_dep = torch.full((sw_h, sw_w), float("inf"), dtype=torch.float32, device=dev)

    def walk():
        ctx.check(ctx.lib.vx_span_walk_quads_device(ctx.handle, C.c_void_p(d_boxes.data_ptr()), C.c_void_p(d_types.data_ptr()), 32, sw_w, sw_h,
                                                    C.c_void_p(d_col.data_ptr()), C.c_void_p(d_dep.data_ptr())))

    walk()  # first call draws; the repeats below re-test equal depths like the reference's bench loop does
    ctx.synchronize()
    oc18 = np.zeros((sw_h, sw_w), dtype=np.uint32)
    od18 = np.full((sw_h, sw_w), np.inf, dtype=np.float32)
    ob18.span_walk_quads(oc18, od18, bx0, by0, bx1, by1, bz, bt)
    same18 = bool(np.array_equal(d_col.cpu().numpy().view(np.uint32), oc18))
    sw_ms = []
    for _ in range(10):
        a, b = event_pair(torch)
        a.record(stream)
        walk()
        b.record(stream)
        torch.cuda.synchronize()
        sw_ms.append(a.elapsed_time(b))
    t0 = time.perf_counter()
    for _ in range(5):
        ob18.span_walk_quads(oc18, od18, bx0, by0, bx1, by1, bz, bt)
    sw_cpu_ms = (time.perf_counter() - t0) / 5 * 1e3
    # macrotile frame of the headline scene: caller's list = every meshed chunk that passes filter A
    vis18 = api.get_visible_chunks_frustum(p, cam.position, vp, VD, True, ctx)
    ids18 = np.flatnonzero((vis18 != 0) & (qc_all > 0)).astype(np.int32)
    cfg_m = api.VxFrameConfig.from_buffer_copy(cfg)
    cfg_m.macrotile = 1
    cfg_m.async_submit = 0
    mt_ms = []
    api.render_frame(batch, vp, cam.position, cfg_m, mesh_ids=ids18, ctx=ctx)
    for _ in range(10):
        t0 = time.perf_counter()
        api.render_frame(batch, vp, cam.position, cfg_m, mesh_ids=ids18, want_depth=False, color_out=loop.color, ctx=ctx)
        mt_ms.append((time.perf_counter() - t0) * 1e3)
    # Hyper-Pipeline (benches/differential_projection.rs:8-36 scene; host framebuffers in and out, wall clock)
    import vx_kat
    hb = api.BinaryGreedyMesher.mesh_batch(vx_kat.chunk_slab().reshape(1, -1), [(0, 0, 0)], None, None, ctx)
    from differential_projection_voxel_renderer_b200 import camera as _cam
    hvp = _cam.mat4_mul(_cam.perspective_rh(np.radians(np.float32(70.0)), 16 / 9, 0.1, 1000.0),
                        _cam.look_at_rh((64.0, 50.0, 100.0), (64.0, 32.0, 64.0), (0.0, 1.0, 0.0))).reshape(16)
    hfb = api.Framebuffer(1280, 720)
    hyper_quads = api.hyper_pipeline_render(hb, [0], hvp, hfb, ctx)
    hp_ms = []
    for _ in range(5):
        hfb = api.Framebuffer(1280, 720)
        t0 = time.perf_counter()
        api.hyper_pipeline_render(hb, [0], hvp, hfb, ctx)
        hp_ms.append((time.perf_counter() - t0) * 1e3)
    hb.release()
    return {"hyper_pipeline_1280x720_one_chunk_ms": float(np.median(hp_ms)), "hyper_pipeline_visible_quads": hyper_quads,
            "span_walker_full_packet_32_quads_1920x1080_ms": float(np.median(sw_ms)), "span_walker_cpu_port_ms": sw_cpu_ms,
            "span_walker_matches_oracle": same18, "span_walker_launches": 5,
            "macrotile_frame_1280x720_vd12_e2e_ms": float(np.median(mt_ms)), "macrotile_meshes": int(ids18.size),
            "note": "vx_span_walk_quads_device (benches/span_walker.rs:36-77 workload, framebuffer resident) and vx_render_frame with cfg.macrotile = 1 (render_frame_macrotile) through the host API into mapped host memory, wall clock"}


_REAL_STDOUT_FD = None


def emit_json_line(obj):
    """The ONE line of the contract, on the process's real stdout."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT_FD, line)


def main():
    # Libraries (NCCL's version banner, for one) print to file descriptor 1.  stdout must carry exactly one JSON line, so
    # fd 1 is pointed at stderr for the whole run and the result line is written to a saved copy of the real stdout.
    global _REAL_STDOUT_FD
    sys.stdout.flush()
    _REAL_STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--lanes", type=int, default=8, help="frames in flight on each GPU (api.FrameLanes)")
    ap.add_argument("--e2e-lanes", type=int, default=3, help="lanes of the e2e host loop (at most --lanes)")
    ap.add_argument("--fused-signal", type=int, default=0, help="N > 1: 1 = every rank's raster kernel publishes its own arrival word")
    ap.add_argument("--composite-buffers", type=int, default=2, help="N > 1: composed-frame buffers per lane")
    ap.add_argument("--composite-depth", type=int, default=0, help="N > 1: 1 = the timed stripes also store their depth plane into GPU0's frame")
    ap.add_argument("--e2e-depth", type=int, default=0, help="frames in flight on the host in the e2e loop (default lanes, at most 2 * lanes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step (colour channels and depth, float32 .npy) into DIR")
    args = ap.parse_args()
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs needs a one-GPU run: at N > 1 the frame is composed across ranks")
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


def leave(rc: int):
    """Exit-time hooks first (the driver's loaded-library report among them), then leave without running static
    destructors: at that point torch would free cached device / page-locked blocks after the CUDA context is gone and abort a
    run that has completed."""
    import atexit
    sys.stdout.flush()
    sys.stderr.flush()
    try:
        atexit._run_exitfuncs()
    except Exception as e:  # noqa: BLE001
        print("exit hook raised:", repr(e), file=sys.stderr)
        rc = rc or 1
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(int(rc))


if __name__ == "__main__":
    try:
        _rc = main()
    except SystemExit as e:
        _rc = int(e.code or 0)
    except BaseException:  # noqa: BLE001
        import traceback
        traceback.print_exc()
        _rc = 1
    leave(int(_rc or 0))
