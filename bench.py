#!/usr/bin/env python
"""bench.py -- full frames/s (voxelize + mip + cone-trace) of the B200 path on BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1..5] [--mode ...]
                    [--dump-outputs DIR]

One process per GPU (torchrun for N > 1).  A step is one full frame: sparse clear -> voxelise (coverage + PCF-lit
shading) -> resolve -> mip pyramid -> primary visibility -> cone trace.  The default workload is config 2 (the one
BASELINE.json's metric is quoted on): the synthetic 260 K-triangle atrium at 256^3 / 1920x1080; the shadow map is
static (the reference draws it once at init) and is timed separately.  Rank 0 prints ONE JSON line.

With the default arguments the line also carries `strong_config3`: BASELINE config 3 (512^3 RGBA16F, 3840x2160, 9+1
cones) rendered as ONE frame stream sharded over the N ranks by the library's own multi-GPU layer (triangle shares +
NVSwitch multicast exchange + row bands written into rank 0's frame), next to its own one-GPU anchor measured in the
same run -- the strong-scaling curve; `value` at N > 1 is the replica (views) aggregate of config 2.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "frames/s"
DTYPE = "u8/u32 grid (f16 grid in config 3), f32 shading"
WORKLOADS = {
    1: "config1: procedural Cornell box 44 tris, 64^3 RGBA8 grid, 256x256, 6 diffuse + 1 specular cone (reference table), "
       "2 bounces (reference semantics), MSAA4 coverage (the reference's window), 1024^2 shadow map",
    2: "config2: synthetic Sponza-scale atrium 259608 tris (seed 1234), 256^3 RGBA8 grid, 1920x1080, "
       "6 diffuse + 1 specular cone (reference table), 2 bounces (reference semantics), conservative coverage, "
       "4096^2 shadow map",
    3: "config3: synthetic atrium 259608 tris, 512^3 RGBA16F grid, 3840x2160, 9 diffuse + 1 specular cone, conservative "
       "coverage, 4096^2 shadow map",
    4: "config4: dynamic 1048576-triangle knot re-generated on the device and re-voxelised every frame (shadow map redrawn "
       "every frame), 256^3 RGBA8 grid, 1920x1080, 6+1 cones, conservative coverage",
    5: "config5: light-probe bake, atrium 259608 tris, 256^3 RGBA8 grid, Bounces=3 (re-injection), 64 views at 1024x1024",
}


def metric_name(args):
    if args.config == 2 and args.grid == 256:
        return "full frames/s (voxelize+mip+cone-trace), 256^3 grid, 1920x1080"
    what = "views/s (one 3-bounce voxelisation per 64 views)" if args.config == 5 else "full frames/s (voxelize+mip+cone-trace)"
    return f"{what}, {args.grid}^3 grid, {args.width}x{args.height}"


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=None, choices=["views", "tiles", "trishard", "shard"],
                    help="N>1: views = one camera per rank, grid replicated (replicas, default for config 2); shard = ONE frame "
                         "stream sharded by the library (vct_comm_init / vct_frame_sharded: triangle shares exchanged over "
                         "NVSwitch multicast + row bands written into rank 0's frame; default for configs 3, 4); tiles = row bands, "
                         "voxelisation replicated, NCCL all-gather (baseline form); trishard = triangle ranges + NCCL all-reduce "
                         "of the dense accumulator (baseline form)")
    ap.add_argument("--serial-shard", action="store_true", help="--mode shard: voxelise / exchange / trace back to back on one stream "
                    "and gather with NCCL instead of the pipelined vct_frame_sharded")
    ap.add_argument("--contiguous", action="store_true", help="triangle sharding by contiguous ranges instead of interleaved blocks")
    ap.add_argument("--no-multicast", action="store_true", help="--mode shard: exchange by peer stores instead of multimem.st")
    ap.add_argument("--shard-shadow", action="store_true", help="--mode shard: triangle-sharded shadow map (every rank rasterises its "
                    "share, depth fragments min-reduced into all ranks' images through the switch); matters for config 4, where the map is redrawn every frame")
    ap.add_argument("--row-bands", action="store_true", help="--mode shard: contiguous row bands instead of interleaved strips of 8 rows")
    ap.add_argument("--exchange", default="inbox", choices=["inbox", "reduce"],
                    help="--mode shard: inbox = touched voxels multicast as records (multimem.st) and merged locally; reduce = "
                         "multimem.red into a dense symmetric accumulator (reduced in the switch; serial form only)")
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json config: 1 = Cornell 64^3 256x256 (per-pass GPU and CPU times); 2 = headline (default); "
                         "3 = 512^3 fp16 grid, 4K, 9+1 cones; 4 = dynamic 1M-triangle mesh re-voxelised every frame; "
                         "5 = light-probe bake: 64 views at 1024^2 from one 3-bounce voxelisation")
    ap.add_argument("--detail", type=float, default=1.0, help="scene tessellation scale (1.0 = config 2)")
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--width", type=int, default=0, help="override the config's frame width")
    ap.add_argument("--height", type=int, default=0, help="override the config's frame height")
    ap.add_argument("--tune", default="", help="comma-separated library tuning knobs, e.g. ChainBlockThreads=64,ConeSmemPad=8192")
    ap.add_argument("--coverage", default=None)
    ap.add_argument("--cones", default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the config-3 strong-scaling leg of the default run")
    ap.add_argument("--strong-steps", type=int, default=0, help="timed steps of the config-3 leg (default: min(steps, 40))")
    ap.add_argument("--flush", action="store_true", help="flush L2 between timed steps (per-step events, frames not pipelined); "
                    "default: no flush -- the per-frame working set (~220 MB, two alternating frame slots) exceeds the 126 MB L2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frame of the last timed step (config 5: its last probe view) as "
                         "DIR/frame.npy, float32 RGBA 0..255; a frame over 64 MB is written as DIR/frame_sample.npy, a fixed "
                         "seeded sample of 2^21 of its pixels.  Inputs are seeded, so two builds can be compared output for output")
    a = ap.parse_args(argv)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.shadow = 4096
    w0, h0 = 1920, 1080
    if a.config == 1:
        a.grid, w0, h0, a.shadow = 64, 256, 256, 1024
        a.coverage = a.coverage or "msaa4"
    elif a.config == 3:
        a.grid, w0, h0 = 512, 3840, 2160
        a.cones = a.cones or "9+1"
        a.mode = a.mode or ("shard" if a.gpus > 1 else "views")
    elif a.config == 4:
        a.mode = a.mode or ("shard" if a.gpus > 1 else "views")
    elif a.config == 5:
        w0, h0, a.mode = 1024, 1024, "probes"
    a.nominal_size = not (a.width or a.height)
    a.width, a.height = a.width or w0, a.height or h0
    a.coverage = a.coverage or "conservative"
    a.cones = a.cones or "6+1"
    a.mode = a.mode or "views"
    return a


def make_scene_and_uniforms(args):
    import vct_b200  # noqa: F401
    from vct_b200 import scenes, uniforms
    if args.config == 4:
        sc = scenes.dynamic_knot()
    elif args.config == 1:
        sc = scenes.cornell()
    else:
        sc = scenes.atrium(detail=args.detail)
    u = uniforms.scene_uniforms(sc, V=args.grid, width=args.width, height=args.height, shadow_map_size=args.shadow,
                                coverage=args.coverage, cones=args.cones, grid_format=1 if args.config == 3 else 0,
                                bounces=3 if args.config == 5 else 2)
    return sc, u


def camera_for(sc, step, rank):
    """Per-step input: a slow camera pan (every step has a new view matrix, as the reference's loop does).  In `views`
    mode every rank renders its own stream: the same pan, 17 steps apart per rank (distinct frames of near-identical
    cost, so that per-GPU work stays fixed as N grows)."""
    return sc.camera_pos, sc.yaw + 0.05 * (step + 17 * rank), sc.pitch


def set_camera(ctx, sc, step, rank):
    import vct_b200.glmath as gm
    pos, yaw, pitch = camera_for(sc, step, rank)
    view = gm.view_matrix(pos, yaw, pitch)
    ctx.set_mat4("ModelViewMatrix", gm.colmajor((view @ gm.scale(0.05)).astype(np.float32)))
    ctx.set_3f("CameraPosition", pos)
    return 64 + 12          # bytes of per-step input handed to the device (as kernel parameters)


class ClockSampler:
    """Samples nvidia-smi during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class Env:
    """Process-level plumbing: rank / world, device, ONE explicit stream for our kernels, torch's events and NCCL."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", 0)); self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.Stream(device=self.dev, priority=int(os.environ.get("VCT_MAIN_STREAM_PRIORITY", "0")))
        torch.cuda.set_stream(self.stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def all_true(self, ok):
        t = self.torch.tensor([1 if ok else 0], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t.item()))

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def session_name(tag):
    from vct_b200 import parallel
    return f"{parallel.default_session()}_{tag}"


# ------------------------------------------------------------------------------------------------ ours
def run_ours(args):
    import vct_b200
    vct_b200.load_library()                         # mandatory extension: raises if missing
    env = Env()
    out = bench_config(env, args)
    if args.config == 2 and args.mode == "views" and not args.no_strong and args.detail == 1.0 and args.grid == 256:
        k = args.strong_steps or min(args.steps, 40)
        try:
            strong = strong_config3(env, steps=k, warmup=max(3, min(args.warmup, 5)))
        except Exception as e:               # the headline line must survive a failure of the extra leg
            strong = {"error": f"{type(e).__name__}: {e}"}
        if out is not None:
            out["strong_config3"] = strong
    if out is not None:
        print(json.dumps(out), flush=True)
    env.close()


def bench_config(env, args):
    torch, dist = env.torch, env.dist
    import vct_b200
    from vct_b200 import capi, parallel
    rank, world, local, dev, stream = env.rank, env.world, env.local, env.dev, env.stream

    sc, u = make_scene_and_uniforms(args)
    ctx = vct_b200.Context(local)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_uniforms(u)
    for kv in filter(None, args.tune.split(",")):
        k, v = kv.split("=")
        ctx.set_i(k, int(v))
    ctx.load_scene(sc)
    H, W = args.height, args.width
    ctx.draw_depth()                                # static light: once, like the reference's init
    ctx.sync()
    depth_us = ctx.pass_time_us("depth")
    sharded = args.mode == "shard"
    pipelined_shard = sharded and args.exchange == "inbox" and not args.serial_shard
    band = None
    tri_rng = None
    shared = None
    if sharded:
        flags = (capi.COMM_NO_MULTICAST if args.no_multicast else 0) | (capi.COMM_ROW_BANDS if args.row_bands else 0)
        if args.shard_shadow:
            ctx.set_i("ShardShadowMap", 1)
        shared = parallel.SharedAccumulator(ctx, rank=rank, world=world, session=session_name(f"c{args.config}"),
                                            exchange=args.exchange, flags=flags)      # deals triangles + row bands
        if args.contiguous:
            tri_rng = parallel.triangle_share(ctx, sc.n_tris, rank, world, interleave=False)
        else:
            tri_rng = (0, sc.n_tris)
    if args.mode == "tiles" and world > 1:
        b0, b1, per = parallel.row_band_equal(H, rank, world)     # equal nominal bands: ONE all-gather per frame
        ctx.set_i("RowBegin", b0); ctx.set_i("RowEnd", b1)
    if args.mode == "trishard":
        tri_rng = parallel.triangle_share(ctx, sc.n_tris, rank, world, interleave=not args.contiguous)
    acc = parallel.accumulator_tensor(ctx, dev) if args.mode == "trishard" else None
    gather_buf = None
    if world > 1 and (args.mode == "tiles" or (sharded and not pipelined_shard)):
        b0, b1, per = parallel.row_band_equal(H, rank, world)
        band = (b0, b1, per)
        fptr, fbytes = ctx.frame_buffer()
        frame_t = torch.as_tensor(parallel._DevicePointer(fptr, fbytes, "|u1"), device=dev)
        chunk = per * W * 4
        gather_buf = torch.zeros(world * chunk, dtype=torch.uint8, device=dev)    # bands in frame order, padded at the end
        my_band = torch.zeros(chunk, dtype=torch.uint8, device=dev)
        own0, own1 = b0 * W * 4, b1 * W * 4

    dyn = None
    if args.config == 4:
        # the mesh is re-generated on the device every frame (time-varying sine displacement along the normal)
        base = torch.from_numpy(np.ascontiguousarray(sc.verts[:, :3])).to(dev)
        nrm = torch.from_numpy(np.ascontiguousarray(sc.verts[:, 3:6])).to(dev)
        phase = (base[:, 0] * 0.004 + base[:, 2] * 0.003)
        dyn = (base, nrm, phase, torch.empty_like(base))

    probes = None
    if args.config == 5:
        import vct_b200.glmath as gm
        from vct_b200 import scenes as _scenes
        cams = _scenes.probe_cameras(64)
        probes = []
        for k in parallel.views_for_rank(len(cams), rank, world):
            pos, yaw, pitch = cams[k]
            view = gm.view_matrix(pos, yaw, pitch)
            probes.append((gm.colmajor((view @ gm.scale(0.05)).astype(np.float32)), tuple(float(x) for x in pos)))
        probe_hosts = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory() for _ in range(2)]

    def bake(to_host):
        """Config 5: one 3-bounce voxelisation, then this rank's probe views rendered from it."""
        ctx.draw_voxels()
        for n, (mv, pos) in enumerate(probes):
            ctx.set_mat4("ModelViewMatrix", mv); ctx.set_3f("CameraPosition", pos)
            ctx.render(probe_hosts[n & 1] if to_host else None)

    def prepare(i):
        """Per-step input: the camera (configs 1, 2, 3) or the re-generated mesh and its shadow map (config 4)."""
        cam_rank = rank if args.mode == "views" else 0
        if args.config == 5:
            return 76 * len(probes)
        if args.config != 4:
            return set_camera(ctx, sc, i, cam_rank)
        base, nrm, phase, out = dyn
        torch.add(base, nrm * (12.0 * torch.sin(phase + 0.21 * i)).unsqueeze(1), out=out)
        ctx.update_positions(device_ptr=out.data_ptr(), n_verts=out.shape[0])
        ctx.draw_depth()                            # the light-space depth map follows the mesh
        return 4                                    # the time parameter; the mesh itself is generated on the device

    def step(i, host_out=None):
        prepare(i)
        if probes is not None:
            bake(host_out is not None)
            return
        if pipelined_shard:
            shared.frame(host_out if rank == 0 else None)     # asynchronous; rows of every rank land in rank 0's frame
            return
        if args.mode == "trishard":
            ctx.voxelize_range(tri_rng[0], tri_rng[1], clear_first=True)
            parallel.allreduce_accumulator(acc)
            ctx.resolve_and_mip()
            ctx.render(None if gather_buf is not None else host_out)
        elif sharded:
            shared.frame_voxels(tri_rng[0], tri_rng[1])       # serial form of the exchange
            ctx.render(None if gather_buf is not None else host_out)
        else:
            ctx.frame(None if gather_buf is not None else host_out)
        if gather_buf is not None:                  # baseline forms: row bands gathered by one NCCL all-gather
            my_band[:own1 - own0].copy_(frame_t[own0:own1])
            dist.all_gather_into_tensor(gather_buf, my_band)
            if host_out is not None:
                host_out.view(-1).copy_(gather_buf[:H * W * 4], non_blocking=False)

    def drain():
        if pipelined_shard:
            shared.wait()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if args.flush else None   # > 126 MB L2

    # ---- correctness gate of the sharded path, before anything is timed: every rank's sharded pyramid and rank 0's
    # assembled frame must equal what one GPU computes alone (this is where the multimem / peer-store kernels and the
    # device barrier are proven on the box that produces the numbers)
    shard_check = None
    if pipelined_shard:
        shard_check = verify_sharded(env, ctx, shared, sc, prepare)

    # nvidia-smi sampling starts before the warm-up and runs until the end-to-end loop has finished: the timed region of
    # a 20-step run lasts ~20 ms, less than one sampling period of the tool
    sampler = ClockSampler(local); sampler.start()
    for i in range(max(args.warmup, 3)):
        step(i)
    drain()
    env.barrier()
    # (1) timed region: per-pass event recording off (it costs ~30 us/frame).  K steps between one pair of CUDA
    # events on the launching stream, barrier + synchronize on both sides.  Consecutive frames pipeline inside the
    # library (the next frame's voxel/visibility stages run beside cone_trace); every frame does all of its work.
    ctx.set_i("Profile", 0)
    ctx.set_i("PipelineFrames", 0 if args.flush else 1)
    launches0 = ctx.kernel_launches()
    env.barrier()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            step(args.warmup + i)
        e1.record(stream)
        drain()
        env.barrier()
        total_ms = e0.elapsed_time(e1)
    else:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for i in range(args.steps):
            flush.fill_(i & 0xFF)                   # untimed: evicts the previous frame's lines from L2
            ev[i][0].record(stream)
            step(args.warmup + i)
            ev[i][1].record(stream)
        drain()
        env.barrier()
        total_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = ctx.kernel_launches() - launches0
    dumped = None
    if args.dump_outputs and rank == 0:
        # row-band modes: each rank's own frame holds only its band; the assembled frame is the all-gather's result
        frame = gather_buf[:H * W * 4].view(H, W, 4).cpu().numpy() if gather_buf is not None else ctx.read_frame()
        dumped = dump_outputs(frame, args.dump_outputs)
    total_ms = env.max_over_ranks([total_ms])[0]
    frames = args.steps * (world if args.mode == "views" else 64 if args.mode == "probes" else 1)
    value = frames / (total_ms * 1e-3)

    # (2) per-pass breakdown and the dominant kernel's average duration: same steps again with pass events on,
    # one frame at a time (no overlap between frames: these are the serial per-pass costs)
    ctx.set_i("Profile", 1)
    if not sharded:
        # one stream: with the visibility pass on its own stream beside the voxel stages (the default), the event
        # pairs of concurrent passes include each other's kernels (round 1 reported 166 us for a 95 us pass that way)
        ctx.set_i("OverlapVisibility", 0)
    pass_names = ["vox_clear", "vox_cover", "vox_shade", "resolve", "mip", "visibility", "cone"]
    if sharded:
        pass_names[3:3] = ["exchange_push"] + (["exchange_merge"] if args.exchange == "inbox" else [])
    pass_sum = {p: 0.0 for p in pass_names}
    samples_sum = 0
    fragments = 0
    n_prof = min(args.steps, 30)
    for i in range(n_prof):
        if flush is not None:
            flush.fill_(i & 0xFF)
        step(args.warmup + i)
        drain()
        torch.cuda.synchronize()
        for p in pass_names:
            try:
                pass_sum[p] += ctx.pass_time_us(p)
            except Exception:
                pass
        samples_sum += ctx.cone_samples()
        fragments = ctx.fragment_count()
    occupied = ctx.occupied_voxels()
    ctx.set_i("Profile", 0); ctx.set_i("OverlapVisibility", 1)
    env.barrier()
    passes = {p: pass_sum[p] / n_prof for p in pass_names}
    passes_max = None
    if world > 1 and args.mode != "views":         # sharded work: the slowest rank sets the pace of every phase
        passes_max = {p: round(v, 2) for p, v in zip(pass_names, env.max_over_ranks([passes[p] for p in pass_names]))}
        samples_sum = env.torch.tensor([samples_sum], dtype=torch.float64, device=dev)
        dist.all_reduce(samples_sum)
        samples_sum = float(samples_sum.item())

    # ---- end to end through the public API with HOST frame buffers (pinned); every frame's D2H copy is inside
    # the timed region.  Render loops use the pipelined calls (vct_frame_async / vct_frame_wait on one GPU,
    # vct_frame_sharded on N: the copy of frame i overlaps the rendering of frame i+1 -- what glfwSwapBuffers gives
    # the reference's loop).
    hosts = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory() for _ in range(3)]
    async_single = args.mode == "views"
    for i in range(3):
        step(i, hosts[0])
    drain()
    if async_single:                                # warm the asynchronous path too (ring buffers, copy stream)
        for i in range(6):
            ctx.frame_async(hosts[i % 3])
            if i >= 2:
                ctx.frame_wait()
        ctx.frame_wait(); ctx.frame_wait()
    env.barrier()
    t0 = time.perf_counter()
    h2d = 0
    for i in range(args.steps):
        if async_single:
            h2d = prepare(args.warmup + i)
            ctx.frame_async(hosts[i % 3])
            if i >= 2:
                ctx.frame_wait()                    # frame i-2 has arrived in host memory (two frames stay queued)
        else:
            h2d = 76 * len(probes) if probes is not None else 76 if args.config != 4 else 4
            step(args.warmup + i, hosts[i % 3])     # sharded: asynchronous, the library bounds the frames in flight
    if async_single:
        ctx.frame_wait(); ctx.frame_wait()
    drain()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    clocks["window"] = "warm-up + timed region + per-pass loop + end-to-end loop"
    if os.environ.get("VCT_BENCH_DEBUG"):
        print(f"[rank {rank}] device loop {total_ms / args.steps:.4f} ms/step (max over ranks), e2e loop {e2e_s / args.steps * 1e3:.4f} ms/step", file=sys.stderr, flush=True)
    e2e_value = frames / env.max_over_ranks([e2e_s])[0]

    # (3) the dense mip kernel alone (roofline_mip): DenseResolve forces the dense resolve + dense pyramid build
    dense_mip_us = None
    if args.config in (1, 2, 3) and not sharded:
        ctx.set_i("Profile", 1); ctx.set_i("DenseResolve", 1)
        acc_us = 0.0
        for i in range(5):
            ctx.frame(); ctx.sync()
            if i >= 2:
                acc_us += ctx.pass_time_us("mip")
        dense_mip_us = acc_us / 3
        ctx.set_i("DenseResolve", 0); ctx.set_i("Profile", 0)
        ctx.frame(); ctx.sync()

    if rank != 0:
        return None

    peaks, peaks_kind = measured_peaks()
    K = args.steps
    fmt = 1 if args.config == 3 else 0
    fmt_name = "RGBA16F" if fmt else "RGBA8"
    bytes_per_sample = 128 if fmt else 64
    cone_us = passes_max["cone"] if passes_max else passes["cone"]
    samples_per_launch = samples_sum / n_prof          # whole frame (all ranks' bands)
    per_rank_samples = samples_per_launch / (world if (passes_max and world > 1) else 1)
    # two-level (trilinear + mip-linear) tex3DLod rate on a pyramid of the same size and format: the best of a fine and a
    # coarser fractional LOD -- at 512^3 RGBA16F the fine levels are HBM-resident and the fine-LOD walk alone (237 Gs/s)
    # is not an upper bound for a kernel whose LOD mix is mostly coarser (profiles/r02_tex3d_sweep.txt)
    tex_peak_frac_lod = max(ctx.bench_tex3d(V=args.grid, n_samples=1 << 28, pattern=0, lod=l, iters=3, grid_format=fmt) for l in (0.5, 2.5))
    tex_peak_int_lod = ctx.bench_tex3d(V=args.grid, n_samples=1 << 28, pattern=0, lod=0.0, iters=3, grid_format=fmt)
    achieved_gs = per_rank_samples / (cone_us * 1e-6) * 1e-9 if cone_us > 0 else 0.0
    traffic = None
    prof = os.path.join(ROOT, "profiles", "cone_trace_traffic.json")
    if os.path.exists(prof) and args.config == 2:
        traffic = json.load(open(prof)).get("dram_bytes_per_launch")
    texel = 8 if fmt else 4
    mip_bytes = sum((args.grid >> l) ** 3 * texel for l in range(args.grid.bit_length()))     # read L0 once + write L1..: 73.14 MiB @256 RGBA8
    hbm = peaks.get("hbm_gbs")
    serial_us = sum(passes.values())
    out = {
        "metric": metric_name(args), "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
        "ms_per_step": round(total_ms / K, 4), "higher_is_better": True,
        "scaling": "weak" if args.mode == "views" else "strong",     # probes / tiles / shards: total work fixed
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config] if (args.detail == 1.0 and args.nominal_size and not args.tune) else f"config{args.config}: {sc.name} {sc.n_tris} tris, V={args.grid} {fmt_name}, {W}x{H}, cones {args.cones}",
                   "mode": args.mode + ("/" + args.exchange if sharded else "") + ("/serial" if sharded and not pipelined_shard else "") + ("/sharded-shadow-map" if sharded and args.shard_shadow else ""),
                   "l2": ("flushed between steps by an untimed 256 MiB write; frames not pipelined" if args.flush else "no flush: per-frame working set ~220 MB (64 MiB level 0 + mips, shadow texels, accumulator lines, queues, vertex cache, visibility) in two alternating frame slots exceeds the 126 MB L2"),
                   "timing": "one CUDA-event pair around the K steps on the launching stream, barrier+synchronize both sides; max over ranks",
                   "step": ("one bake = clear+voxelize+resolve+mip+reinject+mip once, then visibility+cone-trace of 64 probe views (round-robin over ranks); value counts views"
                            if args.mode == "probes" else "clear+voxelize+resolve+mip+visibility+cone-trace (shadow map static, drawn once)" if args.config != 4 else
                            "mesh regeneration + shadow map + clear+voxelize+resolve+mip+visibility+cone-trace")},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": W * H * 4 * (len(probes) if probes is not None else 1),
                "note": ("vct_frame_async(host_rgba)+vct_frame_wait, three pinned host frame buffers (two frames queued), every frame copied to the host inside the timed region; per-step input = view matrix + camera position (kernel parameters)"
                         if async_single else "vct_frame_sharded(host_rgba): every rank writes its rows into rank 0's frame ring over NVLink, rank 0 copies every assembled frame to pinned host memory inside the timed region (up to three frames in flight)"
                         if pipelined_shard else "each step returns after its frame(s) reached pinned host memory (synchronous copy inside the timed region)")},
        "gpu_launches": int(launches),
        # `value` is PIPELINED throughput (three streams, two frame slots: the voxel and visibility stages of frame i+1
        # run beside cone_trace of frame i).  The serial costs, one frame at a time with per-pass events:
        "passes_us": {p: round(v, 2) for p, v in passes.items()},
        "passes_us_max_over_ranks": passes_max,
        "shadow_map_us": round(depth_us, 2),
        "serial": {"sum_of_passes_us": round(serial_us, 1), "frames_s": round(1e6 / serial_us, 1) if serial_us > 0 else None,
                   "frames_s_survey_8d_formula": round(1e6 / (serial_us - passes["visibility"]), 1) if serial_us > 0 else None,
                   "frames_s_including_shadow_map": round(1e6 / (serial_us + depth_us), 1) if serial_us > 0 else None,
                   "note": "SURVEY 8(d): frames/s = 1 / (clear + voxelize + resolve + mip + cone), visibility and shadow map reported both ways"},
        "cone_samples_per_frame": int(samples_per_launch),
        "fragments_per_frame": int(fragments), "occupied_voxels": int(occupied),
        "gcone_samples_per_s": round(achieved_gs * (world if (passes_max and world > 1) else 1), 2),
        # dominant kernel.  It is bound by the texture pipe (tex3DLod wavefronts), not by HBM (28 MB of DRAM traffic per
        # launch at config 2: the pyramid is L1/L2 resident) and not by tensor cores (no dense contraction in this path),
        # so "bound" says "texture"; achieved/peak are ALGORITHMIC texel bytes (2 levels x 8 texels x texel size per
        # sample, SURVEY.md 8d) per second, the peak being the tex3DLod rate measured in this run on a pyramid of the SAME
        # size and format x the same bytes.
        "roofline": {"kernel": "cone_trace", "bound": "texture", "achieved": round(achieved_gs * bytes_per_sample, 1),
                     "peak": round(tex_peak_frac_lod * bytes_per_sample, 1), "unit": "GB/s",
                     "frac": round(achieved_gs / tex_peak_frac_lod, 4) if tex_peak_frac_lod else None,
                     "traffic": traffic,
                     "achieved_gsamples_per_s": round(achieved_gs, 2), "peak_gsamples_per_s": round(tex_peak_frac_lod, 2),
                     "peak_single_level_gsamples_per_s": round(tex_peak_int_lod, 2),
                     "peak_source": f"vct_bench_tex3d_format measured in this run: trilinear + mip-linear tex3DLod, {fmt_name} {args.grid}^3 pyramid, coherent walks, best of LOD 0.5 / 2.5",
                     "algorithmic_bytes_per_sample": bytes_per_sample, "samples_per_launch": int(per_rank_samples),
                     "kernel_us": round(cone_us, 2)},
    }
    mip_us = passes["mip"]
    out["roofline_mip"] = {
        "kernel": "mip_fused3+mip_tail" if not fmt else "mip_level_f16", "bound": "hbm", "peak": hbm, "unit": "GB/s",
        "peak_source": f"MEASURED_PEAKS.json ({peaks_kind})", "algorithmic_bytes": mip_bytes,
        # the HBM figure: the DENSE build reads level 0 once and writes every other level
        "dense_us": round(dense_mip_us, 2) if dense_mip_us else None,
        "achieved": round(mip_bytes / (dense_mip_us * 1e-6) * 1e-9, 1) if dense_mip_us else None,
        "frac": round(mip_bytes / (dense_mip_us * 1e-6) * 1e-9 / hbm, 4) if dense_mip_us else None,
        # the default build is SPARSE (only bricks that changed): not a bandwidth number, a work-avoidance one
        "sparse_us": round(mip_us, 2),
        "sparse_note": "default path: fine levels rebuilt only above changed 32x8x8 bricks; launch-latency bound, reported as time saved against the dense build, not as a fraction of HBM",
    }
    if args.config != 5 and not sharded:
        out["roofline_voxelize"] = voxelize_roofline(ctx, sc, args, passes, fragments, hbm)
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args, sc, u, budget_s=15.0)
    if shard_check is not None:
        out["shard_check"] = shard_check
    if dumped is not None:
        out["dumped_outputs"] = dumped
    return out


DUMP_BYTES = 64_000_000
DUMP_SAMPLE_PIXELS = 1 << 21


def dump_outputs(frame, out_dir):
    """The frame the last timed step rendered (what vct_frame hands its caller), as float32.  Frames above DUMP_BYTES
    (config 3: 3840x2160) are sampled: the same pixels, in raster order, on every run of the same frame size."""
    frame = frame.astype(np.float32)
    H, W, _ = frame.shape
    name = "frame"
    if frame.nbytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(H * W, size=DUMP_SAMPLE_PIXELS, replace=False))
        frame, name = frame.reshape(H * W, 4)[idx], "frame_sample"
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), frame)
    return {name: list(frame.shape)}


def voxelize_roofline(ctx, sc, args, passes, fragments, hbm):
    """SURVEY 8(d): the voxel pass is not HBM-bound; report fragments/s, shadow taps/s and atomics/s against a
    micro-benchmarked atomics peak, and the two triangle set-up kernels against HBM (their algorithmic traffic)."""
    nt = sc.n_tris
    shade_s, cover_s, vis_s = passes["vox_shade"] * 1e-6, passes["vox_cover"] * 1e-6, passes["visibility"] * 1e-6
    atom_peak = ctx.bench_atomics(max(int(fragments), 1), iters=5)      # G atomics/s, same voxel population + multiplicity
    taps = (2 * 2 + 1) ** 2 + 1
    cover_bytes = nt * (12 + 3 * (16 + 16 + 8) + 128) + fragments * 8           # idx + world/dc/uv per vertex + VoxRecord + fragment records
    vis_bytes = nt * (12 + 3 * 16) + args.width * args.height * 8 * 2           # idx + clip per vertex, visibility buffer fill + one update
    r = {
        "vox_shade": {"fragments_per_s": round(fragments / shade_s * 1e-9, 3) if shade_s else None, "unit": "G/s",
                      "texture_taps_per_s": round(fragments * taps / shade_s * 1e-9, 2) if shade_s else None,
                      "atomics_per_s": round(2 * fragments / shade_s * 1e-9, 3) if shade_s else None,
                      "atomics_peak": round(atom_peak, 3),
                      "atomics_frac": round(2 * fragments / shade_s * 1e-9 / atom_peak, 4) if shade_s and atom_peak else None,
                      "peak_source": "vct_bench_atomics in this run: two u64 atomicAdd per fragment on the touched-voxel population at the measured fragments-per-voxel multiplicity, nothing else in the kernel",
                      "note": "issue + latency bound chain (queue -> record -> 9 tex2Dgather -> 55 lerps -> 2 atomics): the atomics alone would take atomics_frac of the pass"},
        "raster_cover": {"bound": "hbm", "algorithmic_bytes": int(cover_bytes), "achieved": round(cover_bytes / cover_s * 1e-9, 1) if cover_s else None,
                         "peak": hbm, "unit": "GB/s", "frac": round(cover_bytes / cover_s * 1e-9 / hbm, 4) if cover_s else None,
                         "triangles_per_s": round(nt / cover_s * 1e-9, 3) if cover_s else None},
        "raster_visibility": {"bound": "hbm", "algorithmic_bytes": int(vis_bytes), "achieved": round(vis_bytes / vis_s * 1e-9, 1) if vis_s else None,
                              "peak": hbm, "unit": "GB/s", "frac": round(vis_bytes / vis_s * 1e-9 / hbm, 4) if vis_s else None,
                              "triangles_per_s": round(nt / vis_s * 1e-9, 3) if vis_s else None},
    }
    return r


def grid_checksums(ctx, levels):
    return [zlib.crc32(np.ascontiguousarray(ctx.grid(l)).view(np.uint8)) for l in range(levels)]


def verify_sharded(env, ctx, shared, sc, prepare):
    """Every rank: one frame alone (vct_frame) -> checksums of every pyramid level + the frame; then the same frame
    sharded over all ranks -> every rank's pyramid must match bit for bit and rank 0 must receive the same frame."""
    torch = env.torch
    levels = ctx.get_i("MipLevels")
    H, W = ctx.get_i("screen_height"), ctx.get_i("screen_width")
    rb, re_, ril, rph = ctx.get_i("RowBegin"), ctx.get_i("RowEnd"), ctx.get_i("RowInterleave"), ctx.get_i("RowPhase")
    interleave = env.world
    ctx.set_i("RowBegin", 0); ctx.set_i("RowEnd", 0); ctx.set_i("RowInterleave", 0); ctx.set_i("RowPhase", 0)
    ctx.set_i("TriangleInterleave", 1); ctx.set_i("TrianglePhase", 0)
    prepare(0)
    ctx.frame(); ctx.sync()
    ref_crc = grid_checksums(ctx, levels)
    ref_frame = ctx.read_frame()
    ctx.set_i("RowBegin", rb); ctx.set_i("RowEnd", re_); ctx.set_i("RowInterleave", ril); ctx.set_i("RowPhase", rph)
    ctx.set_i("TriangleInterleave", interleave); ctx.set_i("TrianglePhase", env.rank)
    host = torch.zeros((H, W, 4), dtype=torch.uint8).pin_memory()
    ok = True
    for _ in range(3):                 # both frame slots and both inbox parities
        prepare(0)
        shared.frame(host if env.rank == 0 else None)
    shared.wait()
    ok &= grid_checksums(ctx, levels) == ref_crc
    frame_ok = True
    if env.rank == 0:
        frame_ok = bool(np.array_equal(host.numpy(), ref_frame))
    all_ok = env.all_true(ok and frame_ok)
    res = {"ranks": env.world, "multicast": bool(shared.info["multicast"]), "pyramid_levels_equal_single_gpu_on_every_rank": env.all_true(ok),
           "assembled_frame_equals_single_gpu": env.all_true(frame_ok)}
    if not all_ok:
        raise RuntimeError(f"sharded frame differs from the single-GPU frame: {res}")
    return res


def strong_config3(env, steps, warmup):
    """BASELINE config 3 as ONE sharded frame stream over all ranks (the strong-scaling number north_star asks for),
    with its own one-GPU anchor measured in the same run on the same context."""
    torch = env.torch
    import vct_b200
    from vct_b200 import parallel
    a3 = parse(["--config", "3", "--gpus", str(env.world), "--mode", "shard", "--steps", str(steps), "--warmup", str(warmup)])
    sc, u = make_scene_and_uniforms(a3)
    ctx = vct_b200.Context(env.local)
    ctx.set_stream(env.stream.cuda_stream)
    ctx.set_uniforms(u); ctx.load_scene(sc)
    ctx.draw_depth(); ctx.sync()
    ctx.set_i("Profile", 0); ctx.set_i("PipelineFrames", 1)
    H, W = a3.height, a3.width

    def prepare(i):
        return set_camera(ctx, sc, i, 0)

    def timed(fn, drain):
        for i in range(warmup):
            fn(i)
        drain(); env.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(env.stream)
        for i in range(steps):
            fn(warmup + i)
        e1.record(env.stream)
        drain(); env.barrier()
        return env.max_over_ranks([e0.elapsed_time(e1)])[0]

    # one-GPU anchor: every rank renders the whole frame stream alone (pipelined vct_frame); rank 0's pace is the anchor
    def alone(i):
        prepare(i); ctx.frame(None)
    n1_ms = timed(alone, lambda: ctx.sync())
    hosts = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory() for _ in range(3)]
    for i in range(6):
        prepare(i); ctx.frame_async(hosts[i % 3])
        if i >= 2:
            ctx.frame_wait()
    ctx.frame_wait(); ctx.frame_wait(); env.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        prepare(warmup + i); ctx.frame_async(hosts[i % 3])
        if i >= 2:
            ctx.frame_wait()
    ctx.frame_wait(); ctx.frame_wait(); torch.cuda.synchronize()
    n1_e2e_s = env.max_over_ranks([time.perf_counter() - t0])[0]

    shared = parallel.SharedAccumulator(ctx, rank=env.rank, world=env.world, session=session_name("strong3"))
    check = verify_sharded(env, ctx, shared, sc, prepare)

    def sharded(i, host=None):
        prepare(i); shared.frame(host if env.rank == 0 else None)
    ms = timed(sharded, shared.wait)
    # per-pass costs, one frame at a time, max over ranks
    ctx.set_i("Profile", 1)
    names = ["vox_clear", "vox_cover", "vox_shade", "exchange_push", "exchange_merge", "resolve", "mip", "visibility", "cone"]
    acc = {p: 0.0 for p in names}
    n_prof = min(steps, 10)
    for i in range(n_prof):
        sharded(warmup + i); shared.wait(); torch.cuda.synchronize()
        for p in names:
            try:
                acc[p] += ctx.pass_time_us(p)
            except Exception:
                pass
    ctx.set_i("Profile", 0)
    passes_max = {p: round(v, 1) for p, v in zip(names, env.max_over_ranks([acc[p] / n_prof for p in names]))}
    # end to end: rank 0 receives every assembled frame in pinned host memory
    for i in range(3):
        sharded(i, hosts[i % 3])
    shared.wait(); env.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        sharded(warmup + i, hosts[i % 3])
    shared.wait(); torch.cuda.synchronize()
    e2e_s = env.max_over_ranks([time.perf_counter() - t0])[0]
    shared.close(); ctx.close()
    fps, n1_fps = steps / (ms * 1e-3), steps / (n1_ms * 1e-3)
    return {"workload": WORKLOADS[3], "mode": "shard/inbox pipelined (vct_frame_sharded)", "n_gpus": env.world, "steps": steps, "warmup": warmup,
            "frames_s": round(fps, 2), "ms_per_step": round(ms / steps, 4),
            "n1_frames_s": round(n1_fps, 2), "n1_ms_per_step": round(n1_ms / steps, 4),
            "speedup_vs_n1": round(fps / n1_fps, 3), "efficiency_vs_n1": round(fps / n1_fps / env.world, 4),
            "e2e_frames_s": round(steps / e2e_s, 2), "n1_e2e_frames_s": round(steps / n1_e2e_s, 2),
            "d2h_bytes_per_step": W * H * 4,
            "passes_us_max_over_ranks": passes_max, "shard_check": check,
            "note": "one frame stream; triangles dealt in blocks of 128, touched voxels exchanged as 16-byte records with multimem.st, "
                    "rows dealt in strips of 8 and written by cone_trace into rank 0's frame ring over NVLink, two device-side barriers per frame; "
                    "no NCCL call in the timed region.  n1_* = the same frames rendered by one GPU alone (pipelined vct_frame) in this run."}


# ------------------------------------------------------------------------------------------------ CPU legs
def host_threads():
    """Gives the OpenMP oracle every core of the affinity mask (torchrun exports OMP_NUM_THREADS=1) and returns the
    number of threads it will really use."""
    from oracle import oracle_py
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return oracle_py.set_num_threads(n)


def cpu_baseline(args, sc, u, budget_s):
    """The oracle ("port": the reference's GLSL cannot run here, SURVEY.md 8c) timed on the host cores, on a
    bounded sample of the same workload: as many full config frames as fit in ~budget_s (at least one)."""
    from oracle.oracle_py import Oracle
    threads = host_threads()
    o = Oracle(); o.set_uniforms(u); o.load_scene(sc)
    t0 = time.perf_counter(); o.draw_depth(); t_depth = time.perf_counter() - t0
    t0 = time.perf_counter(); n = 0; tv = tr = 0.0
    while True:
        a = time.perf_counter(); o.draw_voxels(); b = time.perf_counter(); o.render(); c = time.perf_counter()
        tv += b - a; tr += c - b; n += 1
        if time.perf_counter() - t0 > budget_s or n >= (50 if args.config != 1 else 200):
            break
        if args.config == 1 and n >= 10 and time.perf_counter() - t0 > 3.0:
            break
    dt = time.perf_counter() - t0
    o.close()
    return {"value": round(n / dt, 4), "unit": UNIT, "cores": threads, "kind": "port",
            "passes_ms": {"shadow_map": round(t_depth * 1e3, 3), "voxelize+resolve+mip": round(tv / n * 1e3, 3),
                          "visibility+cone_trace": round(tr / n * 1e3, 3)},
            "sample": f"{n} full frame(s) of the same workload (voxelize+mip+cone-trace) in {dt:.1f} s, OpenMP, {threads} threads"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle.oracle_py import Oracle
    threads = host_threads()
    sc, u = make_scene_and_uniforms(args)
    o = Oracle(); o.set_uniforms(u); o.load_scene(sc)
    o.draw_depth()
    H = args.height
    # size each step so that the whole run fits in ~150 s: full voxelisation + a band of rows, scaled
    t0 = time.perf_counter(); o.draw_voxels(); t_vox = time.perf_counter() - t0
    t0 = time.perf_counter(); o.render_rows(H // 2 - 8, H // 2 + 8); t_rows16 = time.perf_counter() - t0
    n_steps = args.steps + args.warmup
    per_step = max(150.0 / max(n_steps, 1), 0.05)
    rows = int(np.clip((per_step - t_vox) / max(t_rows16 / 16.0, 1e-6), 8, H)) // 8 * 8
    rows = max(8, min(rows, H))
    y0 = (H - rows) // 2
    for i in range(args.warmup):
        o.draw_voxels(); o.render_rows(y0, y0 + rows)
    tv = tr = 0.0
    for i in range(args.steps):
        t0 = time.perf_counter(); o.draw_voxels(); t1 = time.perf_counter(); o.render_rows(y0, y0 + rows); t2 = time.perf_counter()
        tv += t1 - t0; tr += t2 - t1
    K = max(args.steps, 1)
    frame_s = tv / K + (tr / K) * (H / rows)        # time of a full frame extrapolated from the row band
    value = 1.0 / frame_s
    sample = (f"each step = full voxelize+mip ({tv / K * 1e3:.0f} ms) + cone trace of {rows} of {H} rows "
              f"({tr / K * 1e3:.0f} ms), extrapolated linearly to the full frame; CPU oracle (port), OpenMP, {threads} threads")
    out = {"impl": "reference", "metric": metric_name(args), "value": round(value, 4), "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(frame_s * 1e3, 2), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
           "config": {"workload": WORKLOADS[args.config], "mode": "cpu"},
           "cpu_baseline": {"value": round(value, 4), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
           "e2e": {"value": round(value, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
