#!/usr/bin/env python
"""Times the voxel view (vct_render_voxels) at the size of configs 2 and 3 with CUDA events.

    python tools/voxel_view_time.py [--launches 200] [--out FILE.json]

The atrium is voxelised on the device (config 2: 256^3 RGBA8, 1920x1080; config 3: 512^3 RGBA16F, 3840x2160) and each
level is viewed from the scene's camera.  After warm-up launches, one pair of events brackets --launches back-to-back
views on the context's stream (device-only calls, Profile off).  Reported per level: microseconds per view, texels visited
per view (vct_debug_counter 1) and visited texels per second.  The config-2 pyramid (73 MiB) stays in the 126 MB L2
across launches; the config-3 one (1.17 GiB) does not.  The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vct_b200  # noqa: E402
from vct_b200 import scenes, uniforms  # noqa: E402


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def time_levels(c, levels, launches, warmup):
    import torch
    stream = torch.cuda.current_stream()
    c.set_stream(stream.cuda_stream)
    c.set_i("Profile", 0)
    rows = []
    for level in levels:
        for _ in range(warmup):
            c.render_voxels(level)
        torch.cuda.synchronize()
        texels = c.debug_counter(1)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for _ in range(launches):
            c.render_voxels(level)
        t1.record(stream)
        t1.synchronize()
        us = t0.elapsed_time(t1) * 1000.0 / launches
        rows.append({"level": level, "us_per_view": round(us, 2), "texels_visited": texels,
                     "gtexels_per_s": round(texels / (us * 1e-6) * 1e-9, 2)})
    c.set_i("Profile", 1)
    c.use_own_stream()
    return rows


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the result as JSON here")
    a = ap.parse_args(argv)
    if a.launches < 100:
        ap.error("--launches must be at least 100")
    res = gpu_info()
    sc = scenes.atrium()
    c = vct_b200.Context(0)
    c.load_scene(sc)
    for name, kw, levels in (("config2", dict(V=256, width=1920, height=1080), (0, 1, 2, 3)),
                             ("config3", dict(V=512, width=3840, height=2160, cones="9+1", grid_format=1), (0, 2))):
        u = uniforms.scene_uniforms(sc, shadow_map_size=4096, coverage="conservative", **kw)
        c.set_uniforms(u)
        c.draw_depth(); c.draw_voxels(); c.sync()
        res[name] = {"V": kw["V"], "size": f"{kw['width']}x{kw['height']}", "pixels": kw["width"] * kw["height"],
                     "launches": a.launches, "levels": time_levels(c, levels, a.launches, a.warmup)}
        for r in res[name]["levels"]:
            print(f"{name} level {r['level']}: {r['us_per_view']:.1f} us per view, {r['texels_visited']} texels visited, "
                  f"{r['gtexels_per_s']:.1f} Gtexels/s")
    print(f"GPU: {res['gpu']}, power limit / max SM clock: {res['power_limit_and_max_sm_clock']}")
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    c.close()


if __name__ == "__main__":
    main()
