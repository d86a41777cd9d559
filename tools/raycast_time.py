#!/usr/bin/env python
"""Times ray casts (vct_cast_rays, device form) at the size of configs 2 and 3 with CUDA events.

    python tools/raycast_time.py [--launches 50] [--out FILE.json]

The atrium is voxelised on the device (config 2: 256^3 RGBA8; config 3: 512^3 RGBA16F).  Two seeded segment sets of 1 M
and 16 M segments each are cast at levels 0 and 2: "random", both endpoints uniform over the grid's box, and "coherent",
the per-pixel near-to-far segments of the scene's camera on a 1024x1024 and a 4096x4096 screen (neighbouring segments
visit neighbouring texels, as picking or a screen of occlusion rays would).  Segments and all five outputs are torch CUDA
tensors.  After warm-up calls, one pair of events brackets --launches back-to-back casts on the context's stream
(Profile off).  Reported per case: microseconds per call, rays/s, texels visited per call (vct_debug_counter 3) and
texels/s.  The config-2 pyramid (73 MiB) stays in the 126 MB L2 across calls; the config-3 one (1.17 GiB) does not.
The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

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


def random_segments(n, G, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand((n, 6), generator=g, device="cuda", dtype=torch.float32) - 0.5) * float(G)


def pixel_segments(u, W, H):
    """near and far point of every pixel of the scene camera on a W x H screen (the view's rays)"""
    import torch
    m = lambda k: np.asarray(u[k], np.float64).reshape(4, 4).T          # column-major uniforms
    proj = m("ProjectionMatrix").copy()
    proj[0, 0] = proj[1, 1] * H / W                                       # the camera's fov at this aspect
    inv = torch.tensor(m("ModelMatrix") @ np.linalg.inv(proj @ m("ModelViewMatrix")), dtype=torch.float32, device="cuda")
    x = (torch.arange(W, device="cuda", dtype=torch.float32) * 2 + 1) / W - 1
    y = (torch.arange(H, device="cuda", dtype=torch.float32) * 2 + 1) / H - 1
    Y, X = torch.meshgrid(y, x, indexing="ij")
    ends = []
    for z in (-1.0, 1.0):
        p = torch.stack([X, Y, torch.full_like(X, z), torch.ones_like(X)], -1).reshape(-1, 4) @ inv.T
        ends.append(p[:, :3] / p[:, 3:])
    return torch.cat(ends, 1).contiguous()


def time_cast(c, level, seg, launches, warmup):
    import torch
    n = seg.shape[0]
    outs = [torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda"),
            torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty((n, 4), dtype=torch.uint8, device="cuda"),
            torch.empty(n, dtype=torch.int32, device="cuda")]
    call = lambda: c.cast_rays(level, n=n, device_segments=seg.data_ptr(), device_voxel=outs[0].data_ptr(),
                               device_t=outs[1].data_ptr(), device_face=outs[2].data_ptr(), device_rgba=outs[3].data_ptr(),
                               device_steps=outs[4].data_ptr())
    stream = torch.cuda.current_stream()
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    texels = c.debug_counter(3)
    hits = int((outs[0] != -1).sum().item())
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(launches):
        call()
    t1.record(stream)
    t1.synchronize()
    us = t0.elapsed_time(t1) * 1000.0 / launches
    return {"level": level, "segments": n, "hits": hits, "us_per_call": round(us, 2),
            "grays_per_s": round(n / (us * 1e-6) * 1e-9, 3), "texels_visited": texels,
            "gtexels_per_s": round(texels / (us * 1e-6) * 1e-9, 2)}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the result as JSON here")
    a = ap.parse_args(argv)
    if a.launches < 20:
        ap.error("--launches must be at least 20")
    import torch
    res = gpu_info()
    sc = scenes.atrium()
    c = vct_b200.Context(0)
    c.load_scene(sc)
    c.set_stream(torch.cuda.current_stream().cuda_stream)
    for name, kw in (("config2", dict(V=256, width=1920, height=1080)),
                     ("config3", dict(V=512, width=3840, height=2160, cones="9+1", grid_format=1))):
        u = uniforms.scene_uniforms(sc, shadow_map_size=4096, coverage="conservative", **kw)
        c.set_uniforms(u)
        c.draw_depth(); c.draw_voxels(); c.sync()
        c.set_i("Profile", 0)
        rows = []
        for side, n in ((1024, 1 << 20), (4096, 1 << 24)):
            sets = (("random", random_segments(n, u["VoxelGridWorldSize"], seed=n + kw["V"])),
                    ("coherent", pixel_segments(u, side, side)))
            for kind, seg in sets:
                for level in (0, 2):
                    r = dict(set=kind, **time_cast(c, level, seg, a.launches, a.warmup))
                    rows.append(r)
                    print(f"{name} {kind} {n} segments level {level}: {r['us_per_call']:.1f} us per call, "
                          f"{r['grays_per_s']:.2f} Grays/s, {r['texels_visited']} texels visited, "
                          f"{r['gtexels_per_s']:.1f} Gtexels/s, {r['hits']} hits")
            del sets
        c.set_i("Profile", 1)
        res[name] = {"V": kw["V"], "launches": a.launches, "casts": rows}
    c.use_own_stream()
    print(f"GPU: {res['gpu']}, power limit / max SM clock: {res['power_limit_and_max_sm_clock']}")
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    c.close()


if __name__ == "__main__":
    main()
