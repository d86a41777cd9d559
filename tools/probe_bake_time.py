#!/usr/bin/env python
"""Times the irradiance-probe bake (vct_bake_probes, device form) with CUDA events.

    python tools/probe_bake_time.py [--launches 200] [--out FILE.json]

The atrium is voxelised on the device at config 2 (256^3 RGBA8, default 6+1 cones) and config 3 (512^3 RGBA16F, 9+1
cones); the probes are the cell centres of a k^3 lattice over [-G/2, G/2]^3 (k = 16, 32, 64 at config 2; 32 at config 3),
held in torch CUDA tensors.  After warm-up bakes, one pair of events brackets --launches back-to-back bakes on the
context's stream (Profile off).  Reported per lattice: microseconds per bake, probe faces per second, textureLod calls
per bake (vct_debug_counter 2) and Gsamples/s, next to the coherent-walk tex3DLod rate of a pyramid of the same size and
format (vct_bench_tex3d_format, pattern 0) measured in the same run.  The GPU name and power limit are read in the same
run."""
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


def lattice(k, G):
    import torch
    cells = (torch.arange(k, dtype=torch.float32) + 0.5) * (G / k) - G / 2
    z, y, x = torch.meshgrid(cells, cells, cells, indexing="ij")
    return torch.stack([x, y, z], -1).reshape(-1, 3).contiguous().cuda()


def time_lattices(c, G, ks, launches, warmup):
    import torch
    stream = torch.cuda.current_stream()
    c.set_stream(stream.cuda_stream)
    c.set_i("Profile", 0)
    rows = []
    for k in ks:
        xyz = lattice(k, G)
        n = xyz.shape[0]
        out = torch.empty((n, 6, 4), dtype=torch.float32, device="cuda")
        bake = lambda: c.bake_probes(n=n, device_xyz=xyz.data_ptr(), device_out=out.data_ptr())
        for _ in range(warmup):
            bake()
        torch.cuda.synchronize()
        samples = c.debug_counter(2)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for _ in range(launches):
            bake()
        t1.record(stream)
        t1.synchronize()
        us = t0.elapsed_time(t1) * 1000.0 / launches
        rows.append({"k": k, "probes": n, "us_per_bake": round(us, 2), "faces_per_s": round(6 * n / (us * 1e-6), 0),
                     "samples": samples, "gsamples_per_s": round(samples / (us * 1e-6) * 1e-9, 2)})
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
    for name, kw, ks in (("config2", dict(V=256, width=1920, height=1080), (16, 32, 64)),
                         ("config3", dict(V=512, width=3840, height=2160, cones="9+1", grid_format=1), (32,))):
        u = uniforms.scene_uniforms(sc, shadow_map_size=4096, coverage="conservative", **kw)
        c.set_uniforms(u)
        c.draw_depth(); c.draw_voxels(); c.sync()
        rows = time_lattices(c, u["VoxelGridWorldSize"], ks, a.launches, a.warmup)
        fmt = kw.get("grid_format", 0)
        tex = c.bench_tex3d(V=kw["V"], pattern=0, grid_format=fmt)
        res[name] = {"V": kw["V"], "grid_format": "RGBA16F" if fmt else "RGBA8", "cones": kw.get("cones", "6+1"),
                     "launches": a.launches, "tex3d_coherent_gsamples_per_s": round(tex, 2), "lattices": rows}
        for r in rows:
            print(f"{name} k={r['k']} ({r['probes']} probes): {r['us_per_bake']:.1f} us per bake, "
                  f"{r['faces_per_s'] / 1e9:.3f} G faces/s, {r['samples']} samples, {r['gsamples_per_s']:.1f} Gsamples/s "
                  f"(coherent tex3DLod {tex:.1f} Gsamples/s)")
    print(f"GPU: {res['gpu']}, power limit / max SM clock: {res['power_limit_and_max_sm_clock']}")
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    c.close()


if __name__ == "__main__":
    main()
