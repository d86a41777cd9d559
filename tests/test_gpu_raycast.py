"""Ray casts on the device (vct_cast_rays) against the CPU reference (tests/raycast_ref.cpp on the oracle's parameters
and mip pyramid): bit-exact texel index, entry parameter, face, colour and step count on uploaded grids, on a grid
voxelised end to end and at the size of configs 2 and 3; against the device's own voxel view; and how a cast fits the
context's frame state.  Run with -m gpu on a B200."""
import os
import subprocess

import numpy as np
import pytest

from test_gpu_voxel_view import UPLOAD_CAMERAS, cornell_ctx, device_view
from test_raycast import pixel_segments, segment_mix, shaded_pixels
from test_voxel_view import MISS, cam_uniforms, sparse_grid
from vct_b200 import capi, scenes, uniforms
from raycast_ref import cast_rays as ref_cast

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
NAMES = ("voxel", "t", "face", "rgba", "steps")


def assert_same_casts(got, want, what):
    for name, g, w in zip(NAMES, got, want):
        bad = (g.view(np.uint8).reshape(len(g), -1) != w.view(np.uint8).reshape(len(w), -1)).any(1)
        assert not bad.any(), f"{what}: {name} differs on {int(bad.sum())} of {bad.size} segments"


def assert_matches_reference(c, oracle, level, segs, what):
    got = c.cast_rays(level, segs)
    assert_same_casts(got, ref_cast(oracle, level, segs), f"{what} level {level}")
    assert c.debug_counter(3) == int(got[4].astype(np.int64).sum())
    hits = int((got[0] != MISS).sum())
    print(f"[ray casts] {what} level {level}: {hits} of {len(segs)} segments hit, {c.debug_counter(3)} texels visited")
    return hits


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("V", [16, 64, 128])
def test_uploaded_grids_match_the_reference(gpu_ctx, oracle, V, fmt):
    c = gpu_ctx
    G = 150.0
    g = sparse_grid(V, seed=V + fmt, fmt=fmt, density=0.02)
    u = cam_uniforms(V, size=(64, 48), G=G, fmt=fmt, **UPLOAD_CAMERAS["outside"])
    c.set_uniforms(u); c.upload_grid_level0(g)
    oracle.set_uniforms(u); oracle.set_grid_level0(g)
    segs = segment_mix(V, G, seed=100 * V + fmt, n=5000)
    hits = sum(assert_matches_reference(c, oracle, level, segs, f"V={V} fmt={fmt}") for level in range(V.bit_length()))
    assert hits > 1000


def test_config1_cornell_voxelised_end_to_end(gpu_ctx, oracle):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=256, shadow_map_size=1024, coverage="msaa4")
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels()
    oracle.set_uniforms(u); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels()
    assert np.array_equal(c.grid(0), oracle.grid(0))
    segs = segment_mix(64, 150.0, seed=1)
    for level in range(7):
        assert_matches_reference(c, oracle, level, segs, "config 1")


def test_config2_and_config3_size(gpu_ctx, oracle):
    """1 M segments at configs 2 (256^3) and 3 (512^3 RGBA16F) voxelised on the device; the oracle's pyramid is built from
    the device's own level 0, as in test_gpu_voxel_view.py"""
    sc = scenes.atrium()
    c = gpu_ctx
    for what, kw in (("config 2", dict(V=256, width=1920, height=1080)),
                     ("config 3", dict(V=512, width=3840, height=2160, cones="9+1", grid_format=1))):
        u = uniforms.scene_uniforms(sc, shadow_map_size=4096, coverage="conservative", **kw)
        c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels(); c.sync()
        oracle.set_uniforms(u)
        oracle.set_grid_level0(c.grid(0))
        segs = segment_mix(kw["V"], u["VoxelGridWorldSize"], seed=kw["V"], n=1 << 18)      # 4 x 2^18 = 1 M segments
        assert len(segs) == 1 << 20
        for level in (0, 2):
            assert assert_matches_reference(c, oracle, level, segs, what) > 10000


@pytest.mark.parametrize("level", [0, 1, 3])
def test_pixel_segments_reproduce_the_device_view(gpu_ctx, level):
    c = gpu_ctx
    _, u = cornell_ctx(c); c.draw_voxels()
    vrgba, vvox, vsteps = device_view(c, level)
    voxel, t, face, rgba, steps = c.cast_rays(level, pixel_segments(u))
    assert np.array_equal(voxel, vvox.reshape(-1))
    assert int(steps.astype(np.int64).sum()) == vsteps == c.debug_counter(3)
    hit = voxel != MISS
    assert hit.sum() > 1000
    assert np.array_equal(shaded_pixels(face[hit], rgba[hit]), vrgba.reshape(-1, 4)[hit, :3])


def test_host_and_device_forms_give_identical_bytes(gpu_ctx):
    import torch
    c = gpu_ctx
    cornell_ctx(c); c.draw_voxels()
    segs = segment_mix(64, 150.0, seed=9, n=999)
    n = len(segs)
    want = c.cast_rays(1, segs)
    ds = torch.from_numpy(segs).cuda()
    outs = [torch.full((n,), -1, dtype=torch.int32, device="cuda"), torch.full((n,), -1.0, dtype=torch.float32, device="cuda"),
            torch.full((n,), 77, dtype=torch.uint8, device="cuda"), torch.full((n, 4), 77, dtype=torch.uint8, device="cuda"),
            torch.full((n,), -1, dtype=torch.int32, device="cuda")]
    torch.cuda.synchronize()
    c.cast_rays(1, n=n, device_segments=ds.data_ptr(), device_voxel=outs[0].data_ptr(), device_t=outs[1].data_ptr(),
                device_face=outs[2].data_ptr(), device_rgba=outs[3].data_ptr(), device_steps=outs[4].data_ptr())
    c.sync()
    for name, o, w in zip(NAMES, outs, want):
        assert np.array_equal(o.cpu().numpy().view(np.uint8).reshape(n, -1), w.view(np.uint8).reshape(n, -1)), name
    only = torch.zeros(n, dtype=torch.int32, device="cuda")             # the optional outputs may be NULL
    c.cast_rays(1, n=n, device_segments=ds.data_ptr(), device_voxel=only.data_ptr())
    c.sync()
    assert np.array_equal(only.cpu().numpy().view(np.uint32), want[0])
    voxel = np.zeros(n, np.uint32)                                       # ... in the host form too
    c._ck(c.L.vct_cast_rays(c.h, 1, n, capi._ptr(segs), capi._ptr(voxel), None, None, None, None, 0))
    assert np.array_equal(voxel, want[0])
    assert c.debug_counter(3) == int(want[4].astype(np.int64).sum())


def test_frames_around_a_cast_are_unchanged(gpu_ctx):
    c = gpu_ctx
    cornell_ctx(c)
    c.frame(); c.sync()
    before, samples = c.read_frame(), c.cone_samples()
    segs = segment_mix(64, 150.0, seed=3, n=500)
    got = c.cast_rays(0, segs)
    assert (got[0] != MISS).sum() > 100
    assert c.cone_samples() == samples
    assert np.array_equal(c.read_frame(), before)                       # the cast does not write the frame buffer
    c.frame(); c.sync()
    assert np.array_equal(c.read_frame(), before) and c.cone_samples() == samples
    assert_same_casts(c.cast_rays(0, segs), got, "after another frame")


def test_cast_behind_frames_in_flight(gpu_ctx):
    """a cast enqueued behind three vct_frame_async frames reads the pyramid of the last of them"""
    c = gpu_ctx
    sc, u = cornell_ctx(c)
    xyz = sc.verts[:, :3].astype(np.float32)
    segs = segment_mix(64, 150.0, seed=4, n=500)
    hosts = [np.empty((256, 256, 4), np.uint8) for _ in range(3)]
    shift = lambda k: (xyz + np.float32(150.0 * k) * np.array([1, 0, 0], np.float32)).astype(np.float32)
    c.update_positions(shift(0)); c.draw_depth(); c.frame(); c.sync()
    first = c.cast_rays(0, segs)
    for k in range(3):
        c.update_positions(shift(k + 1)); c.draw_depth()
        c.frame_async(hosts[k])
    behind = c.cast_rays(0, segs)
    for _ in range(3):
        c.frame_wait()
    after = c.cast_rays(0, segs)
    assert_same_casts(behind, after, "cast behind frames in flight")
    assert not np.array_equal(first[0], after[0])                       # the frames in flight did move the geometry


def test_camera_and_row_sharding_uniforms_do_not_change_a_cast(gpu_ctx):
    c = gpu_ctx
    cornell_ctx(c); c.draw_voxels()
    segs = segment_mix(64, 150.0, seed=5, n=500)
    want = c.cast_rays(2, segs)
    c.set_3f("CameraPosition", (30.0, -12.0, 80.0))
    c.set_mat4("ModelViewMatrix", np.arange(16, dtype=np.float32))
    c.set_mat4("ProjectionMatrix", np.eye(4, dtype=np.float32) * 2)
    c.set_i("screen_width", 97); c.set_i("screen_height", 31)
    assert_same_casts(c.cast_rays(2, segs), want, "camera uniforms")
    c.set_i("RowInterleave", 2); c.set_i("RowPhase", 1)
    assert_same_casts(c.cast_rays(2, segs), want, "interleaved rows")
    c.set_i("RowInterleave", 0); c.set_i("RowPhase", 0); c.set_i("RowBegin", 5); c.set_i("RowEnd", 9)
    assert_same_casts(c.cast_rays(2, segs), want, "row band")


def test_errors_and_counters(gpu_ctx):
    c = gpu_ctx
    c.set_uniforms(cam_uniforms(32, size=(40, 30), G=150.0, eye=(0.0, 0.0, 200.0), center=(0.0, 0.0, 0.0)))
    segs = segment_mix(32, 150.0, seed=6, n=100)
    voxel, t, face, rgba, steps = c.cast_rays(0, segs)                   # nothing voxelised yet: an empty grid
    assert (voxel == MISS).all() and np.isinf(t).all() and (face == 0).all() and (rgba == 0).all() and steps.sum() > 0
    assert c.pass_time_us("rays") > 0

    def code(level, n, **kw):
        with pytest.raises(capi.VctError) as e:
            c.cast_rays(level, n=n, **kw)
        return e.value.code
    dev = dict(device_segments=1 << 20, device_voxel=1 << 20)
    assert code(-1, 4, **dev) == -1 and code(6, 4, **dev) == -1
    assert code(0, 4, device_segments=0, device_voxel=1 << 20) == -1
    assert code(0, 4, device_segments=1 << 20, device_voxel=0) == -1
    assert code(0, 1 << 60, **dev) == -1
    assert code(0, 4, device_rgba=(1 << 20) + 2, **dev) == -1
    out = c.cast_rays(0, np.zeros((0, 6), np.float32))                  # n = 0: a no-op
    assert all(len(o) == 0 for o in out)
    c.cast_rays(7, n=0, device_segments=0, device_voxel=0)               # ... before any argument is looked at
    rng = np.random.default_rng(11)
    g = np.zeros((32, 32, 32, 4), np.uint8)
    occ = rng.random((32, 32, 32)) < 0.1
    g[occ] = rng.integers(1, 256, (int(occ.sum()), 4), dtype=np.uint8)
    c.upload_grid_level0(g, build_mips=False)
    with pytest.raises(capi.VctError) as e:
        c.cast_rays(1, segs)
    assert e.value.code == -3
    voxel, _, _, _, steps = c.cast_rays(0, segs)                          # level 0 is current
    assert (voxel != MISS).sum() > 10 and c.debug_counter(3) == int(steps.sum())
    c.build_mips()
    c.cast_rays(1, segs)
    bad = segs.copy()
    bad[:3, [0, 4, 2]] = [np.nan, np.inf, -np.inf]
    voxel, t, face, rgba, steps = c.cast_rays(0, bad)
    assert (voxel[:3] == MISS).all() and (steps[:3] == 0).all() and np.isinf(t[:3]).all()


def test_cpp_facade_casts_equal_the_ctypes_binding(gpu_ctx, tmp_path):
    """facade_demo casts a 16x16 fan through Voxel_Cone_Tracing::CastRays after its frames; the same inputs through ctypes
    give the same bytes"""
    root = os.path.dirname(HERE)
    exe = os.path.join(root, "voxel-cone-tracing_b200", "lib", "facade_demo")
    if not os.path.exists(exe):
        import __graft_entry__
        __graft_entry__.build()
    out = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    rd = lambda name, dt: np.fromfile(os.path.join(str(tmp_path), name), dtype=dt)
    verts, idx, trimat = rd("verts.f32", np.float32).reshape(-1, 14), rd("idx.u32", np.uint32).reshape(-1, 3), rd("trimat.u16", np.uint16)
    tex = [np.full((1, 1, 3), v, np.uint8) for v in ((200, 200, 200), (200, 30, 30), (30, 200, 30))] + \
          [np.full((1, 1), 128, np.uint8), np.full((1, 1, 3), 128, np.uint8)]
    sc = scenes.Scene("facade", verts, idx, trimat, tex, [(0, 3, 4, 20.0), (1, 3, 4, 20.0), (2, 3, 4, 20.0)])
    names = ["ModelViewMatrix", "ProjectionMatrix", "DepthModelViewProjectionMatrix", "ProjX", "ProjY", "ProjZ"]
    raw = rd("uniforms_2.f32", np.float32)
    u = uniforms.reference_uniforms(V=64, width=256, height=256, shadow_map_size=4096, coverage="msaa4")
    for k, name in enumerate(names):
        u[name] = raw[16 * k:16 * k + 16].copy()
    u["CameraPosition"] = raw[96:99].copy()
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels()
    segs = rd("rays_seg.f32", np.float32).reshape(-1, 6)
    cells = (np.arange(16, dtype=np.float32) + np.float32(0.5)) * np.float32(150.0 / 16) - np.float32(75.0)
    y, x = np.meshgrid(cells, cells, indexing="ij")
    b = np.stack([x, y, np.full_like(x, -75.0)], -1).reshape(-1, 3)
    assert np.array_equal(segs, np.concatenate([np.zeros_like(b), b], 1))
    voxel, t, _, _, _ = c.cast_rays(0, segs)
    assert (voxel != MISS).sum() > 100
    assert np.array_equal(voxel, rd("rays_voxel.u32", np.uint32)), "C++ facade and ctypes binding disagree"
    assert np.array_equal(t.view(np.uint32), rd("rays_t.f32", np.float32).view(np.uint32))
