"""Voxel view on the device (vct_render_voxels) against the CPU reference (tests/voxel_view_ref.cpp on the oracle's
parameters and mip pyramid): bit-exact RGBA, texel-index map and visited-texel count (vct_debug_counter 1), on uploaded
grids, on a grid voxelised end to end and at the size of configs 2 and 3; and how the view fits the context's frame
state.  Run with -m gpu on a B200."""
import os
import subprocess

import numpy as np
import pytest

from test_voxel_view import MISS, cam_uniforms, sparse_grid
from vct_b200 import capi, scenes, uniforms
from voxel_view_ref import render_voxels as ref_view

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def device_view(c, level):
    H, W = c.get_i("screen_height"), c.get_i("screen_width")
    rgba, vox = np.empty((H, W, 4), np.uint8), np.empty((H, W), np.uint32)
    c.render_voxels(level, rgba, vox)
    return rgba, vox, c.debug_counter(1)


def assert_same_view(c, oracle, level, what):
    rgba, vox, steps = device_view(c, level)
    orgba, ovox, osteps = ref_view(oracle, level)
    hits = int((vox != MISS).sum())
    print(f"[voxel view] {what} level {level}: {hits} of {vox.size} pixels hit, {steps} texels visited")
    assert np.array_equal(vox, ovox), f"{what} level {level}: {(vox != ovox).sum()} texel indices differ"
    assert np.array_equal(rgba, orgba), f"{what} level {level}: {(rgba != orgba).any(-1).sum()} pixels differ"
    assert steps == osteps, f"{what} level {level}: {steps} texels visited vs {osteps}"
    assert np.array_equal(c.read_frame(), rgba)        # the view is the context's frame now
    return hits


# grid of G = 150 world units: [-75, 75]^3
UPLOAD_CAMERAS = {
    "outside": dict(eye=(160.0, 95.0, 210.0), center=(0.0, 0.0, 0.0)),
    "inside": dict(eye=(11.0, -23.0, 31.0), center=(-60.0, 40.0, -150.0)),
    "axis": dict(eye=(0.0, 0.0, 260.0), center=(0.0, 0.0, 0.0)),
}


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("V", [16, 64, 128])
def test_uploaded_grids_match_the_reference(gpu_ctx, oracle, V, fmt):
    c = gpu_ctx
    g = sparse_grid(V, seed=V + fmt, fmt=fmt, density=0.02)
    hits = 0
    for cam, kw in sorted(UPLOAD_CAMERAS.items()):
        u = cam_uniforms(V, size=(123, 77), G=150.0, fmt=fmt, **kw)
        c.set_uniforms(u); c.upload_grid_level0(g)
        oracle.set_uniforms(u); oracle.set_grid_level0(g)
        for level in range(V.bit_length()):
            hits += assert_same_view(c, oracle, level, f"V={V} fmt={fmt} {cam}")
    assert hits > 0


def test_config1_cornell_voxelised_end_to_end(gpu_ctx, oracle):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=256, shadow_map_size=1024, coverage="msaa4")
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels()
    oracle.set_uniforms(u); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels()
    assert np.array_equal(c.grid(0), oracle.grid(0))
    for level in range(7):
        assert_same_view(c, oracle, level, "config 1")


def test_config2_and_config3_size(gpu_ctx, oracle):
    """configs 2 (256^3, 1080p) and 3 (512^3 RGBA16F, 4K) voxelised on the device; the oracle's pyramid is built from the
    device's own level 0 (its textured radiance may differ from the oracle's voxelisation by 1-2 LSB, which
    un-premultiplying magnifies)"""
    sc = scenes.atrium()
    c = gpu_ctx
    for what, kw, levels in (("config 2", dict(V=256, width=1920, height=1080), (0, 1, 2, 4)),
                             ("config 3", dict(V=512, width=3840, height=2160, cones="9+1", grid_format=1), (0, 2))):
        u = uniforms.scene_uniforms(sc, shadow_map_size=4096, coverage="conservative", **kw)
        c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels(); c.sync()
        oracle.set_uniforms(u)
        oracle.set_grid_level0(c.grid(0))
        for level in levels:
            assert assert_same_view(c, oracle, level, what) > 0


def cornell_ctx(c, V=64, size=256):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=V, width=size, height=size, shadow_map_size=1024, coverage="msaa4")
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth()
    return sc, u


def test_frames_around_a_voxel_view_are_unchanged(gpu_ctx):
    c = gpu_ctx
    cornell_ctx(c)
    c.frame(); c.sync()
    before = c.read_frame()
    view, _, _ = device_view(c, 1)
    assert not np.array_equal(view, before)
    c.frame(); c.sync()
    assert np.array_equal(c.read_frame(), before)
    c.render(); c.sync()
    rendered = c.read_frame()
    c.render_voxels(0)                                    # asynchronous form
    c.render(); c.sync()
    assert np.array_equal(c.read_frame(), rendered)


def test_view_behind_frames_in_flight(gpu_ctx):
    """a view enqueued behind three vct_frame_async frames shows the pyramid of the last of them"""
    c = gpu_ctx
    sc, u = cornell_ctx(c)
    xyz = sc.verts[:, :3].astype(np.float32)
    hosts = [np.empty((256, 256, 4), np.uint8) for _ in range(3)]
    shift = lambda k: (xyz + np.float32(150.0 * k) * np.array([1, 0, 0], np.float32)).astype(np.float32)
    c.update_positions(shift(0)); c.draw_depth(); c.frame(); c.sync()
    first, _, _ = device_view(c, 2)
    for k in range(3):
        c.update_positions(shift(k + 1)); c.draw_depth()        # moving the mesh invalidates the shadow map
        c.frame_async(hosts[k])
    behind = np.empty((256, 256, 4), np.uint8)
    behind_vox = np.empty((256, 256), np.uint32)
    c.render_voxels(2, behind, behind_vox)
    for _ in range(3):
        c.frame_wait()
    after, after_vox, _ = device_view(c, 2)
    assert np.array_equal(behind, after) and np.array_equal(behind_vox, after_vox)
    assert not np.array_equal(first, after)               # the frames in flight did move the geometry


def test_row_sharding_uniforms_do_not_change_the_view(gpu_ctx):
    c = gpu_ctx
    cornell_ctx(c, size=200)
    c.draw_voxels()
    want = device_view(c, 1)
    c.set_i("RowInterleave", 2); c.set_i("RowPhase", 1)
    got = device_view(c, 1)
    c.set_i("RowInterleave", 0); c.set_i("RowPhase", 0)
    c.set_i("RowBegin", 50); c.set_i("RowEnd", 60)
    got2 = device_view(c, 1)
    for g in (got, got2):
        assert np.array_equal(g[0], want[0]) and np.array_equal(g[1], want[1]) and g[2] == want[2]


def test_errors_empty_grid_and_pass_time(gpu_ctx):
    c = gpu_ctx
    u = cam_uniforms(32, size=(40, 30), G=150.0, eye=(0.0, 0.0, 200.0), center=(0.0, 0.0, 0.0))
    c.set_uniforms(u)
    rgba, vox, steps = device_view(c, 0)                  # nothing voxelised yet: an empty grid
    assert (rgba.reshape(-1, 4) == (128, 128, 128, 255)).all() and (vox == MISS).all() and steps > 0
    assert c.pass_time_us("voxel_view") > 0
    for level in (-1, 6):
        with pytest.raises(capi.VctError) as e:
            c.render_voxels(level)
        assert e.value.code == -1
    c.upload_grid_level0(sparse_grid(32, seed=1, fmt=0), build_mips=False)
    with pytest.raises(capi.VctError) as e:
        c.render_voxels(1)
    assert e.value.code == -3
    device_view(c, 0)                                     # level 0 is current
    c.build_mips()
    device_view(c, 1)


def test_cpp_facade_voxel_views_equal_the_ctypes_binding(gpu_ctx, tmp_path):
    """facade_demo dumps Voxel_Cone_Tracing::RenderVoxels(1) of each view; the same inputs through ctypes give the same
    bytes"""
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
    c = gpu_ctx
    for f in range(3):
        raw = rd(f"uniforms_{f}.f32", np.float32)
        u = uniforms.reference_uniforms(V=64, width=256, height=256, shadow_map_size=4096, coverage="msaa4")
        for k, name in enumerate(names):
            u[name] = raw[16 * k:16 * k + 16].copy()
        u["CameraPosition"] = raw[96:99].copy()
        c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels()
        want = rd(f"voxels_{f}.rgba", np.uint8).reshape(256, 256, 4)
        got, vox, _ = device_view(c, 1)
        assert (vox != MISS).sum() > 1000
        assert np.array_equal(got, want), f"view {f}: C++ facade and ctypes binding disagree"
