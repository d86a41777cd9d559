"""Calls on host arrays share one device staging buffer per context.  Interleaved on one context, calls of very different
sizes (a large cone trace and voxel sampling, a few ray casts, a probe bake, a voxel view, the visibility read-back and a
position update) give the same bytes as the same call on a fresh context; a call right after one that failed is still
right; and each call launches exactly its own kernels.  Run with -m gpu on a B200."""
import numpy as np
import pytest

from test_gpu_probes import seeded_probes
from test_raycast import segment_mix
from test_voxel_view import sparse_grid
from vct_b200 import capi, scenes, uniforms

pytestmark = pytest.mark.gpu

G, V, SIZE = 150.0, 64, 256


def cornell(c):
    sc = scenes.cornell()
    c.set_uniforms(uniforms.scene_uniforms(sc, V=V, width=SIZE, height=SIZE, shadow_map_size=1024, coverage="msaa4"))
    c.load_scene(sc); c.draw_depth(); c.frame(); c.sync()
    return sc


def on_fresh_context(call, *setup):
    c = capi.Context(0)
    try:
        cornell(c)
        for s in setup:
            s(c)
        return call(c)
    finally:
        c.close()


def cones(n, seed):
    rng = np.random.default_rng(seed)
    starts = rng.uniform(-0.5 * G, 0.5 * G, (n, 3)).astype(np.float32)
    dirs = rng.normal(size=(n, 3)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    return starts, dirs, rng.uniform(0.05, 0.6, n).astype(np.float32)


def view(c, level):
    rgba, vox = np.empty((SIZE, SIZE, 4), np.uint8), np.empty((SIZE, SIZE), np.uint32)
    c.render_voxels(level, rgba, vox)
    return rgba, vox


def frame(c):
    c.draw_depth(); c.frame(); c.sync()
    return c.read_frame(), c.visibility()


def as_bytes(result):
    parts = result if isinstance(result, tuple) else (result,)
    return [np.ascontiguousarray(p).view(np.uint8).tobytes() for p in parts]


def test_interleaved_host_calls_equal_fresh_contexts(gpu_ctx):
    c = gpu_ctx
    sc = cornell(c)
    big, small = cones(1 << 20, seed=1), cones(999, seed=2)
    pos = np.random.default_rng(3).uniform(-0.5 * G, 0.5 * G, (1 << 20, 3)).astype(np.float32)
    lod = np.random.default_rng(4).uniform(0.0, 5.0, 1 << 20).astype(np.float32)
    moved = (sc.verts[:, :3] + np.array([7.5, 0.0, -3.0], np.float32)).astype(np.float32)
    # (name, call, kernels it launches): large, small and medium arrays in turn, in and out of the same buffer
    calls = [("trace_cones 1M", lambda x: x.trace_cones(*big), 1),
             ("cast_rays 32", lambda x: x.cast_rays(2, segment_mix(V, G, seed=5, n=8)), 1),
             ("bake_probes 500", lambda x: x.bake_probes(seeded_probes(500, G, seed=6)), 1),
             ("render_voxels", lambda x: view(x, 1), 1),
             ("visibility", lambda x: x.visibility(), 1),
             ("sample_voxels 1M", lambda x: x.sample_voxels(pos, lod), 1),
             ("trace_cones 999", lambda x: x.trace_cones(*small), 1),
             ("cast_rays 16K", lambda x: x.cast_rays(0, segment_mix(V, G, seed=7)), 1)]
    got = {}
    for name, call, kernels in calls:
        before = c.kernel_launches()
        got[name] = as_bytes(call(c))
        assert c.kernel_launches() - before == kernels, name
    before = c.kernel_launches()
    c.update_positions(moved)                                            # host form: one scatter kernel
    assert c.kernel_launches() - before == 1
    got["frame after update_positions"] = as_bytes(frame(c))
    got["trace_cones 999 after the update"] = as_bytes(c.trace_cones(*small))
    for name, call, _ in calls:
        assert on_fresh_context(lambda x: as_bytes(call(x))) == got[name], name
    move = lambda x: x.update_positions(moved)
    assert on_fresh_context(lambda x: as_bytes(frame(x)), move) == got["frame after update_positions"]
    assert on_fresh_context(lambda x: as_bytes(x.trace_cones(*small)), move, frame) == got["trace_cones 999 after the update"]


def test_host_call_after_a_failed_call(gpu_ctx):
    c = gpu_ctx
    cornell(c)
    g = sparse_grid(V, seed=8, fmt=0, density=0.05)
    segs = segment_mix(V, G, seed=9, n=2000)
    c.trace_cones(*cones(1 << 18, seed=10))                              # leaves a large staging buffer behind
    c.upload_grid_level0(g, build_mips=False)
    before = c.kernel_launches()
    for fail in (lambda: c.cast_rays(1, segs), lambda: c.bake_probes(seeded_probes(64, G, seed=11)),
                 lambda: c.render_voxels(1, np.empty((SIZE, SIZE, 4), np.uint8))):
        with pytest.raises(capi.VctError) as e:                          # the mip levels are stale
            fail()
        assert e.value.code == -3
    assert c.kernel_launches() == before                                 # a refused call launches nothing
    got = as_bytes(c.cast_rays(0, segs))                                 # level 0 is current
    assert c.kernel_launches() == before + 1
    upload = lambda x: x.upload_grid_level0(g, build_mips=False)
    assert on_fresh_context(lambda x: as_bytes(x.cast_rays(0, segs)), upload) == got
