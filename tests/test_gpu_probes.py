"""Irradiance probes on the device (vct_bake_probes): bit-exact against the float32 composition of vct_trace_cones on
the same device, against hand-derived answers, within the cone bars of test_trace_cones_vs_oracle against the CPU
reference (tests/probe_ref.py on the oracle), and how a bake fits the context's frame state.  Run with -m gpu on a
B200."""
import os
import subprocess

import numpy as np
import pytest

from probe_ref import PROBES_KAT, bake_probes as ref_bake, combine, face_directions, face_starts
from vct_b200 import capi, scenes, uniforms

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def cone_table(kind):
    if kind == "16":
        rng = np.random.default_rng(16)
        d = rng.normal(size=(16, 3))
        d[:, 2] = np.abs(d[:, 2]) + 0.3                          # a hemisphere around the surface normal
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        return d.astype(np.float32), np.full(16, 1.0 / 16.0, dtype=np.float32)
    return uniforms.cone_set(kind)


def seeded_probes(n, G, seed):
    """n points in [-0.65 G, 0.65 G]^3: inside the grid and (about half of them) outside it, where it repeats"""
    return np.random.default_rng(seed).uniform(-0.65 * G, 0.65 * G, (n, 3)).astype(np.float32)


def composed(c, xyz, dirs, weights, G, V, tan=0.577):
    """every cone of every face traced by vct_trace_cones, then summed in cone order in float32"""
    fd = face_directions(dirs)                                    # (6, nc, 3)
    st = face_starts(xyz, G, V)                                   # (n, 6, 3)
    n, nc = xyz.shape[0], fd.shape[1]
    S = np.ascontiguousarray(np.broadcast_to(st[:, :, None, :], (n, 6, nc, 3))).reshape(-1, 3)
    D = np.ascontiguousarray(np.broadcast_to(fd[None], (n, 6, nc, 3))).reshape(-1, 3)
    r, steps = c.trace_cones(S, D, np.float32(tan))
    return combine(r.reshape(n, 6, nc, 4), weights), steps.reshape(n, 6, nc).sum(-1)


def assert_bit_identical(got, want, what):
    (o, s), (wo, ws) = got, want
    bad = (o.view(np.uint32) != wo.view(np.uint32)).any(-1)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} faces differ, e.g. {o[bad][:2]} vs {wo[bad][:2]}"
    assert np.array_equal(s.astype(np.int64), ws.astype(np.int64)), f"{what}: step counts differ"


SCENES = {
    "config1 cornell": (scenes.cornell, dict(V=64, width=256, height=256, shadow_map_size=1024, coverage="msaa4")),
    "config2 atrium": (scenes.atrium, dict(V=256, width=1920, height=1080, shadow_map_size=4096, coverage="conservative")),
}


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("scene", sorted(SCENES))
def test_bake_equals_the_composition_of_trace_cones(gpu_ctx, scene, fmt):
    factory, kw = SCENES[scene]
    sc = factory()
    u = uniforms.scene_uniforms(sc, grid_format=fmt, **kw)
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels(); c.sync()
    G, V = u["VoxelGridWorldSize"], u["VoxelDimensions"]
    xyz = seeded_probes(2000, G, seed=V + fmt)
    for kind in ("6+1", "5+1", "9+1", "16"):
        dirs, w = cone_table(kind)
        c.set_cones(dirs, w)
        got = c.bake_probes(xyz)
        assert_bit_identical(got, composed(c, xyz, dirs, w, G, V), f"{scene} fmt {fmt} cones {kind}")
        assert (got[0][..., 3] < 1.0).mean() > 0.1                # the probes do see the scene


@pytest.mark.parametrize("cones", ["6+1", "5+1", "9+1"])
def test_uniform_and_empty_grid_known_answers(gpu_ctx, cones):
    V = 128
    c = gpu_ctx
    c.set_uniforms(uniforms.reference_uniforms(V=V, cones=cones))
    n_cones = len(uniforms.cone_set(cones)[1])
    g = np.empty((V, V, V, 4), dtype=np.uint8); g[..., :3] = 153; g[..., 3] = 255
    c.upload_grid_level0(g)
    out, steps = c.bake_probes(PROBES_KAT)
    vws = 150.0 / V
    np.testing.assert_allclose(out[..., :3], 153 / 255.0, atol=1e-4)
    np.testing.assert_allclose(out[..., 3], 1.0 - 1.0 / (1.0 + 0.03 * 2 * 0.577 * vws), atol=1e-4)
    assert np.all(steps == n_cones)
    c.upload_grid_level0(np.zeros_like(g))
    out, steps = c.bake_probes(PROBES_KAT)
    assert np.all(out[..., :3] == 0.0) and np.all(out[..., 3] == 1.0) and np.all(steps == 6 * n_cones)


def assert_close_to_reference(got, want, what):
    (o, s), (wo, ws) = got, want
    ds = np.abs(s.astype(np.int64) - ws)
    same = ds == 0
    err = np.abs(o - wo)[same]
    p999, mean = float(np.percentile(err, 99.9)), float(err.mean())
    print(f"[probes] {what}: steps within 1 on {100 * (ds <= 1).mean():.3f} % of faces, equal on "
          f"{100 * same.mean():.3f} %; |diff| p99.9 {p999 * 255:.3f}/255, mean {mean * 255:.4f}/255")
    # the alpha >= MaxAlpha early-out may fire one step apart when alpha sits on the threshold
    assert (ds <= 1).mean() >= 0.995, what
    assert p999 <= 2.5 / 255 and mean < 0.5 / 255, (what, p999, mean)


def test_blob_grid_and_cornell_vs_oracle(gpu_ctx, oracle):
    V = 64
    rng = np.random.default_rng(3)
    g = np.zeros((V, V, V, 4), dtype=np.uint8)                   # the grid of test_trace_cones_vs_oracle
    blob = np.kron(rng.random((V // 4, V // 4, V // 4)) < 0.25, np.ones((4, 4, 4), dtype=bool))
    g[blob] = rng.integers(30, 255, (int(blob.sum()), 4), dtype=np.uint8)
    g[..., 3][blob] = 255
    u = uniforms.reference_uniforms(V=V)
    c = gpu_ctx
    c.set_uniforms(u); oracle.set_uniforms(u)
    c.upload_grid_level0(g); oracle.set_grid_level0(g)
    xyz = seeded_probes(1000, 150.0, seed=5)
    assert_close_to_reference(c.bake_probes(xyz), ref_bake(oracle, xyz), "blob grid")

    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=256, shadow_map_size=1024, coverage="msaa4")
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels()
    oracle.set_uniforms(u); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels()
    assert np.array_equal(c.grid(0), oracle.grid(0))
    xyz = seeded_probes(1000, 150.0, seed=6)
    assert_close_to_reference(c.bake_probes(xyz), ref_bake(oracle, xyz), "config 1 cornell")


def test_config3_size_vs_oracle(gpu_ctx, oracle):
    """512^3 RGBA16F with 9+1 cones; the oracle's pyramid is built from the device's level 0"""
    sc = scenes.atrium()
    u = uniforms.scene_uniforms(sc, V=512, width=3840, height=2160, cones="9+1", grid_format=1, shadow_map_size=4096,
                                coverage="conservative")
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth(); c.draw_voxels(); c.sync()
    oracle.set_uniforms(u)
    oracle.set_grid_level0(c.grid(0))
    xyz = seeded_probes(500, 150.0, seed=512)
    assert_close_to_reference(c.bake_probes(xyz), ref_bake(oracle, xyz), "config 3")


def test_host_and_device_forms_give_identical_bytes(gpu_ctx):
    import torch
    c = gpu_ctx
    cornell_ctx(c); c.draw_voxels()
    xyz = seeded_probes(777, 150.0, seed=9)
    out, steps = c.bake_probes(xyz)
    dx = torch.from_numpy(xyz).cuda()
    dout = torch.full((777, 6, 4), -1.0, dtype=torch.float32, device="cuda")
    dsteps = torch.zeros((777, 6), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    c.bake_probes(n=777, device_xyz=dx.data_ptr(), device_out=dout.data_ptr(), device_steps=dsteps.data_ptr())
    c.sync()
    assert np.array_equal(dout.cpu().numpy().view(np.uint32), out.view(np.uint32))
    assert np.array_equal(dsteps.cpu().numpy().view(np.uint32), steps)
    c.bake_probes(n=777, device_xyz=dx.data_ptr(), device_out=dout.data_ptr())   # steps are optional
    c.sync()
    assert np.array_equal(dout.cpu().numpy().view(np.uint32), out.view(np.uint32))


def cornell_ctx(c, V=64, size=256):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=V, width=size, height=size, shadow_map_size=1024, coverage="msaa4")
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth()
    return sc, u


def test_frames_around_a_bake_are_unchanged(gpu_ctx):
    c = gpu_ctx
    cornell_ctx(c)
    c.frame(); c.sync()
    before, samples = c.read_frame(), c.cone_samples()
    c.bake_probes(seeded_probes(300, 150.0, seed=1))
    assert c.cone_samples() == samples
    assert np.array_equal(c.read_frame(), before)                # the bake does not write the frame buffer
    c.frame(); c.sync()
    assert np.array_equal(c.read_frame(), before) and c.cone_samples() == samples


def test_bake_behind_frames_in_flight(gpu_ctx):
    """a bake enqueued behind three vct_frame_async frames reads the pyramid of the last of them"""
    c = gpu_ctx
    sc, u = cornell_ctx(c)
    xyz = sc.verts[:, :3].astype(np.float32)
    probes = seeded_probes(500, 150.0, seed=2)
    hosts = [np.empty((256, 256, 4), np.uint8) for _ in range(3)]
    shift = lambda k: (xyz + np.float32(150.0 * k) * np.array([1, 0, 0], np.float32)).astype(np.float32)
    c.update_positions(shift(0)); c.draw_depth(); c.frame(); c.sync()
    first = c.bake_probes(probes)
    for k in range(3):
        c.update_positions(shift(k + 1)); c.draw_depth()
        c.frame_async(hosts[k])
    behind = c.bake_probes(probes)
    for _ in range(3):
        c.frame_wait()
    after = c.bake_probes(probes)
    assert_bit_identical(behind, after, "bake behind frames in flight")
    assert not np.array_equal(first[0], after[0])                 # the frames in flight did move the geometry


def test_camera_and_row_sharding_uniforms_do_not_change_the_bake(gpu_ctx):
    c = gpu_ctx
    cornell_ctx(c); c.draw_voxels()
    probes = seeded_probes(400, 150.0, seed=4)
    want = c.bake_probes(probes)
    c.set_3f("CameraPosition", (30.0, -12.0, 80.0))
    c.set_mat4("ModelViewMatrix", np.arange(16, dtype=np.float32))
    c.set_mat4("ProjectionMatrix", np.eye(4, dtype=np.float32) * 2)
    c.set_i("screen_width", 97); c.set_i("screen_height", 31)
    assert_bit_identical(c.bake_probes(probes), want, "camera uniforms")
    c.set_i("RowInterleave", 2); c.set_i("RowPhase", 1)
    assert_bit_identical(c.bake_probes(probes), want, "interleaved rows")
    c.set_i("RowInterleave", 0); c.set_i("RowPhase", 0); c.set_i("RowBegin", 5); c.set_i("RowEnd", 9)
    assert_bit_identical(c.bake_probes(probes), want, "row band")


def test_errors_nan_probes_and_counters(gpu_ctx):
    c = gpu_ctx
    c.set_uniforms(uniforms.reference_uniforms(V=32))
    out, steps = c.bake_probes(PROBES_KAT)                          # nothing voxelised yet: an empty grid
    assert np.all(out[..., :3] == 0.0) and np.all(out[..., 3] == 1.0)
    for kw in (dict(device_xyz=0, device_out=1 << 20), dict(device_xyz=1 << 20, device_out=0)):
        with pytest.raises(capi.VctError) as e:
            c.bake_probes(n=4, **kw)
        assert e.value.code == -1
    with pytest.raises(capi.VctError) as e:
        c.bake_probes(n=1 << 60, device_xyz=1 << 20, device_out=1 << 20)
    assert e.value.code == -1
    out, steps = c.bake_probes(np.zeros((0, 3), np.float32))     # n = 0: a no-op
    assert out.shape == (0, 6, 4) and steps.shape == (0, 6)
    rng = np.random.default_rng(11)
    g = np.zeros((32, 32, 32, 4), np.uint8)
    occ = rng.random((32, 32, 32)) < 0.1
    g[occ] = rng.integers(1, 256, (int(occ.sum()), 4), dtype=np.uint8)
    c.upload_grid_level0(g, build_mips=False)
    with pytest.raises(capi.VctError) as e:
        c.bake_probes(PROBES_KAT)
    assert e.value.code == -3
    c.build_mips()
    xyz = seeded_probes(64, 150.0, seed=12)
    want, want_steps = c.bake_probes(xyz)
    bad = xyz.copy()
    bad[10, 1] = np.nan; bad[11, 0] = np.inf; bad[12, 2] = -np.inf
    out, steps = c.bake_probes(bad)
    assert np.all(np.isnan(out[10:13])) and np.all(steps[10:13] == 0)
    keep = np.ones(64, bool); keep[10:13] = False
    assert np.array_equal(out[keep].view(np.uint32), want[keep].view(np.uint32))
    assert np.array_equal(steps[keep], want_steps[keep])
    assert c.debug_counter(2) == int(steps.sum()) > 0
    assert c.pass_time_us("probes") > 0


def test_cpp_facade_probes_equal_the_ctypes_binding(gpu_ctx, tmp_path):
    """facade_demo bakes the cell centres of an 8x8x8 lattice through Voxel_Cone_Tracing::BakeProbes after its frames;
    the same inputs through ctypes give the same bytes"""
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
    xyz = rd("probe_xyz.f32", np.float32).reshape(-1, 3)
    cells = (np.arange(8, dtype=np.float32) + np.float32(0.5)) * np.float32(150.0 / 8) - np.float32(75.0)
    z, y, x = np.meshgrid(cells, cells, cells, indexing="ij")
    assert np.array_equal(xyz, np.stack([x, y, z], -1).reshape(-1, 3))
    want = rd("probes.f32", np.float32).reshape(-1, 6, 4)
    got, _ = c.bake_probes(xyz)
    assert (got[..., 3] < 1.0).any()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), "C++ facade and ctypes binding disagree"
