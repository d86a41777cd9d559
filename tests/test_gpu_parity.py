"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against the CPU
oracle on the same seeded inputs, against the committed golden fixtures, and -- at BASELINE config-2 size --
through size-independent properties.

Bars (BASELINE.json north_star): shadow map, voxel occupancy and fragment counts bit-exact; radiance and
frames PSNR >= 40 dB and |diff| <= 2/255 on >= 99.9 % of voxels/pixels.
"""
import importlib.util
import os
import zlib

import numpy as np
import pytest

from conftest import frac_within, psnr
from vct_b200 import capi, scenes, uniforms

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
make_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(make_golden)

PSNR_MIN = 40.0       # dB, north_star
LSB_TOL = 2           # /255
FRAC_MIN = 0.999      # the bar on the BASELINE configs (config 1 at 256x256, config 2 at 1080p)
# The reference's cone loop `while (dist < MAX_DISTANCE && alpha < 0.95)` (VoxelConeTracing.fs:94) is a hard
# threshold: a sub-LSB filtering difference on a sample whose alpha lands on 0.95 adds or drops a whole
# step (up to 0.05 * radiance, ~5/255 through the specular cone).  On the 96x96 / 32^3 fixtures a few dozen
# border pixels sit exactly there (tools/probe_outliers.py), so the small fixtures use a slightly wider bar.
FRAC_MIN_SMALL = 0.995


def run_gpu(c, sc, u):
    c.set_uniforms(u)
    c.load_scene(sc)
    c.draw_depth()
    c.draw_voxels()
    c.render()
    c.sync()


def run_oracle(o, sc, u):
    o.set_uniforms(u)
    o.load_scene(sc)
    o.draw_depth()
    o.draw_voxels()
    o.render()


def assert_radiance_close(a, b, what):
    assert a.shape == b.shape
    occ = (a[..., 3] > 0) | (b[..., 3] > 0) if a.shape[-1] == 4 else np.ones(a.shape[:-1], bool)
    if occ.any():
        d = np.abs(a.astype(int) - b.astype(int)).max(-1)[occ]
        assert (d <= LSB_TOL).mean() >= FRAC_MIN, f"{what}: {(d <= LSB_TOL).mean():.5f} within {LSB_TOL}"
    assert psnr(a, b) >= PSNR_MIN, f"{what}: psnr {psnr(a, b):.2f}"


def assert_frame_close(fg, fo, what, frac_min=FRAC_MIN):
    p, f = psnr(fg[..., :3], fo[..., :3]), frac_within(fg, fo, LSB_TOL)
    print(f"[parity] {what}: psnr {p:.2f} dB, {100 * f:.4f} % of pixels within {LSB_TOL}/255 (bar {100 * frac_min:.1f} %)")
    assert p >= PSNR_MIN, f"{what}: psnr {p:.2f}"
    assert f >= frac_min, f"{what}: {f:.5f}"


# ------------------------------------------------------------------------------------------ golden fixtures
@pytest.mark.parametrize("name", sorted(make_golden.CASES))
def test_gpu_matches_golden_fixture(gpu_ctx, name):
    gold = np.load(os.path.join(HERE, "golden", name + ".npz"))
    factory, kw = make_golden.CASES[name]
    sc = factory()
    run_gpu(gpu_ctx, sc, uniforms.scene_uniforms(sc, **kw))
    d = gpu_ctx.depth()
    assert np.uint32(zlib.crc32(d.tobytes())) == gold["depth_crc"]
    assert np.array_equal(gpu_ctx.counts().astype(np.uint16), gold["counts"])          # bit-exact
    assert np.array_equal(gpu_ctx.grid(0)[..., 3], gold["grid0"][..., 3])               # occupancy bit-exact
    for lvl, key in ((0, "grid0"), (1, "grid1"), (2, "grid2"), (4, "grid4")):
        assert_radiance_close(gpu_ctx.grid(lvl), gold[key], f"{name} grid L{lvl}")
    vis = gpu_ctx.visibility()
    assert (vis != gold["visibility"]).mean() <= 1e-3
    assert_frame_close(gpu_ctx.read_frame(), gold["frame"], name, FRAC_MIN_SMALL)
    if "cornell" in name:      # 1x1 textures: no hardware texture filtering involved => exact integers
        assert np.array_equal(gpu_ctx.sums(), gold["sums"])
        assert np.array_equal(gpu_ctx.grid(0), gold["grid0"]) and np.array_equal(gpu_ctx.grid(2), gold["grid2"])
        assert np.array_equal(vis, gold["visibility"])


# ------------------------------------------------------------------------------------------ config 1
@pytest.mark.parametrize("coverage", ["center", "msaa4", "conservative"])
def test_cornell_config1_vs_oracle(gpu_ctx, oracle, coverage):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=256, shadow_map_size=1024, coverage=coverage)
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    assert np.array_equal(gpu_ctx.depth(), oracle.depth())
    assert np.array_equal(gpu_ctx.counts(), oracle.counts())
    assert np.array_equal(gpu_ctx.sums(), oracle.sums())
    for l in range(7):
        assert np.array_equal(gpu_ctx.grid(l), oracle.grid(l)), f"level {l}"
    assert np.array_equal(gpu_ctx.visibility(), oracle.visibility())
    assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), f"cornell {coverage}")
    assert abs(gpu_ctx.cone_samples() - oracle.cone_samples()) <= 1e-4 * oracle.cone_samples()
    assert gpu_ctx.occupied_voxels() == int((oracle.counts() > 0).sum())


def test_reference_default_cone_sets(gpu_ctx, oracle):
    sc = scenes.cornell()
    for cones in ("5+1", "9+1"):
        u = uniforms.scene_uniforms(sc, V=32, width=128, height=128, shadow_map_size=512, cones=cones)
        run_gpu(gpu_ctx, sc, u)
        run_oracle(oracle, sc, u)
        assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), cones, FRAC_MIN_SMALL)


# ------------------------------------------------------------------------------------------ textured scene
def test_atrium_reduced_vs_oracle(gpu_ctx, oracle):
    sc = scenes.atrium(detail=0.3, tex_size=128)
    u = uniforms.scene_uniforms(sc, V=128, width=640, height=360, shadow_map_size=2048, coverage="conservative")
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    assert np.array_equal(gpu_ctx.depth(), oracle.depth())
    cg, co = gpu_ctx.counts(), oracle.counts()
    assert np.array_equal(cg, co)                                     # occupancy and counts: bit-exact
    assert cg.sum() > 100_000
    # sums differ only through the hardware-filtered albedo fetch: <= 1 LSB per fragment
    ds = np.abs(gpu_ctx.sums().astype(np.int64) - oracle.sums().astype(np.int64)).max(-1)
    assert np.all(ds <= cg)
    for l in range(8):
        g, o = gpu_ctx.grid(l), oracle.grid(l)
        assert np.array_equal(g[..., 3] > 0, o[..., 3] > 0)
        assert np.abs(g.astype(int) - o.astype(int)).max() <= LSB_TOL
    assert (gpu_ctx.visibility() != oracle.visibility()).mean() <= 1e-3
    assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), "atrium reduced")


# ------------------------------------------------------------------------------------------ mip kernel
@pytest.mark.parametrize("V", [2, 8, 16, 32, 64, 128, 256])
def test_mip_pyramid_bit_exact(gpu_ctx, oracle, V):
    rng = np.random.default_rng(V)
    g = rng.integers(0, 256, (V, V, V, 4), dtype=np.uint8)
    g[rng.random((V, V, V)) < 0.7] = 0                                # sparse like a voxelised scene
    gpu_ctx.set_i("VoxelDimensions", V)
    oracle.set_uniforms(uniforms.reference_uniforms(V=V))
    gpu_ctx.upload_grid_level0(g)
    oracle.set_grid_level0(g)
    gpu_ctx.sync()
    for l in range(V.bit_length()):
        assert np.array_equal(gpu_ctx.grid(l), oracle.grid(l)), f"V={V} level {l}"


def test_mip_rounding_kat_on_gpu(gpu_ctx):
    V = 16
    gpu_ctx.set_i("VoxelDimensions", V)
    g = np.zeros((V, V, V, 4), dtype=np.uint8)
    g[5, 9, 3] = 255
    gpu_ctx.upload_grid_level0(g)
    assert gpu_ctx.grid(1)[2, 4, 1, 0] == 32 and gpu_ctx.grid(2)[1, 2, 0, 0] == 4
    assert gpu_ctx.grid(3)[0, 1, 0, 0] == 1 and gpu_ctx.grid(4)[0, 0, 0, 0] == 0


# ------------------------------------------------------------------------------------------ cone marching
def test_trace_cones_vs_oracle(gpu_ctx, oracle):
    V = 64
    rng = np.random.default_rng(3)
    # smooth-ish random field so that the 8-bit hardware filter weights stay inside the tolerance
    g = np.zeros((V, V, V, 4), dtype=np.uint8)
    blob = rng.random((V // 4, V // 4, V // 4)) < 0.25
    blob = np.kron(blob, np.ones((4, 4, 4), dtype=bool))
    g[blob] = rng.integers(30, 255, (int(blob.sum()), 4), dtype=np.uint8)
    g[..., 3][blob] = 255
    u = uniforms.reference_uniforms(V=V)
    gpu_ctx.set_uniforms(u); oracle.set_uniforms(u)
    gpu_ctx.upload_grid_level0(g); oracle.set_grid_level0(g)
    n = 4000
    starts = rng.uniform(-70, 70, (n, 3)).astype(np.float32)
    dirs = rng.normal(size=(n, 3)); dirs = (dirs / np.linalg.norm(dirs, axis=1, keepdims=True)).astype(np.float32)
    tans = np.where(np.arange(n) % 2 == 0, 0.577, 0.07).astype(np.float32)
    out, steps = gpu_ctx.trace_cones(starts, dirs, tans)
    ref = np.zeros_like(out); rsteps = np.zeros(n, dtype=np.int64)
    for i in range(n):
        ref[i], rsteps[i] = oracle.cone(starts[i], dirs[i], float(tans[i]))
    # the alpha >= 0.95 early-out may fire one step apart when alpha sits on the threshold
    assert (np.abs(steps.astype(np.int64) - rsteps) <= 1).mean() > 0.995
    same = steps == rsteps
    err = np.abs(out - ref)[same]
    assert np.percentile(err, 99.9) <= 2.5 / 255 and err.mean() < 0.5 / 255, (np.percentile(err, 99.9), err.mean())


def test_uniform_grid_cone_kat_on_gpu(gpu_ctx):
    V = 128
    gpu_ctx.set_uniforms(uniforms.reference_uniforms(V=V))
    g = np.empty((V, V, V, 4), dtype=np.uint8); g[..., :3] = 153; g[..., 3] = 255
    gpu_ctx.upload_grid_level0(g)
    out, steps = gpu_ctx.trace_cones([[1.0, 2.0, 3.0]] * 2, [[0, 1, 0]] * 2, [0.07, 0.577])
    assert list(steps) == [1, 1]
    np.testing.assert_allclose(out[0, :3], 153 / 255.0, atol=1e-3)
    np.testing.assert_allclose(out[0, 3], 0.966038, atol=1e-4)         # 1/(1+0.03*vws), SURVEY A.7
    g[:] = 0
    gpu_ctx.upload_grid_level0(g)
    out, steps = gpu_ctx.trace_cones([[0, 0, 0]] * 2, [[0, 0, 1]] * 2, [0.577, 0.07])
    assert list(steps) == [6, 23] and np.all(out == 0)                 # A.5 step table at V=128


# ------------------------------------------------------------------------------------------ edge cases
def _tri_mesh(tris_world):
    t = np.asarray(tris_world, dtype=np.float64).reshape(-1, 3, 3) * 20.0
    v = np.zeros((t.shape[0] * 3, 14), dtype=np.float32)
    v[:, :3] = t.reshape(-1, 3)
    v[:, 3:6] = (0, 0, 1); v[:, 8:11] = (1, 0, 0); v[:, 11:14] = (0, 1, 0)
    v[:, 6:8] = np.tile([[0, 0], [1, 0], [0, 1]], (t.shape[0], 1))
    return v, np.arange(t.shape[0] * 3, dtype=np.uint32).reshape(-1, 3)


def test_degenerate_offgrid_and_huge_triangles(gpu_ctx, oracle):
    nan = float("nan")
    tris = [
        [(0, 0, 0), (0, 0, 0), (0, 0, 0)],                      # point
        [(0, 0, 0), (10, 10, 10), (20, 20, 20)],                # zero area (collinear)
        [(200, 200, 200), (210, 200, 200), (200, 210, 200)],    # entirely outside the grid
        [(-9000, -3.3, -9000), (9000, -3.3, -9000), (0, -3.3, 18000)],   # far larger than the grid (guard band)
        [(-80, 20, 5), (80, 20.5, 5), (0, 21, -70)],            # straddles the grid boundary
        [(nan, 0, 0), (1, 0, 0), (0, 1, 0)],                    # NaN vertex
        [(1e30, 0, 0), (0, 1e30, 0), (0, 0, 1e30)],             # overflowing coordinates
        [(10, 10, 74.9), (20, 10, 75.2), (10, 20, 75.0)],       # touches the far clip plane of ProjZ
    ]
    v, i = _tri_mesh(tris)
    for cov in ("center", "msaa4", "conservative"):
        u = uniforms.reference_uniforms(V=64, width=64, height=64, shadow_map_size=256, coverage=cov)
        for x in (gpu_ctx, oracle):
            x.set_uniforms(u)
            x.upload_texture(0, scenes.solid_texture((200, 100, 50)))
            x.upload_mesh(v, i)
            x.draw_depth(); x.draw_voxels(); x.render()
        gpu_ctx.sync()
        assert np.array_equal(gpu_ctx.depth(), oracle.depth()), cov
        assert np.array_equal(gpu_ctx.counts(), oracle.counts()), cov
        assert oracle.counts().sum() > 64 * 64                   # the huge triangle fills a slab
        assert np.array_equal(gpu_ctx.visibility(), oracle.visibility()), cov


def test_errors_are_reported_not_swallowed(gpu_ctx):
    c = gpu_ctx
    with pytest.raises(capi.VctError) as e:
        c.set_i("NoSuchUniform", 1)
    assert e.value.code == -1 and "NoSuchUniform" in str(e.value)
    with pytest.raises(capi.VctError):
        c.set_i("VoxelDimensions", 100)                          # not a power of two
    with pytest.raises(capi.VctError):
        c.set_mat4("NoSuchMatrix", np.eye(4))
    with pytest.raises(capi.VctError) as e:
        c.draw_depth()                                           # no mesh yet
    assert e.value.code == -3
    v, i = _tri_mesh([[(0, 0, 0), (10, 0, 0), (0, 10, 0)]])
    with pytest.raises(capi.VctError):
        c.upload_mesh(v, np.array([[0, 1, 7]], dtype=np.uint32))  # index out of range
    c.upload_mesh(v, i)
    with pytest.raises(capi.VctError) as e:
        c.draw_voxels()                                          # shadow map missing
    assert e.value.code == -3


def test_queue_overflow_is_detected(gpu_ctx):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=64, height=64, shadow_map_size=256)
    gpu_ctx.set_uniforms(u)
    gpu_ctx.set_i("MaxFragments", 2048)
    gpu_ctx.load_scene(sc)
    gpu_ctx.draw_depth()
    gpu_ctx.draw_voxels()
    with pytest.raises(capi.VctError) as e:
        gpu_ctx.sync()
    assert e.value.code == -4
    gpu_ctx.set_i("MaxFragments", 1 << 20)
    gpu_ctx.draw_voxels()
    gpu_ctx.sync()


def test_maximum_grid_size_512(gpu_ctx):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=512, width=128, height=128, shadow_map_size=1024, coverage="center")
    run_gpu(gpu_ctx, sc, u)
    c = gpu_ctx.counts()
    assert c.sum() > 500_000 and gpu_ctx.occupied_voxels() == int((c > 0).sum())
    g0 = gpu_ctx.grid(0)
    assert np.array_equal(g0[..., 3] == 255, c > 0)
    s = g0.astype(np.int64).reshape(256, 2, 256, 2, 256, 2, 4).sum((1, 3, 5))
    assert np.array_equal(((s + 4) >> 3).astype(np.uint8), gpu_ctx.grid(1))
    assert gpu_ctx.grid(9).shape == (1, 1, 1, 4)


# ------------------------------------------------------------------------------------------ config-2 size
@pytest.fixture(scope="module")
def atrium_full():
    return scenes.atrium()


def _cfg2(sc, **kw):
    kw.setdefault("coverage", "conservative")
    return uniforms.scene_uniforms(sc, V=256, width=1920, height=1080, shadow_map_size=4096, **kw)


def test_config2_properties(gpu_ctx, atrium_full):
    sc, c = atrium_full, gpu_ctx
    run_gpu(c, sc, _cfg2(sc))
    counts, sums, g0, frame = c.counts(), c.sums(), c.grid(0), c.read_frame()
    occ = counts > 0
    assert 200_000 < occ.sum() < 2_000_000 and c.occupied_voxels() == int(occ.sum())
    assert np.array_equal(g0[..., 3] == 255, occ)
    avg = (sums.astype(np.int64) + (counts // 2)[..., None]) // np.maximum(counts, 1)[..., None]
    assert np.array_equal(g0[..., :3][occ], avg[occ].astype(np.uint8))            # resolve rule, every voxel
    for l in range(1, 9):                                                         # mip rule, every level
        p = c.grid(l - 1).astype(np.int64)
        n = p.shape[0] // 2
        s = p.reshape(n, 2, n, 2, n, 2, 4).sum((1, 3, 5))
        assert np.array_equal(((s + 4) >> 3).astype(np.uint8), c.grid(l)), f"level {l}"
    # idempotence: a second full frame (sparse clear + re-voxelise) reproduces everything bit for bit
    c.frame(); c.sync()
    assert np.array_equal(c.counts(), counts) and np.array_equal(c.sums(), sums)
    assert np.array_equal(c.grid(0), g0) and np.array_equal(c.read_frame(), frame)
    # order independence: shuffled triangle order gives identical integer accumulators
    perm = np.random.default_rng(0).permutation(sc.n_tris)
    c.upload_mesh(sc.verts, sc.idx[perm], sc.tri_material[perm])
    c.draw_depth(); c.draw_voxels(); c.sync()
    assert np.array_equal(c.counts(), counts) and np.array_equal(c.sums(), sums)
    # triangle-range split (what each GPU does when voxelisation is sharded) == single pass
    k = sc.n_tris // 3
    c.voxelize_range(0, k, clear_first=True)
    c.voxelize_range(k, sc.n_tris, clear_first=False)
    c.resolve_and_mip(); c.sync()
    assert np.array_equal(c.counts(), counts) and np.array_equal(c.sums(), sums) and np.array_equal(c.grid(0), g0)
    # and back to the sparse path after a dense one
    c.draw_voxels(); c.sync()
    assert np.array_equal(c.counts(), counts) and np.array_equal(c.grid(0), g0)
    # host-buffer path returns the same frame
    c.upload_mesh(sc.verts, sc.idx, sc.tri_material)
    c.draw_depth()
    out = np.zeros_like(frame)
    c.frame(out)
    assert np.array_equal(out, frame)


def test_config2_full_size_vs_oracle(gpu_ctx, oracle, atrium_full):
    """The headline configuration itself (259 608 triangles, 256^3, 1920x1080, conservative coverage) against the
    oracle: shadow map, occupancy and fragment counts bit-exact; radiance and the frame within the north_star bar."""
    sc = atrium_full
    u = _cfg2(sc)
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    assert np.array_equal(gpu_ctx.depth(), oracle.depth())
    cg, co = gpu_ctx.counts(), oracle.counts()
    assert np.array_equal(cg, co) and cg.sum() > 1_500_000
    for l in range(9):
        g, o = gpu_ctx.grid(l), oracle.grid(l)
        assert np.array_equal(g[..., 3] > 0, o[..., 3] > 0)
        assert np.abs(g.astype(int) - o.astype(int)).max() <= LSB_TOL, f"level {l}"
    vis_g, vis_o = gpu_ctx.visibility(), oracle.visibility()
    assert (vis_g != vis_o).mean() <= 1e-4
    fg, fo = gpu_ctx.read_frame(), oracle.frame()
    assert psnr(fg[..., :3], fo[..., :3]) >= PSNR_MIN and frac_within(fg, fo, LSB_TOL) >= FRAC_MIN
    assert abs(gpu_ctx.cone_samples() - oracle.cone_samples()) <= 2e-4 * oracle.cone_samples()
    # pipelined frames (three streams, alternating slots) reproduce the same frame
    out = np.zeros_like(fg)
    for _ in range(3):
        gpu_ctx.frame()
    gpu_ctx.frame(out)
    assert np.array_equal(out, fg)


def test_dynamic_positions_round_trip(gpu_ctx):
    sc = scenes.dynamic_knot(nu=256, nv=128)
    u = uniforms.scene_uniforms(sc, V=128, width=320, height=180, shadow_map_size=1024, coverage="conservative")
    c = gpu_ctx
    run_gpu(c, sc, u)
    c0, g0 = c.counts(), c.grid(0)
    P1 = scenes.torus_knot_positions(256, 128, t=0.7).reshape(-1, 3) * 20.0
    c.update_positions(P1.astype(np.float32))
    c.draw_depth(); c.draw_voxels(); c.sync()
    c1 = c.counts()
    assert not np.array_equal(c1 > 0, c0 > 0)                       # the mesh really moved
    assert np.array_equal(c.grid(0)[..., 3] == 255, c1 > 0)         # stale voxels were cleared
    c.update_positions(sc.verts[:, :3])
    c.draw_depth(); c.draw_voxels(); c.sync()
    assert np.array_equal(c.counts(), c0) and np.array_equal(c.grid(0), g0)


def test_bounce_extension_vs_oracle(gpu_ctx, oracle):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=32, width=96, height=96, shadow_map_size=512, bounces=3)
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    g, o = gpu_ctx.grid(0), oracle.grid(0)
    assert np.array_equal(g[..., 3], o[..., 3])
    assert np.abs(g.astype(int) - o.astype(int)).max() <= LSB_TOL
    u2 = dict(u); u2["Bounces"] = 2
    oracle.set_uniforms(u2); oracle.draw_voxels()
    assert oracle.grid(0)[..., :3].astype(int).sum() < o[..., :3].astype(int).sum()   # the extra bounce adds light
    assert_frame_close(gpu_ctx.read_frame(), oracle_frame_with(oracle, u), "bounces=3", FRAC_MIN_SMALL)


def test_config5_light_probe_views_vs_oracle(gpu_ctx, oracle):
    """BASELINE config 5 in small: one voxelisation with Bounces = 3 (re-injection, extension), then several cameras of
    the 4x4x4 probe lattice -- arbitrary position, yaw and pitch inside the atrium -- rendered from that grid."""
    sc = scenes.atrium(detail=0.2, tex_size=64)
    cams = scenes.probe_cameras(64)
    assert len(cams) == 64 and len({c[0] for c in cams}) == 64
    base = dict(V=64, width=192, height=192, shadow_map_size=1024, coverage="conservative", bounces=3)
    u0 = uniforms.scene_uniforms(sc, **base)
    c = gpu_ctx
    c.set_uniforms(u0); c.load_scene(sc); c.draw_depth(); c.draw_voxels(); c.sync()
    oracle.set_uniforms(u0); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels()
    g, o = c.grid(0), oracle.grid(0)
    assert np.array_equal(g[..., 3], o[..., 3])
    assert np.abs(g.astype(int) - o.astype(int)).max() <= LSB_TOL
    for k in (5, 22, 47):
        pos, yaw, pitch = cams[k]
        u = uniforms.scene_uniforms(sc, camera_pos=pos, yaw=yaw, pitch=pitch, **base)
        c.set_uniforms(u); c.render(); c.sync()
        oracle.set_uniforms(u); oracle.render()
        assert_frame_close(c.read_frame(), oracle.frame(), f"probe {k}", FRAC_MIN_SMALL)
    assert np.array_equal(c.grid(0), g)          # rendering views does not touch the grid


def oracle_frame_with(oracle, u):
    oracle.set_uniforms(u)
    oracle.draw_voxels()
    oracle.render()
    return oracle.frame()


def test_runs_on_a_caller_stream_and_reports_pass_times(gpu_ctx):
    import torch
    s = torch.cuda.Stream()
    gpu_ctx.set_stream(s.cuda_stream)
    sc = scenes.cornell()
    run_gpu(gpu_ctx, sc, uniforms.scene_uniforms(sc, V=64, width=128, height=128, shadow_map_size=512))
    s.synchronize()
    for p in ("depth", "vox_cover", "vox_shade", "resolve", "mip", "visibility", "cone"):
        assert gpu_ctx.pass_time_us(p) > 0
    assert gpu_ctx.kernel_launches() > 10
    gpu_ctx.use_own_stream()


def test_pipelined_frames_equal_synchronous_frames(gpu_ctx):
    import torch
    import vct_b200.glmath as gm
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=160, height=96, shadow_map_size=512)
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.draw_depth()

    def cam(i):
        view = gm.view_matrix((2.0 * i, 0.0, 205.0), -90.0 + 1.5 * i, 0.0)
        c.set_mat4("ModelViewMatrix", gm.colmajor((view @ gm.scale(0.05)).astype(np.float32)))
        c.set_3f("CameraPosition", (2.0 * i, 0.0, 205.0))

    ref = []
    for i in range(5):
        cam(i)
        out = np.zeros((96, 160, 4), dtype=np.uint8)
        c.frame(out)
        ref.append(out)
    assert not np.array_equal(ref[0], ref[4])
    hosts = [torch.zeros((96, 160, 4), dtype=torch.uint8).pin_memory() for _ in range(5)]
    for i in range(5):
        cam(i)
        c.frame_async(hosts[i])
        if i >= 1:
            c.frame_wait()
            assert np.array_equal(hosts[i - 1].numpy(), ref[i - 1])      # frame i-1 is complete after the wait
    c.frame_wait()
    c.frame_wait()                                                       # idempotent when nothing is in flight
    for i in range(5):
        assert np.array_equal(hosts[i].numpy(), ref[i])


def test_cpp_facade_with_the_reference_class_surface_runs(gpu_ctx, oracle, tmp_path):
    """host/Voxel_Cone_Tracing.h (same struct / method names as the reference) driven by host/facade_demo.cpp.  The
    demo dumps its flattened scene, the uniforms of each frame and the frames; the same inputs replayed through the
    ctypes binding must give the same bytes, and the oracle the same frame within the bar."""
    import subprocess
    root = os.path.dirname(HERE)
    exe = os.path.join(root, "voxel-cone-tracing_b200", "lib", "facade_demo")
    if not os.path.exists(exe):
        import __graft_entry__
        __graft_entry__.build()
    out = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    sums = [int(l.split()[-1]) for l in out.stdout.splitlines() if l.startswith("frame")]
    assert len(sums) == 3 and all(s > 256 * 256 * 4 * 20 for s in sums) and len(set(sums)) == 3   # three different views
    rd = lambda name, dt: np.fromfile(os.path.join(str(tmp_path), name), dtype=dt)
    verts, idx, trimat = rd("verts.f32", np.float32).reshape(-1, 14), rd("idx.u32", np.uint32).reshape(-1, 3), rd("trimat.u16", np.uint16)
    tex = [np.full((1, 1, 3), c, np.uint8) for c in ((200, 200, 200), (200, 30, 30), (30, 200, 30))] + \
          [np.full((1, 1), 128, np.uint8), np.full((1, 1, 3), 128, np.uint8)]
    sc = scenes.Scene("facade", verts, idx, trimat, tex, [(0, 3, 4, 20.0), (1, 3, 4, 20.0), (2, 3, 4, 20.0)])
    names = ["ModelViewMatrix", "ProjectionMatrix", "DepthModelViewProjectionMatrix", "ProjX", "ProjY", "ProjZ"]
    for f in range(3):
        raw = rd(f"uniforms_{f}.f32", np.float32)
        u = uniforms.reference_uniforms(V=64, width=256, height=256, shadow_map_size=4096, coverage="msaa4")
        for k, name in enumerate(names):
            u[name] = raw[16 * k:16 * k + 16].copy()
        u["CameraPosition"] = raw[96:99].copy()
        want = rd(f"frame_{f}.rgba", np.uint8).reshape(256, 256, 4)
        run_gpu(gpu_ctx, sc, u)
        assert np.array_equal(gpu_ctx.read_frame(), want), f"frame {f}: C++ facade and ctypes binding disagree"
        assert int(want.astype(np.uint64).sum()) == sums[f]
        run_oracle(oracle, sc, u)
        assert_frame_close(want, oracle.frame(), f"facade frame {f} vs oracle")


def test_cpp_facade_renders_sharded_frames_over_two_ranks():
    """host/Voxel_Cone_Tracing.h: Voxel_Cone_Tracing_Sharded (vct_comm_init_multi / vct_frame_sharded_multi behind the
    reference's class surface) -- two ranks from one C++ host thread, frames byte-identical to the single-GPU ones."""
    import subprocess
    import tempfile
    import torch
    root = os.path.dirname(HERE)
    exe = os.path.join(root, "voxel-cone-tracing_b200", "lib", "facade_demo")
    second = 1 if torch.cuda.device_count() >= 2 else 0
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([exe, d, "sharded", str(second)], capture_output=True, text=True, timeout=180)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("identical") == 3 and "DIFFERENT" not in out.stdout, out.stdout


def test_tile_item_queue_overflow_is_detected_and_harmless(gpu_ctx):
    """MaxTileItems too small for the scene's large triangles: the pass must report VCT_ERR_OVERFLOW (not fault on the
    stale part of the queue) and the context must keep working once the queue is large enough."""
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=256, width=512, height=512, shadow_map_size=2048)
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc)
    c.draw_depth(); c.draw_voxels(); c.render(); c.sync()
    good_counts, good_frame = c.counts(), c.read_frame()
    assert c.debug_counter(0) > 0
    c.set_i("MaxTileItems", 1024)
    c.draw_depth()                                # 2048^2 shadow map: one wall triangle alone needs ~1024 items
    with pytest.raises(capi.VctError) as e:
        c.sync()
    assert e.value.code == -4
    c.draw_depth()
    out = np.zeros_like(good_frame)
    with pytest.raises(capi.VctError) as e:
        c.frame(out)                              # the synchronous host-buffer path reports the truncated pass too
    assert e.value.code == -4
    c.set_i("MaxTileItems", 4 << 20)
    c.draw_depth(); c.draw_voxels(); c.render(); c.sync()
    assert np.array_equal(c.counts(), good_counts) and np.array_equal(c.read_frame(), good_frame)


# ------------------------------------------------------------------------------------------ RGBA16F grid (config 3)
@pytest.mark.parametrize("V", [8, 32, 128])
def test_fp16_mip_pyramid_bit_exact(gpu_ctx, oracle, V):
    rng = np.random.default_rng(100 + V)
    g = (rng.random((V, V, V, 4)) * 4.0).astype(np.float16)
    g[rng.random((V, V, V)) < 0.7] = 0
    gpu_ctx.set_i("GridFormat", 1)
    gpu_ctx.set_i("VoxelDimensions", V)
    oracle.set_uniforms(uniforms.reference_uniforms(V=V, grid_format=1))
    gpu_ctx.upload_grid_level0(g)
    oracle.set_grid_level0(g)
    for l in range(V.bit_length()):
        a, b = gpu_ctx.grid(l), oracle.grid(l)
        assert a.dtype == np.float16 and np.array_equal(a.view(np.uint16), b.view(np.uint16)), f"V={V} level {l}"


def test_fp16_grid_cornell_vs_oracle(gpu_ctx, oracle):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=256, shadow_map_size=1024, coverage="conservative",
                                cones="9+1", grid_format=1)
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    assert np.array_equal(gpu_ctx.counts(), oracle.counts())
    for l in range(7):          # untextured scene: integer sums equal => half values and every mip level bit-exact
        assert np.array_equal(gpu_ctx.grid(l).view(np.uint16), oracle.grid(l).view(np.uint16)), f"level {l}"
    g0 = gpu_ctx.grid(0).astype(np.float32)
    assert set(np.unique(g0[..., 3])) == {0.0, 1.0} and g0[..., :3].max() <= 1.0
    assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), "fp16 grid, 9+1 cones")
    # the fp16 grid keeps what RGBA8 rounds away: same scene in RGBA8 differs slightly but stays close
    u8 = dict(u); u8["GridFormat"] = 0
    gpu_ctx.set_uniforms(u8); gpu_ctx.draw_voxels(); gpu_ctx.render(); gpu_ctx.sync()
    assert gpu_ctx.grid(0).dtype == np.uint8
    assert psnr(gpu_ctx.read_frame()[..., :3], oracle.frame()[..., :3]) > 40.0


def test_config3_shape_fp16_512_tiles(gpu_ctx):
    """BASELINE config 3 at reduced mesh detail: 512^3 RGBA16F grid, 3840x2160, 9 diffuse cones + specular, rendered
    as two row bands (what two ranks would do) and as one frame: identical pixels."""
    from vct_b200 import parallel
    sc = scenes.atrium(detail=0.25, tex_size=64)
    u = uniforms.scene_uniforms(sc, V=512, width=3840, height=2160, shadow_map_size=4096, coverage="conservative",
                                cones="9+1", grid_format=1)
    c = gpu_ctx
    run_gpu(c, sc, u)
    full = c.read_frame()
    cnt = c.counts()
    assert cnt.sum() > 1_000_000 and c.grid(0).dtype == np.float16
    g1 = c.grid(1).astype(np.float32)
    assert np.isfinite(g1).all() and g1[..., 3].max() <= 1.0
    bands = []
    for r in range(2):
        b0, b1 = parallel.row_band(2160, r, 2)
        c.set_i("RowBegin", b0); c.set_i("RowEnd", b1)
        c.render(); c.sync()
        bands.append(c.read_frame()[b0:b1])
    c.set_i("RowBegin", 0); c.set_i("RowEnd", 0)
    assert np.array_equal(np.concatenate(bands, 0), full)
    assert c.cone_samples() > 0


def test_fp16_bounce_extension_vs_oracle(gpu_ctx, oracle):
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=32, width=96, height=96, shadow_map_size=512, bounces=3, grid_format=1)
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    g, o = gpu_ctx.grid(0).astype(np.float32), oracle.grid(0).astype(np.float32)
    assert np.array_equal(g[..., 3], o[..., 3])
    assert np.abs(g - o).max() <= 2.0 / 255
    assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), "fp16 bounces=3", FRAC_MIN_SMALL)


# ------------------------------------------------------------------------------------------ fused sharded voxelisation
def test_shared_accumulator_path_single_rank(gpu_ctx):
    """In-switch-reduction flavour of vct_voxelize_shared / vct_resolve_shared with a one-rank accumulator (plain atomics
    + occupancy mask): identical to vct_draw_voxels, also across frames, a moving mesh and a switch back to the private
    path."""
    import torch
    from vct_b200 import parallel
    sc = scenes.dynamic_knot(nu=256, nv=128)
    u = uniforms.scene_uniforms(sc, V=128, width=320, height=180, shadow_map_size=1024, coverage="conservative")
    c = gpu_ctx
    run_gpu(c, sc, u)
    g_ref = [c.grid(l) for l in range(8)]
    shared = parallel.SharedAccumulator(c, rank=0, world=1, session="t_reduce1", exchange="reduce")
    n = sc.n_tris
    for it in range(3):
        c.voxelize_shared(0, n // 2)          # two ranges into the same accumulator = what two ranks would add
        c.voxelize_shared(n // 2, n)
        c.resolve_shared(); c.sync()
        for l in range(8):
            assert np.array_equal(c.grid(l), g_ref[l]), (it, l)
    P1 = scenes.torus_knot_positions(256, 128, t=0.9).reshape(-1, 3) * 20.0
    c.update_positions(P1.astype(np.float32)); c.draw_depth()
    c.voxelize_shared(0, n); c.resolve_shared(); c.sync()
    moved = c.grid(0)
    c.draw_voxels(); c.sync()                  # private path on the same mesh
    assert np.array_equal(c.grid(0), moved) and not np.array_equal(moved, g_ref[0])
    c.update_positions(sc.verts[:, :3]); c.draw_depth()
    c.voxelize_shared(0, n); c.resolve_shared(); c.sync()
    assert np.array_equal(c.grid(0), g_ref[0]) and np.array_equal(c.grid(3), g_ref[3])     # stale voxels removed
    shared.close()


@pytest.mark.parametrize("grid_format,bounces", [(0, 2), (1, 2), (0, 3)])
def test_sparse_mip_build_tracks_a_moving_mesh(gpu_ctx, grid_format, bounces):
    """The pyramid is rebuilt only above level-0 bricks that changed (dirty flags set by the sparse clear and resolve).
    Over frames of a moving mesh -- both frame slots, stale voxels disappearing, switches to the dense path and back --
    every level must equal what the dense build (DenseResolve=1: dense clear, resolve and mip) produces."""
    sc = scenes.dynamic_knot(nu=192, nv=96)
    u = uniforms.scene_uniforms(sc, V=128, width=64, height=64, shadow_map_size=1024, coverage="conservative",
                                grid_format=grid_format)
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc); c.set_i("Bounces", bounces)
    levels = 8
    for frame in range(7):
        P = scenes.torus_knot_positions(192, 96, t=0.35 * frame).reshape(-1, 3) * 20.0
        c.update_positions(P.astype(np.float32)); c.draw_depth()
        c.set_i("DenseResolve", 0)
        c.draw_voxels(); c.sync()
        sparse = [c.grid(l) for l in range(levels)]
        if frame in (0, 1, 3, 6):              # the dense build of the same frame (also leaves a densely written slot behind)
            c.set_i("DenseResolve", 1)
            c.draw_voxels(); c.sync()
            for l in range(levels):
                assert np.array_equal(c.grid(l), sparse[l]), (frame, l)
        assert (sparse[0][..., 3] > 0).sum() > 1000 and sparse[levels - 1].max() > 0


def test_interleaved_triangle_shares_sum_to_the_whole(gpu_ctx):
    """TriangleInterleave / TrianglePhase: the three interleaved shares of a mesh, accumulated, give exactly the
    accumulator (counts and sums) of one full voxelisation."""
    sc = scenes.atrium(detail=0.25, tex_size=64)
    u = uniforms.scene_uniforms(sc, V=128, width=64, height=64, shadow_map_size=1024, coverage="conservative")
    c = gpu_ctx
    run_gpu(c, sc, u)
    counts, sums, g_ref = c.counts(), c.sums(), [c.grid(l) for l in range(8)]
    n = sc.n_tris
    c.set_i("TriangleInterleave", 3)
    total = 0
    for phase in range(3):
        c.set_i("TrianglePhase", phase)
        c.voxelize_range(0, n, clear_first=(phase == 0))
        c.sync(); total += c.fragment_count()
        assert c.fragment_count() > 0
    c.set_i("TriangleInterleave", 1); c.set_i("TrianglePhase", 0)
    assert np.array_equal(c.counts(), counts) and np.array_equal(c.sums(), sums)
    assert total >= int(counts.sum())        # queued fragments (those outside the slice range are dropped when shaded)
    c.resolve_and_mip(); c.sync()
    for l in range(8):
        assert np.array_equal(c.grid(l), g_ref[l]), l


def test_inbox_exchange_two_contexts_one_gpu(gpu_ctx):
    """Inbox flavour (default): two handles on ONE device act as ranks 0 and 1 of a world of two and share one exchange
    buffer (no multicast mapping -> plain stores).  After push / merge both hold the single-GPU grid bit for bit, over
    several frames, with a moving mesh, after a switch to the private path and back, and an undersized inbox is
    reported as an overflow."""
    import torch
    sc = scenes.dynamic_knot(nu=256, nv=128)
    u = uniforms.scene_uniforms(sc, V=128, width=320, height=180, shadow_map_size=1024, coverage="conservative")
    a = gpu_ctx
    run_gpu(a, sc, u)
    g_ref = [a.grid(l) for l in range(8)]
    b = capi.Context(0)
    b.set_uniforms(u); b.load_scene(sc); b.draw_depth(); b.sync()
    for rank, c in enumerate((a, b)):
        c.set_i("SharedExchange", 0); c.set_i("SharedWorld", 2); c.set_i("SharedRank", rank)
    nbytes = a.shared_accum_bytes()
    assert nbytes == b.shared_accum_bytes()
    buf = torch.zeros((nbytes + 7) // 8, dtype=torch.int64, device="cuda:0")
    a.set_shared_accum(buf.data_ptr(), 0); b.set_shared_accum(buf.data_ptr(), 0)
    n = sc.n_tris
    cut = n // 3                                  # unequal shares

    def exchange(interleaved=False):
        for rank, c in enumerate((a, b)):         # contiguous unequal ranges, or blocks of 128 triangles dealt in turn
            c.set_i("TriangleInterleave", 2 if interleaved else 1); c.set_i("TrianglePhase", rank if interleaved else 0)
        if interleaved:
            a.voxelize_shared(0, n); b.voxelize_shared(0, n)
        else:
            a.voxelize_shared(0, cut); b.voxelize_shared(cut, n)
        a.sync(); b.sync()                        # the cross-rank barrier
        a.resolve_shared(); b.resolve_shared()
        a.sync(); b.sync()
        for c in (a, b):
            c.set_i("TriangleInterleave", 1); c.set_i("TrianglePhase", 0)

    for it in range(4):
        exchange(interleaved=it >= 2)
        for l in range(8):
            assert np.array_equal(a.grid(l), g_ref[l]), (it, l)
            assert np.array_equal(b.grid(l), g_ref[l]), (it, l)
    assert a.occupied_voxels() == int((g_ref[0][..., 3] > 0).sum())
    P1 = scenes.torus_knot_positions(256, 128, t=0.9).reshape(-1, 3) * 20.0
    for c in (a, b):
        c.update_positions(P1.astype(np.float32)); c.draw_depth()
    exchange()
    moved = a.grid(0)
    assert np.array_equal(b.grid(0), moved)
    a.draw_voxels(); a.sync()                     # private path on the same mesh
    assert np.array_equal(a.grid(0), moved) and not np.array_equal(moved, g_ref[0])
    for c in (a, b):
        c.update_positions(sc.verts[:, :3]); c.draw_depth()
    exchange()
    for c in (a, b):
        assert np.array_equal(c.grid(0), g_ref[0]) and np.array_equal(c.grid(3), g_ref[3])   # stale voxels removed
    # frames rendered from the merged grid equal the single-GPU frame
    a.draw_voxels(); a.render(); a.sync(); f_ref = a.read_frame()
    exchange(interleaved=True); b.render(); b.sync()
    assert np.array_equal(b.read_frame(), f_ref)
    # an inbox smaller than the touched set is an error, not a silent truncation
    for c in (a, b):
        c.set_i("MaxExchangeVoxels", 1024)
    small = torch.zeros((a.shared_accum_bytes() + 7) // 8, dtype=torch.int64, device="cuda:0")
    a.set_shared_accum(small.data_ptr(), 0); b.set_shared_accum(small.data_ptr(), 0)
    a.voxelize_shared(0, cut); b.voxelize_shared(cut, n); a.sync(); b.sync()
    a.resolve_shared()
    with pytest.raises(capi.VctError):
        a.sync()
    b.close()


def test_pipelined_shared_frames_match_plain_frames(gpu_ctx):
    """vct_frame_shared_begin / _end (the pipelined sharded frame) with a world of one, and with two handles acting as
    two ranks on one device: frames and grids equal those of the plain path while the mesh and the camera move."""
    import torch
    import vct_b200.glmath as gm
    from vct_b200 import parallel
    sc = scenes.dynamic_knot(nu=192, nv=96)
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=144, shadow_map_size=1024, coverage="conservative")
    a = gpu_ctx
    a.set_uniforms(u); a.load_scene(sc)
    b = capi.Context(0)
    b.set_uniforms(u); b.load_scene(sc)
    n = sc.n_tris

    def inputs(c, i):
        if i % 2 == 0:      # the mesh moves every other frame (ordered path); the camera every frame (pipelined path)
            P = scenes.torus_knot_positions(192, 96, t=0.4 * i).reshape(-1, 3) * 20.0
            c.update_positions(P.astype(np.float32)); c.draw_depth()
        view = gm.view_matrix(sc.camera_pos, sc.yaw + 3.0 * i, sc.pitch)
        c.set_mat4("ModelViewMatrix", gm.colmajor((view @ gm.scale(0.05)).astype(np.float32)))

    a.set_i("PipelineFrames", 0); a.set_i("OverlapVisibility", 0)
    ref = []
    for i in range(6):
        inputs(a, i); a.frame(); a.sync()
        ref.append((a.read_frame(), a.grid(0), a.grid(2)))
    a.set_i("PipelineFrames", 1); a.set_i("OverlapVisibility", 1)
    # (1) a world of one through the library's own multi-GPU layer (vct_comm_init / vct_frame_sharded)
    shared = parallel.SharedAccumulator(a, rank=0, world=1, session="t_pipe1")
    host = np.zeros_like(ref[0][0])
    for i in range(6):
        inputs(a, i); shared.frame(host); shared.wait()
        assert np.array_equal(host, ref[i][0]) and np.array_equal(a.read_frame(), ref[i][0]), i
        assert np.array_equal(a.grid(0), ref[i][1]) and np.array_equal(a.grid(2), ref[i][2]), i
    with pytest.raises(capi.VctError):
        a.frame_shared_end()                         # nothing begun
    with pytest.raises(capi.VctError):
        a.set_shared_accum(0, 0)                     # the exchange buffer belongs to the library now
    shared.close()
    # (2) two handles = two ranks sharing one inbox; the device-wide synchronize stands in for the cross-rank barrier
    b.set_i("PipelineFrames", 1)
    for rank, c in enumerate((a, b)):
        c.set_i("SharedWorld", 2); c.set_i("SharedRank", rank)
        c.set_i("TriangleInterleave", 2); c.set_i("TrianglePhase", rank)
    buf = torch.zeros((a.shared_accum_bytes() + 7) // 8, dtype=torch.int64, device="cuda:0")
    a.set_shared_accum(buf.data_ptr(), 0); b.set_shared_accum(buf.data_ptr(), 0)
    for i in range(6):
        inputs(a, i); inputs(b, i)
        a.frame_shared_begin(0, n); b.frame_shared_begin(0, n)
        torch.cuda.synchronize()
        a.frame_shared_end(); b.frame_shared_end()
        a.sync(); b.sync()
        for c in (a, b):
            assert np.array_equal(c.read_frame(), ref[i][0]), i
            assert np.array_equal(c.grid(0), ref[i][1]) and np.array_equal(c.grid(2), ref[i][2]), i
    b.close()


def _run_ranks(world, devices, extra=(), timeout=600):
    """Launches `world` processes of tests/mgpu_comm_worker.py (plain subprocesses: the library does its own bootstrap)."""
    import subprocess
    import sys
    import uuid
    root = os.path.dirname(HERE)
    session = "t_" + uuid.uuid4().hex[:12]
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "mgpu_comm_worker.py"), str(r), str(world), session,
                               str(devices[r]), *extra], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=root)
             for r in range(world)]
    outs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            p.kill(); o, _ = p.communicate()
        outs.append(o)
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"MGPU_COMM_OK {r}" in o, f"rank {r} rc={p.returncode}\n" + o[-3000:]
    return outs


def test_loaded_obj_asset_vs_oracle(gpu_ctx, oracle, tmp_path):
    """The real-asset path (SURVEY 8f rank 2): an OBJ + MTL + PNG / TGA textures on disk -> objloader (assimp's
    post-processing restated, textures decoded by images.py) -> the device, against the oracle on the same loaded scene.
    The asset has a noise albedo, a height map, a cut-out (alpha) quad in front of a wall and a quad without normals."""
    from vct_b200 import images, objloader
    rng = np.random.default_rng(11)
    d = str(tmp_path)
    images.save_png(rng.integers(60, 230, (64, 64, 3), dtype=np.uint8), os.path.join(d, "albedo.png"))
    images.save_png((scenes.value_noise(64, 4, rng) * 255).astype(np.uint8), os.path.join(d, "height.png"))
    cut = np.zeros((32, 32, 4), np.uint8); cut[..., :3] = (40, 200, 60); cut[8:24, 8:24, 3] = 255     # opaque square in the middle
    images.save_png(cut, os.path.join(d, "cutout.png"))
    open(os.path.join(d, "room.mtl"), "w").write(
        "newmtl wall\nKd 0.7 0.7 0.7\nKs 0.2 0.2 0.2\nmap_Kd albedo.png\nmap_Ka height.png\n"
        "newmtl leaf\nKd 0.2 0.8 0.3\nKs 0 0 0\nmap_Kd cutout.png\nnewmtl plain\nKd 0.8 0.3 0.2\nKs 0.4 0.4 0.4\n")
    S = 1100.0      # model units (ModelMatrix = scale(0.05): +-55 world)
    v = [(-S, -S, -S), (S, -S, -S), (S, S, -S), (-S, S, -S), (-S, -S, S), (S, -S, S), (S, S, S), (-S, S, S),
         (-400, -400, -300), (400, -400, -300), (400, 400, -300), (-400, 400, -300)]
    with open(os.path.join(d, "room.obj"), "w") as f:
        f.write("mtllib room.mtl\n" + "".join("v %g %g %g\n" % p for p in v) + "vt 0 0\nvt 3 0\nvt 3 3\nvt 0 3\nvt 1 0\nvt 1 1\nvt 0 1\n")
        f.write("usemtl wall\nf 1/1 2/2 3/3 4/4\nf 1/1 5/2 6/3 2/4\nf 1/1 4/2 8/3 5/4\nf 2/1 6/2 7/3 3/4\n")       # back, floor, left, right
        f.write("usemtl plain\nf 4/1 3/2 7/3 8/4\n")                                                                 # ceiling
        f.write("usemtl leaf\nf 9/1 10/5 11/6 12/7\n")                                                               # cut-out card
    sc = objloader.load_obj(os.path.join(d, "room.obj"))
    assert sc.n_tris == 12 and sc.textures[sc.materials[2][0]].shape == (32, 32, 4)     # wall, plain, leaf
    u = uniforms.reference_uniforms(V=64, width=320, height=240, shadow_map_size=1024, camera_pos=(0.0, 0.0, 52.0), coverage="msaa4")
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    assert np.array_equal(gpu_ctx.depth(), oracle.depth())
    assert np.array_equal(gpu_ctx.counts(), oracle.counts()) and gpu_ctx.counts().sum() > 5000
    vg, vo = gpu_ctx.visibility(), oracle.visibility()
    assert (vg != vo).mean() <= 1e-3
    card = np.isin(vo, [10, 11])
    assert card.any() and (vo[120, 160] in (10, 11)) and not np.isin(vo[120, 60], [10, 11])      # alpha discard: only the middle of the card
    assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), "loaded OBJ asset", FRAC_MIN_SMALL)


def test_library_comm_three_ranks_one_gpu():
    """Three processes on device 0: more than one remote rank, i.e. the single-launch atomic merge (vox_merge_inbox_all)."""
    _run_ranks(3, [0, 0, 0], extra=("nomc",))


def test_library_comm_two_processes_one_gpu():
    """The library's own bootstrap (handle exchange over a unix socket, peer mapping, device barrier, frame gather into
    rank 0, asynchronous host ring) with two PROCESSES acting as two ranks on device 0: no multicast object (one device
    cannot join a team twice), so the records travel as peer stores (vox_push_inbox<2>)."""
    _run_ranks(2, [0, 0], extra=("nomc",))
    _run_ranks(2, [0, 0], extra=("nomc", "bands", "shadow"))


@pytest.mark.parametrize("extra", [(), ("nomc",), ("reduce",), ("bands",), ("shadow",), ("shadow", "nomc")])
def test_library_comm_two_gpus(extra):
    """Two processes on two GPUs: multimem.st inbox through the library's multicast mapping, the same without a multicast
    object, and the multimem.red flavour.  Needs two GPUs on the box (skipped otherwise)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    outs = _run_ranks(2, [0, 1], extra=extra)
    if "nomc" not in extra:
        assert "multicast=True" in outs[0]


def test_one_process_driving_several_devices(gpu_ctx):
    """vct_create_multi / vct_comm_init_multi / vct_frame_sharded_multi: one host thread, n handles.  On a one-GPU box the
    two handles share device 0 (peer stores instead of multicast); with two GPUs the multicast path runs."""
    import torch
    import vct_b200.glmath as gm
    devices = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    sc = scenes.atrium(detail=0.25, tex_size=64)
    H, W = 288, 512
    u = uniforms.scene_uniforms(sc, V=128, width=W, height=H, shadow_map_size=2048, coverage="conservative")

    def camera(c, i):
        view = gm.view_matrix(sc.camera_pos, sc.yaw + 5.0 * i, sc.pitch)
        c.set_mat4("ModelViewMatrix", gm.colmajor((view @ gm.scale(0.05)).astype(np.float32)))

    ref = []
    gpu_ctx.set_uniforms(u); gpu_ctx.load_scene(sc); gpu_ctx.draw_depth()
    for i in range(4):
        camera(gpu_ctx, i); gpu_ctx.frame(); gpu_ctx.sync()
        ref.append(gpu_ctx.read_frame())
    ref_grid = [gpu_ctx.grid(l) for l in range(8)]
    m = capi.MultiContext(devices)
    for c in m.ctx:
        c.set_uniforms(u); c.load_scene(sc); c.draw_depth()
    m.comm_init()
    assert m.ctx[0].comm_info()["multicast"] == (devices[0] != devices[1])
    assert m.ctx[1].get_i("RowInterleave") == 2 and m.ctx[1].get_i("RowPhase") == 1      # rows dealt in strips of 8
    hosts = [np.zeros((H, W, 4), np.uint8) for _ in range(4)]
    for i in range(4):
        for c in m.ctx:
            camera(c, i)
        m.frame_sharded(hosts[i])
    m.wait()
    for i in range(4):
        assert np.array_equal(hosts[i], ref[i]), f"frame {i}"
    for c in m.ctx:
        for l in range(8):
            assert np.array_equal(c.grid(l), ref_grid[l]), l
    m.close()


def test_pipelined_frames_with_a_moving_mesh_and_camera(gpu_ctx):
    """vct_frame overlaps frame i+1's voxel / visibility stages with frame i's cone_trace; device-side input changes
    (positions, shadow map) between frames must still be honoured.  Compare against the unpipelined, unoverlapped path."""
    import vct_b200.glmath as gm
    sc = scenes.dynamic_knot(nu=192, nv=96)
    u = uniforms.scene_uniforms(sc, V=64, width=256, height=144, shadow_map_size=1024, coverage="conservative")
    c = gpu_ctx
    c.set_uniforms(u); c.load_scene(sc)

    def run(pipe, overlap):
        c.set_i("PipelineFrames", pipe); c.set_i("OverlapVisibility", overlap)
        frames, grids = [], []
        for i in range(6):
            if i % 2 == 0:      # the mesh moves every other frame; the camera every frame
                P = scenes.torus_knot_positions(192, 96, t=0.4 * i).reshape(-1, 3) * 20.0
                c.update_positions(P.astype(np.float32)); c.draw_depth()
            view = gm.view_matrix(sc.camera_pos, sc.yaw + 3.0 * i, sc.pitch)
            c.set_mat4("ModelViewMatrix", gm.colmajor((view @ gm.scale(0.05)).astype(np.float32)))
            c.frame()
            if i in (1, 3, 5):
                c.sync(); frames.append(c.read_frame()); grids.append(c.grid(0))
            else:
                c.frame()       # a second frame with unchanged device inputs: this one pipelines
        c.sync()
        return frames, grids

    fa, ga = run(0, 0)
    fb, gb = run(1, 1)
    for k in range(3):
        assert np.array_equal(fa[k], fb[k]) and np.array_equal(ga[k], gb[k]), k
    assert not np.array_equal(ga[0], ga[2])
    assert c.counts().sum() == c.fragment_count()


@pytest.mark.parametrize("cones", ["6+1", "9+1"])
def test_cone_trace_shapes_vs_oracle(gpu_ctx, oracle, cones):
    """The cone_trace shapes launched for 6 and for 9 diffuse cones (one template instantiation each) render the
    oracle's frame."""
    sc = scenes.atrium(detail=0.3, tex_size=64)
    u = uniforms.scene_uniforms(sc, V=128, width=640, height=360, shadow_map_size=2048, coverage="conservative", cones=cones)
    c = gpu_ctx
    run_gpu(c, sc, u)
    run_oracle(oracle, sc, u)
    assert_frame_close(c.read_frame(), oracle.frame(), f"default cone_trace, {cones}", FRAC_MIN_SMALL)
