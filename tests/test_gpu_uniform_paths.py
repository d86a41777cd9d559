"""GPU tests of the kernel paths that only non-default uniforms reach (run with -m gpu on a B200): the cone_trace shape
for 10-16 diffuse cones (cone_trace<16, 2, 8>), the generic PCF loop (every PcfRadius but 2), the unaligned
depth_to_array path and clamped tex2Dgather edges of small or odd shadow maps, the march limits StepMultiplier,
MaxDistance and MaxAlpha, n_cones = 0, and frames whose sizes are not multiples of the 8x8 cone_trace block.

Exact checks come first and do not depend on the oracle's filter model:
  * zero-weight cones appended to a table leave the frame byte-identical whichever cone_trace shape runs it
    (fmaf(0, s, acc) == acc for finite s; the real cones keep their shared distance sequence; the specular chain
    composites the same fetches in the same order whatever the fetch-ahead depth SU), and duplicates of a cone add
    exactly its step count per pixel to vct_cone_samples -- which proves every cone slot up to 15 was marched;
  * on a uniform grid every cone's step count has a closed form (test_uniform_paths.uniform_steps), so
    vct_cone_samples must equal covered pixels * (n * k_d + k_s) exactly;
  * voxelisation of the untextured Cornell box is integer arithmetic, so the shadow map, the accumulators and the
    pyramid must equal the oracle's bit for bit at any PcfRadius and ShadowMapSize.
Frames against the oracle keep the bars of test_gpu_parity.py.
"""
import numpy as np
import pytest

from conftest import frac_within, psnr
from test_gpu_parity import FRAC_MIN_SMALL, assert_frame_close, run_gpu, run_oracle
from test_uniform_paths import LIMITS, UNIFORM_ALPHAS, limit_uniforms, uniform_steps
from vct_b200 import scenes, uniforms

pytestmark = pytest.mark.gpu

MISS = 0xFFFFFFFF
FLIP_LSB = 5          # DESIGN.md section 2: one cone step added or dropped at the alpha threshold moves a pixel <= 5/255


def ring_table(n, w_normal=0.1):
    """n diffuse cones: the normal plus n - 1 at 60 degrees, the remaining weight shared equally (n = 0: no cone)"""
    if n == 0:
        return np.zeros((0, 3), np.float32), np.zeros(0, np.float32)
    a = np.arange(n - 1) * (2 * np.pi / max(n - 1, 1))
    d = np.concatenate([[[0, 0, 1]], np.stack([0.866025 * np.cos(a), 0.866025 * np.sin(a), np.full(n - 1, 0.5)], 1)])
    w = np.concatenate([[w_normal if n > 1 else 1.0], np.full(n - 1, (1 - w_normal) / max(n - 1, 1))])
    return d.astype(np.float32), w.astype(np.float32)


def padded(dirs, wts, pad_dirs, rng):
    """the table with zero-weight cones along pad_dirs inserted at random places; the real cones keep their order"""
    n = len(dirs) + len(pad_dirs)
    real_at = np.sort(rng.choice(n, len(dirs), replace=False))
    d = np.empty((n, 3), np.float32); w = np.zeros(n, np.float32)
    pad_at = np.setdiff1d(np.arange(n), real_at)
    d[real_at], w[real_at] = dirs, wts
    d[pad_at] = pad_dirs
    return d, w


def other_directions(k):
    """k unit directions at 40 degrees from the normal, none of them in a cone table used here"""
    a = np.arange(k) * (2 * np.pi / max(k, 1)) + 0.3
    return np.stack([np.sin(0.7) * np.cos(a), np.sin(0.7) * np.sin(a), np.full(k, np.cos(0.7))], 1).astype(np.float32)


def render(c, dirs, wts):
    c.set_cones(dirs, wts)
    c.render()
    c.sync()
    return c.read_frame(), c.cone_samples()


# --------------------------------------------------------------------------------- exact: zero-weight padding
PADDING_CASES = {
    "cornell 128x128": dict(V=64, width=128, height=128, shadow_map_size=512),
    "cornell 128x128 rgba16f": dict(V=64, width=128, height=128, shadow_map_size=512, grid_format=1),
    "cornell config 1": dict(V=64, width=256, height=256, shadow_map_size=1024, coverage="msaa4"),
}


@pytest.mark.parametrize("case", sorted(PADDING_CASES))
def test_zero_weight_padding_renders_identical_frames_in_every_shape(gpu_ctx, case):
    """The reference's six cones padded to 7, 9, 10 and 16 (cone_trace<6,4,10>, <9,4,8> and <16,2,8>) render the
    six-cone frame byte for byte; one cone of weight 1 padded with 1..15 zero-weight copies of itself renders the
    one-cone frame, and each copy adds exactly the one cone's steps to vct_cone_samples."""
    sc = scenes.cornell()
    c = gpu_ctx
    run_gpu(c, sc, uniforms.scene_uniforms(sc, **PADDING_CASES[case]))
    rng = np.random.default_rng(7)
    d6, w6 = uniforms.cone_set("6+1")
    ref6, s6 = render(c, d6, w6)
    for n in (7, 9, 10, 16):
        d, w = padded(d6, w6, other_directions(n - 6), rng)
        frame, samples = render(c, d, w)
        assert np.array_equal(frame, ref6), f"{case}: 6 cones padded to {n}"
        assert samples > s6
    one_d, one_w = np.array([[0, 0, 1]], np.float32), np.ones(1, np.float32)
    ref1, s1 = render(c, one_d, one_w)
    assert not np.array_equal(ref1, ref6)
    steps = []
    for k in range(1, 16):
        d = np.repeat(one_d, k + 1, 0)
        w = np.zeros(k + 1, np.float32); w[k // 2] = 1.0      # the weighted copy moves through the table
        frame, samples = render(c, d, w)
        assert np.array_equal(frame, ref1), f"{case}: one cone + {k} zero-weight copies"
        steps.append(samples - s1)
    per_copy = steps[0]
    assert per_copy > 0 and steps == [k * per_copy for k in range(1, 16)], (per_copy, steps)


def test_zero_weight_padding_bakes_identical_probes(gpu_ctx):
    """vct_bake_probes with the same padded tables: outputs bit-identical, steps linear in the number of copies."""
    sc = scenes.cornell()
    c = gpu_ctx
    run_gpu(c, sc, uniforms.scene_uniforms(sc, V=64, width=64, height=64, shadow_map_size=512))
    g = np.linspace(-45, 45, 4, dtype=np.float32)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(11)
    d6, w6 = uniforms.cone_set("6+1")
    c.set_cones(d6, w6)
    ref6, st6 = c.bake_probes(xyz)
    assert np.isfinite(ref6).all() and (st6 > 0).all()
    for n in (7, 10, 16):
        c.set_cones(*padded(d6, w6, other_directions(n - 6), rng))
        out, st = c.bake_probes(xyz)
        assert np.array_equal(out.view(np.uint32), ref6.view(np.uint32)), n
        assert (st > st6).all()
    one_d = np.array([[0, 0, 1]], np.float32)
    c.set_cones(one_d, np.ones(1, np.float32))
    ref1, st1 = c.bake_probes(xyz)
    for k in range(1, 16):
        w = np.zeros(k + 1, np.float32); w[(3 * k) % (k + 1)] = 1.0
        c.set_cones(np.repeat(one_d, k + 1, 0), w)
        out, st = c.bake_probes(xyz)
        assert np.array_equal(out.view(np.uint32), ref1.view(np.uint32)), k
        assert np.array_equal(st.astype(np.int64), (k + 1) * st1.astype(np.int64)), k


# --------------------------------------------------------------------------------- exact: uniform-grid step counts
CONE_COUNTS = (0, 1, 6, 9, 16)


def test_uniform_grid_step_counts_in_the_frame(gpu_ctx):
    """A voxelised Cornell box whose level 0 is then replaced by a uniform grid (rgb 153, alpha A): under every march
    limit of test_uniform_paths.LIMITS and with 0, 1, 6, 9 and 16 diffuse cones, vct_cone_samples is exactly
    covered pixels * (n * k_d + k_s), and vct_trace_cones gives k_d and k_s per cone."""
    V = 64
    sc = scenes.cornell()
    base = uniforms.scene_uniforms(sc, V=V, width=120, height=100, shadow_map_size=512)
    c = gpu_ctx
    run_gpu(c, sc, base)
    vis = c.visibility()
    covered = int((vis != MISS).sum())
    assert covered > 0.5 * vis.size
    rng = np.random.default_rng(5)
    starts = rng.uniform(-70, 70, (64, 3)).astype(np.float32)
    dirs = rng.normal(size=(64, 3)); dirs = (dirs / np.linalg.norm(dirs, axis=1, keepdims=True)).astype(np.float32)
    tans = np.where(np.arange(64) % 2 == 0, base["DiffuseTanHalfAngle"], base["SpecularTanHalfAngle"]).astype(np.float32)
    checked = 0
    for alpha8 in UNIFORM_ALPHAS:
        g = np.empty((V, V, V, 4), np.uint8); g[..., :3] = 153; g[..., 3] = alpha8
        c.upload_grid_level0(g)                  # a render after an uploaded level 0 traces that grid
        for name, value in [(None, None)] + LIMITS:
            u = limit_uniforms(base, name, value)
            for k in ("StepMultiplier", "MaxDistance", "MaxAlpha"):
                c.set_f(k, u[k])
            want = uniform_steps(V, alpha8, u)
            if want is None:
                continue                         # a step sits within KAT_MARGIN of a limit
            kd, ks = want
            _, steps = c.trace_cones(starts, dirs, tans)
            assert np.array_equal(steps, np.where(np.arange(64) % 2 == 0, kd, ks)), (alpha8, name, value)
            for n in CONE_COUNTS:
                _, samples = render(c, *ring_table(n))
                assert samples == covered * (n * kd + ks), (alpha8, name, value, n, samples, covered, kd, ks)
                checked += 1
    assert checked >= 90, checked
    assert np.array_equal(c.visibility(), vis)


# --------------------------------------------------------------------------------- exact: voxelisation
VOX_CASES = [(r, 1024) for r in (0, 1, 3, 8)] + [(2, S) for S in (1, 2, 3, 5, 257, 1023)]


@pytest.mark.parametrize("coverage", ["center", "msaa4"])
@pytest.mark.parametrize("r,S", VOX_CASES)
def test_voxelisation_bit_exact_at_any_pcf_radius_and_map_size(gpu_ctx, oracle, r, S, coverage):
    """Cornell has 1x1 textures, so every fragment's value is an exact function of its lit-tap count: the shadow map,
    counts, sums and every level of the pyramid equal the oracle's.  Radius 2 runs the tex2Dgather path on the array
    copy that depth_to_array writes (four texels per thread; a map whose size is not a multiple of 4 takes the
    per-texel path), every other radius the generic loop."""
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=64, height=64, shadow_map_size=S, coverage=coverage)
    u["PcfRadius"] = r
    for x in (gpu_ctx, oracle):
        x.set_uniforms(u); x.load_scene(sc); x.draw_depth(); x.draw_voxels()
    gpu_ctx.sync()
    assert np.array_equal(gpu_ctx.depth(), oracle.depth())
    assert np.array_equal(gpu_ctx.counts(), oracle.counts())
    assert np.array_equal(gpu_ctx.sums(), oracle.sums())
    for l in range(7):
        assert np.array_equal(gpu_ctx.grid(l), oracle.grid(l)), f"level {l}"
    assert oracle.counts().sum() > 10_000


# --------------------------------------------------------------------------------- frames against the oracle
@pytest.fixture(scope="module")
def frame_scenes():
    """scene, size, and the bar on the relative difference of vct_cone_samples.  Every flip of a cone exit at the alpha
    threshold adds or drops one sample, and on the 128x128 Cornell frame about 120 cones sit that close: there the
    oracle's own two filter models (FilterMode 0 and 1) differ by 1.7e-4 at the reference's limits (up to 7e-4 with
    MaxAlpha = 0.5), so the 1e-4 of the larger frames is below what the filter model resolves and that frame takes 2e-4,
    the bar of test_gpu_parity.test_config2_full_size_vs_oracle."""
    return {"cornell": (scenes.cornell(), dict(V=64, width=128, height=128, shadow_map_size=1024), 2e-4),
            "atrium": (scenes.atrium(detail=0.3, tex_size=64),
                       dict(V=128, width=640, height=360, shadow_map_size=2048, coverage="conservative"), 1e-4)}


FRAME_SETTINGS = ([("cones", "16+1"), ("cones", 10), ("cones", 13), ("cones", 0)] +
                  [("PcfRadius", r) for r in (0, 1, 3, 8)] + LIMITS)


@pytest.mark.parametrize("name,value", FRAME_SETTINGS, ids=[f"{n}={v}" for n, v in FRAME_SETTINGS])
@pytest.mark.parametrize("scene", ["cornell", "atrium"])
def test_frames_vs_oracle_under_non_default_uniforms(gpu_ctx, oracle, frame_scenes, scene, name, value):
    """The 10-16 cone shape, no diffuse cone at all, the generic PCF loop in both voxelisation and the frame, and the
    march limits: frames within the bars of test_gpu_parity.py, textureLod counts within 1e-4 (2e-4 on the small frame,
    see frame_scenes)."""
    sc, kw, samples_bar = frame_scenes[scene]
    u = uniforms.scene_uniforms(sc, **kw)
    if name == "cones":
        u["ConeDirections"], u["ConeWeights"] = uniforms.cone_set(value) if isinstance(value, str) else ring_table(value)
    else:
        u[name] = value
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    # MaxAlpha = 0.5 ends a cone where the rest of the ray still carries half of its light: one step added or dropped at
    # that threshold moves a pixel by far more than the 5/255 of the reference's 0.95.  The share of pixels within
    # 2/255 is the measure that stays meaningful there, and its bar is the same as for every other small frame.
    assert_frame_close(gpu_ctx.read_frame(), oracle.frame(), f"{scene} {name}={value}", FRAC_MIN_SMALL)
    assert abs(gpu_ctx.cone_samples() - oracle.cone_samples()) <= samples_bar * oracle.cone_samples()


@pytest.mark.parametrize("W,H", [(1, 1), (7, 5), (13, 97), (250, 131)])
def test_odd_frame_sizes_vs_oracle(gpu_ctx, oracle, W, H):
    """Frames whose sizes are not multiples of the 8x8 cone_trace block or of the raster tiles: visibility equal to the
    oracle's, every pixel within one threshold flip (5/255), and on frames of 1000 pixels or more the share bar."""
    sc = scenes.cornell()
    u = uniforms.scene_uniforms(sc, V=64, width=W, height=H, shadow_map_size=1024)
    run_gpu(gpu_ctx, sc, u)
    run_oracle(oracle, sc, u)
    vis = gpu_ctx.visibility()
    assert np.array_equal(vis, oracle.visibility())
    assert (vis != MISS).any()
    fg, fo = gpu_ctx.read_frame(), oracle.frame()
    d = np.abs(fg.astype(int) - fo.astype(int)).max()
    print(f"[parity] cornell {W}x{H}: psnr {psnr(fg[..., :3], fo[..., :3]):.2f} dB, "
          f"{100 * frac_within(fg, fo, 2):.4f} % of pixels within 2/255, max |diff| {d}")
    assert d <= FLIP_LSB, d
    if W * H >= 1000:
        assert_frame_close(fg, fo, f"cornell {W}x{H}", FRAC_MIN_SMALL)
