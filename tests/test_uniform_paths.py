"""The oracle under the uniforms the reference never changes: PCF radius and shadow-map size, StepMultiplier, MaxDistance
and MaxAlpha.  The library takes PcfRadius 0-8, ShadowMapSize 1-16384 and any march limits, so the float64
restatements of test_oracle_independent.py are run at those values too, and on uniform grids the cone march has a
closed form that gives exact step counts (tests/test_gpu_uniform_paths.py holds the device to the same answers)."""
import numpy as np
import pytest

from test_oracle_independent import cone, mip_chain, pcf_lit_taps, random_grid
from test_oracle_kat import quad_mesh, setup

G = 150.0

# (uniform, value) changed one at a time from the reference's StepMultiplier 1, MaxDistance 75, MaxAlpha 0.95
LIMITS = [("StepMultiplier", 0.5), ("StepMultiplier", 1.7), ("MaxDistance", 20.0), ("MaxDistance", 150.0),
          ("MaxAlpha", 0.5), ("MaxAlpha", 0.99)]
UNIFORM_ALPHAS = (32, 96, 255)
KAT_MARGIN = 1e-4


# ------------------------------------------------------------------------------------- closed form, uniform grids
def uniform_cone(V, alpha8, tan_half, step_mult=1.0, max_dist=75.0, max_alpha=0.95, grid_world=G):
    """The cone loop of VoxelConeTracing.fs:82-107 on a grid whose every texel has alpha byte `alpha8`: every mip level
    is the same grid ((8 v + 4) >> 3 = v) and every filter weight set sums to one, so each sample is exactly a = A/255.
    Alpha after k steps is 1 - (1 - a)^k and the distance runs d <- d + max(vws, 2 tan d) * StepMultiplier from
    d = vws.  Returns (steps, sum of (1 - alpha) over the steps, occlusion), or None when alpha or the distance of any
    step lands within KAT_MARGIN of its limit (relative for the distance), where float32 rounding may decide the exit.
    The uniforms are rounded to float32 first, as the library and the oracle store them."""
    f32 = lambda x: float(np.float32(x))
    tan_half, step_mult, max_dist, max_alpha = f32(tan_half), f32(step_mult), f32(max_dist), f32(max_alpha)
    a = alpha8 / 255.0
    vws = f32(grid_world) / V
    dist, alpha, k, trans, occ = vws, 0.0, 0, 0.0, 0.0
    if abs(dist - max_dist) <= KAT_MARGIN * max_dist:
        return None
    while dist < max_dist and alpha < max_alpha:
        diameter = max(vws, 2.0 * tan_half * dist)
        trans += 1.0 - alpha
        occ += (1.0 - alpha) * a / (1.0 + 0.03 * diameter)
        k += 1
        alpha = 1.0 - (1.0 - a) ** k
        dist += diameter * step_mult
        if abs(alpha - max_alpha) <= KAT_MARGIN or abs(dist - max_dist) <= KAT_MARGIN * max_dist:
            return None
    return k, trans, occ


def uniform_steps(V, alpha8, u):
    """(k_d, k_s): textureLod calls of one diffuse and of the specular cone on a uniform grid under the uniforms `u`
    (a dict as uniforms.reference_uniforms returns), or None if either is too close to a limit to call."""
    lim = dict(step_mult=u["StepMultiplier"], max_dist=u["MaxDistance"], max_alpha=u["MaxAlpha"],
               grid_world=u["VoxelGridWorldSize"])
    d = uniform_cone(V, alpha8, u["DiffuseTanHalfAngle"], **lim)
    s = uniform_cone(V, alpha8, u["SpecularTanHalfAngle"], **lim)
    if d is None or s is None:
        return None
    return d[0], s[0]


def limit_uniforms(u, name=None, value=None):
    u = dict(u)
    if name is not None:
        u[name] = value
    return u


def test_uniform_grid_closed_form_known_values():
    """Hand-checked anchors: the reference's step table on an empty grid at V = 128 (6 diffuse, 23 specular steps, the
    A.5 table of test_gpu_parity.test_uniform_grid_cone_kat_on_gpu) and one step on an opaque grid."""
    from vct_b200 import uniforms
    u = uniforms.reference_uniforms(V=128)
    assert uniform_steps(128, 0, u) == (6, 23)
    assert uniform_steps(128, 255, u) == (1, 1)
    k, trans, occ = uniform_cone(128, 255, 0.07)            # first diameter = vws: occlusion 1 / (1 + 0.03 vws)
    assert (k, trans) == (1, 1.0) and occ == pytest.approx(0.966038, abs=1e-6)
    # a = 96/255 reaches 0.95 after ceil(log(0.05) / log(1 - a)) = 7 steps unless the distance runs out first
    k, _, _ = uniform_cone(32, 96, 0.07, max_dist=1e4)
    assert k == int(np.ceil(np.log(0.05) / np.log(1 - 96 / 255)))


@pytest.mark.parametrize("V", [32, 64])
@pytest.mark.parametrize("alpha8", UNIFORM_ALPHAS)
def test_uniform_grid_closed_form_matches_oracle_cone(oracle, V, alpha8):
    """The closed form against the oracle's float32 cone loop under every march-limit setting: step counts exact, colour
    and occlusion to float32 accuracy."""
    rng = np.random.default_rng(V + alpha8)
    base = setup(oracle, V=V)
    g = np.empty((V, V, V, 4), dtype=np.uint8)
    g[..., :3] = 153
    g[..., 3] = alpha8
    oracle.set_grid_level0(g)
    checked = 0
    for name, value in [(None, None)] + LIMITS:
        u = limit_uniforms(base, name, value)
        oracle.set_uniforms(u)
        lim = dict(step_mult=u["StepMultiplier"], max_dist=u["MaxDistance"], max_alpha=u["MaxAlpha"])
        for tan_half in (0.577, 0.07):
            want = uniform_cone(V, alpha8, tan_half, **lim)
            if want is None:
                continue                                 # a step sits on a limit (KAT_MARGIN)
            k, trans, occ = want
            for _ in range(4):                           # the grid is uniform: position and direction do not matter
                start = rng.uniform(-70, 70, 3)
                d = rng.normal(size=3); d /= np.linalg.norm(d)
                got, n = oracle.cone(start, d, tan_half)
                assert n == k, (name, value, tan_half)
                np.testing.assert_allclose(got[:3], trans * 153 / 255, rtol=1e-5, atol=1e-6)
                assert got[3] == pytest.approx(occ, rel=1e-5, abs=1e-6)
            checked += 1
    assert checked >= 12, checked                         # of 14: at most two settings may sit on a limit


# -------------------------------------------------------------------------------------- float64 cone loop, limits
@pytest.mark.parametrize("name,value", LIMITS)
@pytest.mark.parametrize("tan_half", [0.577, 0.07])
def test_cone_march_under_non_default_limits(oracle, name, value, tan_half):
    """test_oracle_independent.test_cone_march_against_float64_loop with one march limit changed: the float64 loop
    (step = diameter * StepMultiplier) against the oracle on a sparse random grid, step counts exact."""
    V = 32
    rng = np.random.default_rng(int(tan_half * 1000) + int(value * 10))
    u = setup(oracle, V=V)
    u["FilterMode"] = 0
    u[name] = value
    oracle.set_uniforms(u)
    g = random_grid(V, rng, fill=0.02)
    oracle.set_grid_level0(g)
    levels = mip_chain(g)
    lim = dict(max_dist=float(np.float32(u["MaxDistance"])), max_alpha=float(np.float32(u["MaxAlpha"])),
               step_mult=float(np.float32(u["StepMultiplier"])))
    checked = 0
    for _ in range(60):
        start = rng.uniform(-60, 60, 3)
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        want, n_want, margin = cone(levels, V, start, d, tan_half, **lim)
        if margin < 1e-4:                    # a float32/float64 difference could add or drop a whole step here
            continue
        got, n_got = oracle.cone(start, d.astype(np.float32), tan_half)
        assert n_got == n_want
        assert np.abs(got - want).max() < 2e-5 * max(1, n_want), (got, want)
        checked += 1
    assert checked > 40, checked
    # the empty grid: only the distance limit and the step multiplier decide
    oracle.set_grid_level0(np.zeros_like(g))
    _, n_empty = oracle.cone((0, 0, 0), (0, 0, 1), tan_half)
    _, n_want, _ = cone(mip_chain(np.zeros_like(g)), V, (0, 0, 0), (0, 0, 1), tan_half, **lim)
    assert n_empty == n_want


# ------------------------------------------------------------------------------------------------ PCF
def _two_quad_depth_map(oracle, S, r):
    """the two overlapping tilted quads of test_oracle_independent.test_pcf_against_numpy_bilinear_taps, S x S map"""
    u = setup(oracle, V=32, shadow_map_size=S)
    u["PcfRadius"] = r
    oracle.set_uniforms(u)
    v1, i1 = quad_mesh((-70, -10, -60), (-70, 0, 60), (70, 6, 60), (70, -4, -60))
    v2, i2 = quad_mesh((-25, 20, -25), (-28, 26, 22), (26, 30, 28), (30, 24, -20))
    oracle.upload_mesh(np.concatenate([v1, v2]), np.concatenate([i1, i2 + 4]))
    oracle.draw_depth()
    return oracle.depth().astype(np.float64) / 16777215.0


@pytest.mark.parametrize("S", [1, 3, 64, 257])
@pytest.mark.parametrize("r", [0, 1, 3, 8])
def test_pcf_any_radius_and_map_size_against_numpy_taps(oracle, r, S):
    """PCF_Shadow_Mapping with a (2r+1)^2 kernel on an S x S map: GL_LINEAR, CLAMP_TO_EDGE, taps at coord + k/S, against
    the oracle's lit count exactly.  Taps within 2e-6 of the compare threshold are skipped."""
    tex = _two_quad_depth_map(oracle, S, r)
    covered = (tex < 1.0).sum()
    assert covered >= (1 if S < 64 else S * S // 8)
    taps = (2 * r + 1) ** 2
    rng = np.random.default_rng(100 * r + S)
    # half of the taps anywhere, half around texels next to a depth step with the compare depth inside the step
    step = np.zeros_like(tex, dtype=bool)
    step[:, :-1] |= np.abs(np.diff(tex, axis=1)) > 0.01
    step[:-1, :] |= np.abs(np.diff(tex, axis=0)) > 0.01
    edge = np.argwhere(step)
    trials, checked, partial = 300, 0, 0
    for t in range(trials):
        if t % 2 and len(edge):
            j, i = edge[rng.integers(len(edge))]
            lo, hi = tex[j:j + 2, i:i + 2].min(), tex[j:j + 2, i:i + 2].max()
            dc = [(i + rng.uniform(0, 2)) / S, (j + rng.uniform(0, 2)) / S, rng.uniform(lo, hi) + 0.002, 1.0]
        else:
            dc = [rng.uniform(-0.05, 1.05), rng.uniform(-0.05, 1.05), rng.uniform(0.2, 0.8), 1.0]
        dc = np.array(dc, dtype=np.float32).astype(np.float64)
        lit, safe = pcf_lit_taps(tex, S, dc, r=r)
        if not safe:
            continue
        got = oracle.pcf(dc) * taps
        assert got == pytest.approx(round(got), abs=1e-3) and round(got) == lit, (dc, got, lit)
        checked += 1
        partial += 0 < lit < taps
    assert checked > 0.9 * trials, checked
    if r > 0 and S >= 64:
        assert partial > 30, partial          # the kernel straddles the depth steps, so the radius matters
