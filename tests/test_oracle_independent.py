"""Second, independent restatement of the arithmetic-heavy pieces of the path, in float64 numpy / exact Python
integers, written from the GLSL and the GL 4.3 filtering rules rather than from the C++ oracle, and compared with
the oracle on random inputs.  The reference has no tests of its own (SURVEY.md 8c); next to the executed reference
shaders of test_reference_glsl.py, these cross-checks, the hand-derived vectors in test_oracle_kat.py and the golden
fixtures are what pins the oracle.

  * SampleVoxels / textureLod        VoxelConeTracing.fs:59-66, GL 4.3 8.14 (weighted-sum form, float64)
  * Voxel_Cone_Tracing loop          VoxelConeTracing.fs:82-107
  * PCF_Shadow_Mapping               Voxelization.fs:18-52 (bilinear GL_LINEAR taps, CLAMP_TO_EDGE)
  * ortho rasteriser coverage        GL 4.3 14.6.1: interior / exterior / shared-edge exactly-once, exact integers
"""
import numpy as np
import pytest

from vct_b200 import scenes, uniforms
from test_oracle_kat import quad_mesh, setup

G = 150.0


# ---------------------------------------------------------------------------------------------- voxel texture
def mip_chain(g0):
    """(sum of 8 + 4) >> 3 per channel (DESIGN.md, defined semantics) -- integer, so exact."""
    levels = [g0.astype(np.int64)]
    while levels[-1].shape[0] > 1:
        p = levels[-1]
        n = p.shape[0] // 2
        levels.append((p.reshape(n, 2, n, 2, n, 2, 4).sum((1, 3, 5)) + 4) >> 3)
    return [l.astype(np.float64) / 255.0 for l in levels]


def sample_level(level, uvw):
    """GL_LINEAR on a 3D level with GL_REPEAT: eight texels weighted by the products of (1 - f) / f."""
    n = level.shape[0]
    t = np.asarray(uvw, dtype=np.float64) * n - 0.5
    i0 = np.floor(t).astype(int)
    f = t - i0
    out = np.zeros(4)
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                w = (f[0] if dx else 1 - f[0]) * (f[1] if dy else 1 - f[1]) * (f[2] if dz else 1 - f[2])
                out += w * level[(i0[2] + dz) % n, (i0[1] + dy) % n, (i0[0] + dx) % n]
    return out


def sample_voxels(levels, pos, lod):
    uvw = np.asarray(pos, dtype=np.float64) / (G / 2) * 0.5 + 0.5       # VoxelConeTracing.fs:61-63
    lod = min(max(lod, 0.0), len(levels) - 1.0)
    l0 = int(np.floor(lod))
    f = lod - l0
    a = sample_level(levels[l0], uvw)
    if f > 0 and l0 + 1 < len(levels):
        a = (1 - f) * a + f * sample_level(levels[l0 + 1], uvw)
    return a


def cone(levels, V, start, direction, tan_half, max_dist=75.0, max_alpha=0.95, step_mult=1.0):
    """VoxelConeTracing.fs:82-107 in float64 (the step is diameter * StepMultiplier, 1 in the reference); also returns
    how close alpha and distance came to their exit thresholds."""
    vws = G / V
    dist, alpha, occ, color, n, margin = vws, 0.0, 0.0, np.zeros(3), 0, 1.0
    start, direction = np.asarray(start, dtype=np.float64), np.asarray(direction, dtype=np.float64)
    while dist < max_dist and alpha < max_alpha:
        diameter = max(vws, 2 * tan_half * dist)
        s = sample_voxels(levels, start + dist * direction, np.log2(diameter / vws))
        color += (1 - alpha) * s[:3]
        occ += (1 - alpha) * s[3] / (1 + 0.03 * diameter)
        alpha += (1 - alpha) * s[3]
        dist += diameter * step_mult
        n += 1
        margin = min(margin, abs(alpha - max_alpha), abs(dist - max_dist) / max_dist)
    return np.append(color, occ), n, margin


def random_grid(V, rng, fill=0.08):
    g = np.zeros((V, V, V, 4), dtype=np.uint8)
    occ = rng.random((V, V, V)) < fill
    g[occ, :3] = rng.integers(0, 256, (int(occ.sum()), 3))
    g[occ, 3] = 255
    return g


@pytest.mark.parametrize("V", [16, 32])
def test_sample_voxels_against_float64_weighted_sum(oracle, V):
    rng = np.random.default_rng(V)
    u = setup(oracle, V=V)
    u["FilterMode"] = 0                      # fp32 filter weights (mode 1 models the 8-bit hardware weights)
    oracle.set_uniforms(u)
    g = random_grid(V, rng, fill=0.3)
    oracle.set_grid_level0(g)
    levels = mip_chain(g)
    for l in range(len(levels)):             # the oracle's own pyramid is the integer one
        assert np.array_equal(np.rint(levels[l] * 255).astype(np.uint8), oracle.grid(l))
    worst = 0.0
    for _ in range(300):
        pos = rng.uniform(-110, 110, 3)      # beyond +-75: GL_REPEAT wraps (the reference never sets a wrap mode)
        lod = float(rng.uniform(-0.5, np.log2(V) + 0.5))
        worst = max(worst, np.abs(oracle.sample_voxels(pos, lod) - sample_voxels(levels, pos, lod)).max())
    assert worst < 3e-6, worst


def test_quantised_filter_mode_stays_within_one_weight_step(oracle):
    """FilterMode 1 (default; 8-bit weights, LOD fraction truncated to 1/256 as measured on the texture hardware) differs
    from the exact filter by at most the weight quantisation: 3 axes * 1/512 + the LOD step 1/256."""
    V = 16
    rng = np.random.default_rng(5)
    u = setup(oracle, V=V)
    g = random_grid(V, rng, fill=0.3)
    levels = mip_chain(g)
    oracle.set_grid_level0(g)
    worst = 0.0
    for _ in range(300):
        pos = rng.uniform(-75, 75, 3)
        lod = float(rng.uniform(0, np.log2(V)))
        worst = max(worst, np.abs(oracle.sample_voxels(pos, lod) - sample_voxels(levels, pos, lod)).max())
    assert 1e-5 < worst <= 3 / 512 + 1 / 256 + 1e-6, worst


@pytest.mark.parametrize("tan_half", [0.577, 0.07])
def test_cone_march_against_float64_loop(oracle, tan_half):
    V = 32
    rng = np.random.default_rng(int(tan_half * 1000))
    u = setup(oracle, V=V)
    u["FilterMode"] = 0
    oracle.set_uniforms(u)
    g = random_grid(V, rng, fill=0.02)
    oracle.set_grid_level0(g)
    levels = mip_chain(g)
    checked = 0
    for _ in range(60):
        start = rng.uniform(-60, 60, 3)
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        want, n_want, margin = cone(levels, V, start, d, tan_half)
        if margin < 1e-4:                    # a float32/float64 difference could add or drop a whole step here
            continue
        got, n_got = oracle.cone(start, d.astype(np.float32), tan_half)
        assert n_got == n_want
        assert np.abs(got - want).max() < 2e-5 * max(1, n_want), (got, want)
        checked += 1
    assert checked > 40
    # step counts on an empty grid: distances 75/16 * (1 + 2 tan)^k style growth until 75 (SURVEY.md A.5)
    oracle.set_grid_level0(np.zeros_like(g))
    _, n_empty = oracle.cone((0, 0, 0), (0, 0, 1), tan_half)
    _, n_want, _ = cone(mip_chain(np.zeros_like(g)), V, (0, 0, 0), (0, 0, 1), tan_half)
    assert n_empty == n_want


# ---------------------------------------------------------------------------------------------------- PCF
def test_pcf_against_numpy_bilinear_taps(oracle):
    S = 64
    u = setup(oracle, V=32, shadow_map_size=S)
    # two overlapping tilted quads so that the map holds a depth discontinuity
    # (wound to face the light at +y: the shadow pass culls back faces, Voxel_Cone_Tracing.h:198-199)
    v1, i1 = quad_mesh((-70, -10, -60), (-70, 0, 60), (70, 6, 60), (70, -4, -60))
    v2, i2 = quad_mesh((-25, 20, -25), (-28, 26, 22), (26, 30, 28), (30, 24, -20))
    oracle.upload_mesh(np.concatenate([v1, v2]), np.concatenate([i1, i2 + 4]))
    oracle.draw_depth()
    d24 = oracle.depth().astype(np.float64)                  # [row][col] of D24 integers
    assert (d24 < 0xFFFFFF).sum() > 500
    tex = d24 / 16777215.0

    def bilinear(uv):
        x, y = uv[0] * S - 0.5, uv[1] * S - 0.5
        i, j = int(np.floor(x)), int(np.floor(y))
        a, b = x - i, y - j
        cl = lambda k: min(max(k, 0), S - 1)                 # CLAMP_TO_EDGE, Voxel_Cone_Tracing.h:95-96
        t = lambda ii, jj: tex[cl(jj), cl(ii)]
        return (1 - b) * ((1 - a) * t(i, j) + a * t(i + 1, j)) + b * ((1 - a) * t(i, j + 1) + a * t(i + 1, j + 1))

    rng = np.random.default_rng(3)
    checked = 0
    for _ in range(400):
        dc = np.array([rng.uniform(-0.05, 1.05), rng.uniform(-0.05, 1.05), rng.uniform(0.2, 0.8), 1.0])
        cur = dc[2] / dc[3]
        lit, safe = 0, True
        for x in range(-2, 3):                               # Voxelization.fs:32-44
            for y in range(-2, 3):
                closest = bilinear((dc[0] + x / S, dc[1] + y / S))
                if abs((cur - 0.002) - closest) < 1e-5:
                    safe = False
                lit += (cur - 0.002) <= closest
        if not safe:
            continue
        assert oracle.pcf(dc) == pytest.approx(lit / 25.0, abs=1e-6)
        checked += 1
    assert checked > 300


# ------------------------------------------------------------------------------------------------ rasteriser
def edge(a, b, p):
    return (b[0] - a[0]) * (p[1] - a[1]) - (b[1] - a[1]) * (p[0] - a[0])


def classify(tri, p):
    """+1 strictly inside, 0 on the boundary, -1 outside; exact integers"""
    e = [edge(tri[k], tri[(k + 1) % 3], p) for k in range(3)]
    if edge(tri[0], tri[1], tri[2]) < 0:
        e = [-x for x in e]
    if min(e) > 0:
        return 1
    return 0 if min(e) == 0 else -1


def test_center_coverage_of_random_triangle_pairs_exact(oracle):
    """Pixel-centre coverage (CoveragePolicy 0) of two triangles sharing an edge, vertices on the 1/256-pixel lattice so
    that the snap is exact: strictly interior centres are hit, exterior ones are not, centres on the shared edge are
    hit exactly once, centres on the outer boundary at most once (GL 4.3 14.6.1; no reliance on which edge owns)."""
    V = 32
    rng = np.random.default_rng(11)
    sub = 256
    for trial in range(25):
        setup(oracle, V=V, coverage="center")
        # convex quad A-B-D-C in window lattice units, split along B-C; some vertices ON pixel centres
        while True:
            q = rng.integers(2 * sub, (V - 2) * sub, (4, 2))
            if trial % 3 == 0:
                q = (q // sub) * sub + sub // 2
            A, B, C, D = [tuple(int(x) for x in p) for p in q]
            o1, o2 = edge(A, B, C), edge(C, B, D)
            if o1 != 0 and o2 != 0 and (o1 > 0) == (o2 > 0) and (edge(A, B, D) > 0) == (o1 > 0) and (edge(A, D, C) < 0) == (o1 < 0):
                break
        z_world = 75.0 - (rng.integers(0, V) + 0.5) * G / V   # mid-voxel plane: the slice index is unambiguous
        to_world = lambda p: (p[0] / sub * G / V - 75.0, p[1] / sub * G / V - 75.0, z_world)
        verts = np.zeros((4, 14), dtype=np.float32)
        verts[:, :3] = np.array([to_world(p) for p in (A, B, C, D)]) * 20.0
        verts[:, 3:6] = (0, 0, 1); verts[:, 8:11] = (1, 0, 0); verts[:, 11:14] = (0, 1, 0)
        oracle.upload_mesh(verts, np.array([[0, 1, 2], [2, 1, 3]], dtype=np.uint32))
        oracle.draw_depth(); oracle.draw_voxels()
        c = oracle.counts()
        zs = np.nonzero(c.sum((1, 2)))[0]
        assert len(zs) == 1 and zs[0] == int(np.floor((z_world / G + 0.5) * V))
        cov = c[zs[0]]                                        # [y][x]
        t1, t2 = (A, B, C), (C, B, D)
        n_inside = 0
        for j in range(V):
            for i in range(V):
                p = (i * sub + sub // 2, j * sub + sub // 2)
                k1, k2 = classify(t1, p), classify(t2, p)
                got = int(cov[j, i])
                if k1 == 1 or k2 == 1:
                    assert got == 1, (trial, i, j)
                    n_inside += 1
                elif k1 == -1 and k2 == -1:
                    assert got == 0, (trial, i, j)
                elif k1 == 0 and k2 == 0 and edge(B, C, p) == 0 and p not in (B, C):
                    assert got == 1, ("shared edge", trial, i, j)
                else:
                    assert got in (0, 1), (trial, i, j)
        assert n_inside == 0 or cov.sum() >= n_inside


# ------------------------------------------------------------------------------------------ material textures
def test_material_texture_trilinear_repeat_against_float64(oracle):
    """texture()/textureLod on a 2D material texture: RGBA8 + 2x2 box mips (sum of 4 + 2) >> 2, GL_REPEAT, trilinear
    (Model.h:172-175).  Quantised hardware-style weights (FilterMode 1) stay within the weight step of the exact filter."""
    rng = np.random.default_rng(21)
    tex = rng.integers(0, 256, (16, 32, 4), dtype=np.uint8)          # h = 16, w = 32
    u = setup(oracle, V=16)
    levels = [tex.astype(np.int64)]
    while levels[-1].shape[0] > 1 or levels[-1].shape[1] > 1:
        p = levels[-1]
        h, w = max(p.shape[0] // 2, 1), max(p.shape[1] // 2, 1)
        if p.shape[0] == 1:
            p = np.concatenate([p, p], 0)
        if p.shape[1] == 1:
            p = np.concatenate([p, p], 1)
        levels.append((p.reshape(h, 2, w, 2, 4).sum((1, 3)) + 2) >> 2)
    levels = [l.astype(np.float64) / 255.0 for l in levels]

    def sample2d(level, s, t):
        h, w = level.shape[:2]
        x, y = s * w - 0.5, t * h - 0.5
        i, j = int(np.floor(x)), int(np.floor(y))
        a, b = x - i, y - j
        at = lambda ii, jj: level[jj % h, ii % w]
        return (1 - b) * ((1 - a) * at(i, j) + a * at(i + 1, j)) + b * ((1 - a) * at(i, j + 1) + a * at(i + 1, j + 1))

    for mode, tol in ((0, 3e-6), (1, 2 / 512 + 1 / 256 + 1e-6)):
        u["FilterMode"] = mode
        oracle.set_uniforms(u)
        oracle.upload_texture(3, tex)
        worst = 0.0
        for _ in range(300):
            s, t = rng.uniform(-2, 3, 2)
            lod = float(rng.uniform(0, len(levels) - 1))
            l0 = int(np.floor(lod)); f = lod - l0
            want = sample2d(levels[l0], s, t)
            if f > 0 and l0 + 1 < len(levels):
                want = (1 - f) * want + f * sample2d(levels[l0 + 1], s, t)
            worst = max(worst, np.abs(oracle.sample_texture(3, s, t, lod) - want).max())
        assert worst <= tol, (mode, worst)


# ------------------------------------------------------------------------------------------ primary visibility
def test_visibility_against_float64_ray_casting(oracle):
    """S2 (VoxelConeTracing.vs + GL raster, depth test LESS, back-face culling): the triangle the oracle's homogeneous
    rasteriser finds per pixel must be the nearest front-facing triangle hit by the ray through the pixel centre."""
    sc = scenes.cornell()
    W, H = 80, 64
    u = uniforms.scene_uniforms(sc, V=32, width=W, height=H, shadow_map_size=256)
    oracle.set_uniforms(u); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels(); oracle.render()
    vis = oracle.visibility()                                   # [row][col], row 0 = bottom (GL window order)
    MV = np.asarray(u["ModelViewMatrix"], dtype=np.float64).reshape(4, 4).T     # column-major -> maths form
    P = np.asarray(u["ProjectionMatrix"], dtype=np.float64).reshape(4, 4).T
    inv = np.linalg.inv(P @ MV)
    pos = sc.verts[:, :3].astype(np.float64)
    tri = pos[sc.idx.astype(np.int64)]                          # [nt][3][3], model space
    e1, e2 = tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]
    nrm = np.cross(e1, e2)
    mism = total = 0
    for j in range(H):
        for i in range(W):
            ndc = np.array([(i + 0.5) / W * 2 - 1, (j + 0.5) / H * 2 - 1])
            a = inv @ np.array([ndc[0], ndc[1], -1.0, 1.0]); b = inv @ np.array([ndc[0], ndc[1], 1.0, 1.0])
            o, d = a[:3] / a[3], b[:3] / b[3] - a[:3] / a[3]
            # Moeller-Trumbore for all triangles at once
            pv = np.cross(d, e2)
            det = (e1 * pv).sum(1)
            ok = np.abs(det) > 1e-12
            inv_det = np.where(ok, 1.0 / np.where(ok, det, 1.0), 0.0)
            tv = o - tri[:, 0]
            uu = (tv * pv).sum(1) * inv_det
            qv = np.cross(tv, e1)
            vv = (qv * d).sum(1) * inv_det
            tt = (qv * e2).sum(1) * inv_det
            eps = 1e-4
            live = ok & (tt > 0) & (tt < 1) & ((nrm * d).sum(1) < 0)      # between the planes, front facing (CCW)
            hit = live & (uu > eps) & (vv > eps) & (uu + vv < 1 - eps)
            edge_case = live & (uu > -eps) & (vv > -eps) & (uu + vv < 1 + eps) & ~hit
            if edge_case.any():
                continue                                        # on or next to an edge: the fill rule decides
            want = 0xFFFFFFFF
            if hit.any():
                cand = np.nonzero(hit)[0]
                t_min = tt[cand].min()
                near = cand[tt[cand] < t_min + 1e-9]
                if len(near) > 1:
                    continue                                    # coplanar duplicates: tie broken by triangle id
                want = int(near[0])
            total += 1
            mism += int(vis[j, i]) != want
    assert total > 0.8 * W * H
    assert mism == 0, (mism, total)


# ------------------------------------------------------------------------------------- whole fragment shader
def pcf_lit_taps(tex, S, dc, bias=0.002, r=2):
    """Voxelization.fs:18-52 / VoxelConeTracing.fs:132-163 without the final normalisation, for a (2r+1)^2 tap kernel
    (r = 2 in the reference); also says whether any tap sits on the compare threshold."""
    def bilinear(s, t):
        x, y = s * S - 0.5, t * S - 0.5
        i, j = int(np.floor(x)), int(np.floor(y))
        a, b = x - i, y - j
        cl = lambda k: min(max(k, 0), S - 1)
        at = lambda ii, jj: tex[cl(jj), cl(ii)]
        return (1 - b) * ((1 - a) * at(i, j) + a * at(i + 1, j)) + b * ((1 - a) * at(i, j + 1) + a * at(i + 1, j + 1))
    cur = dc[2] / dc[3]
    lit, safe = 0, True
    for x in range(-r, r + 1):
        for y in range(-r, r + 1):
            closest = bilinear(dc[0] + x / S, dc[1] + y / S)
            safe &= abs((cur - bias) - closest) > 2e-6
            lit += (cur - bias) <= closest
    return lit, safe


def bilinear_repeat(tex, s, t):
    """level 0 of a material texture, GL_LINEAR + GL_REPEAT; channel rules of Model.h:159-169 (RED -> (r,0,0,1), RGB -> a=1)"""
    h, w = tex.shape[:2]
    x, y = s * w - 0.5, t * h - 0.5
    i, j = int(np.floor(x)), int(np.floor(y))
    a, b = x - i, y - j
    at = lambda ii, jj: tex[jj % h, ii % w].astype(np.float64) / 255.0
    c = (1 - b) * ((1 - a) * at(i, j) + a * at(i + 1, j)) + b * ((1 - a) * at(i, j + 1) + a * at(i + 1, j + 1))
    c = np.atleast_1d(c)
    if len(c) == 1:
        return np.array([c[0], 0.0, 0.0, 1.0])
    return np.append(c[:3], 1.0) if len(c) == 3 else c


def material_levels(tex):
    """RGBA8 + 2x2 box mips (sum of 4 + 2) >> 2 (glGenerateMipmap on the material textures, Model.h:171)"""
    levels = [tex.astype(np.int64)]
    while levels[-1].shape[0] > 1 or levels[-1].shape[1] > 1:
        p = levels[-1]
        h, w = max(p.shape[0] // 2, 1), max(p.shape[1] // 2, 1)
        if p.shape[0] == 1:
            p = np.concatenate([p, p], 0)
        if p.shape[1] == 1:
            p = np.concatenate([p, p], 1)
        levels.append((p.reshape(h, 2, w, 2, -1).sum((1, 3)) + 2) >> 2)
    return [l.astype(np.uint8) for l in levels]


def trilinear_repeat(levels, s, t, lod):
    lod = min(max(lod, 0.0), len(levels) - 1.0)
    l0 = int(np.floor(lod)); f = lod - l0
    c = bilinear_repeat(levels[l0], s, t)
    if f > 0 and l0 + 1 < len(levels):
        c = (1 - f) * c + f * bilinear_repeat(levels[l0 + 1], s, t)
    return c


def _check_fragment_shader(oracle, sc, min_checked, use_lod=False, tol=1.0):
    W, H, V, S = 48, 40, 32, 256
    u = uniforms.scene_uniforms(sc, V=V, width=W, height=H, shadow_map_size=S)
    u["FilterMode"] = 0
    oracle.set_uniforms(u); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels(); oracle.render()
    frame, vis = oracle.frame(), oracle.visibility()
    levels = mip_chain(oracle.grid(0))
    shadow_tex = oracle.depth().astype(np.float64) / 16777215.0
    col = lambda name: np.asarray(u[name], dtype=np.float64).reshape(4, 4).T
    M, MV, P, DMVP = col("ModelMatrix"), col("ModelViewMatrix"), col("ProjectionMatrix"), col("DepthModelViewProjectionMatrix")
    inv = np.linalg.inv(P @ MV)
    cam = np.asarray(u["CameraPosition"], dtype=np.float64)
    L = np.asarray(u["LightDirection"], dtype=np.float64); L /= np.linalg.norm(L)
    dirs = np.asarray(u["ConeDirections"], dtype=np.float64).reshape(-1, 3)
    wts = np.asarray(u["ConeWeights"], dtype=np.float64)
    assert len(dirs) == 6 and wts[0] == pytest.approx(0.25)
    norm = lambda v: v / np.linalg.norm(v)

    def hit(i, j, p0, e1, e2):
        """ray through the centre of pixel (i, j) against the triangle's plane: barycentrics (perspective correct)"""
        ndc = np.array([(i + 0.5) / W * 2 - 1, (j + 0.5) / H * 2 - 1])
        a, b = inv @ np.array([*ndc, -1.0, 1.0]), inv @ np.array([*ndc, 1.0, 1.0])
        o, d = a[:3] / a[3], b[:3] / b[3] - a[:3] / a[3]
        pv = np.cross(d, e2); det = e1 @ pv
        tv = o - p0; bu = (tv @ pv) / det; bv = (np.cross(tv, e1) @ d) / det
        return np.array([1 - bu - bv, bu, bv])

    checked = 0
    rng = np.random.default_rng(2)
    for _ in range(600):
        i, j = int(rng.integers(0, W - 1)), int(rng.integers(0, H - 1))
        tri_id = int(vis[j, i])
        if tri_id == 0xFFFFFFFF:
            continue
        idx = sc.idx[tri_id].astype(int)
        p0, p1, p2 = sc.verts[idx, :3].astype(np.float64)
        bary = hit(i, j, p0, p1 - p0, p2 - p0)
        if bary.min() < 0.02:
            continue                                            # keep away from edges (visibility ties)
        attr = lambda bb, lo, hi: bb @ sc.verts[idx, lo:hi].astype(np.float64)
        uv = attr(bary, 6, 8)
        mat = sc.materials[int(sc.tri_material[tri_id])]
        t_diff, t_spec, t_height = (sc.textures[mat[k]] for k in range(3))
        # implicit LOD (GL 4.3 8.14) from forward differences of uv: only magnified pixels (lambda <= 0 -> level 0) are compared
        uvx, uvy = attr(hit(i + 1, j, p0, p1 - p0, p2 - p0), 6, 8), attr(hit(i, j + 1, p0, p1 - p0, p2 - p0), 6, 8)
        rho, lods = 0.0, []
        for t in (t_diff, t_spec, t_height):
            size = np.array([t.shape[1], t.shape[0]], dtype=np.float64)
            r = max(np.linalg.norm((uvx - uv) * size), np.linalg.norm((uvy - uv) * size))
            lods.append(np.log2(max(r, 1e-12)))
            rho = max(rho, r)
        if not use_lod and max(t.shape[0] * t.shape[1] for t in (t_diff, t_spec, t_height)) > 1 and rho > 0.85:
            continue
        if use_lod:                                             # minified too: trilinear with the implicit LOD
            sample = lambda t, k, s_, t_: trilinear_repeat(material_levels(t), s_, t_, lods[k])
        else:
            sample = lambda t, k, s_, t_: bilinear_repeat(t, s_, t_)
        Pm = bary @ np.stack([p0, p1, p2])
        Pw = (M @ np.append(Pm, 1.0))[:3]                       # VoxelConeTracing.vs:27-34
        Nw, Tw, Bw = (M[:3, :3] @ attr(bary, 3, 6)), (M[:3, :3] @ attr(bary, 8, 11)), (M[:3, :3] @ attr(bary, 11, 14))
        Pd = DMVP @ np.append(Pm, 1.0); Pd[:3] = Pd[:3] * 0.5 + 0.5
        albedo, spec_c = sample(t_diff, 0, *uv), sample(t_spec, 1, *uv)
        TBN = np.linalg.inv(np.stack([Tw, Bw, Nw]))             # inverse(transpose(mat3(T, B, N))), :175
        offx, offy = 1.0 / t_height.shape[1], 1.0 / t_height.shape[0]      # CalcBumpNormal, :110-128
        h0 = sample(t_height, 2, *uv)[0]
        dx = sample(t_height, 2, uv[0] + offx, uv[1])[0] - h0
        dy = sample(t_height, 2, uv[0], uv[1] + offy)[0] - h0
        bump = norm(np.cross(norm(np.array([1.0, 0.0, dx])), norm(np.array([0.0, 1.0, dy]))))
        N = norm(TBN @ bump)
        E = norm(cam - Pw)
        lit, safe = pcf_lit_taps(shadow_tex, S, Pd)
        if not safe:
            continue
        shadow = lit * 0.111                                     # :160
        start = Pw + Nw * (G / V)                                # :92, Normal_world is NOT normalised
        ind, margin = np.zeros(4), 1.0
        for k in range(6):
            c4, _, m = cone(levels, V, start, norm(TBN @ dirs[k]), 0.577)
            ind += wts[k] * c4; margin = min(margin, m)
        occlusion = 1 - ind[3]
        diffuse = (shadow * max(N @ L, 0.0) + occlusion * ind[:3]) * albedo[:3]
        if np.linalg.norm(spec_c[1:3]) == 0:
            spec_c = np.array([spec_c[0]] * 3 + [spec_c[3]])     # specColor.rrra, :208
        R = norm(2 * (N @ L) * N - L)                            # reflect(-L, N)
        direct_spec = max(E @ R, 0.0) ** mat[3] * shadow
        isp, _, m = cone(levels, V, start, norm(2 * (N @ E) * N - E), 0.07)
        margin = min(margin, m)
        if margin < 1e-4:
            continue                                             # a cone exit sits on its threshold
        specular = (isp[:3] + (1 - isp[3]) * direct_spec) * spec_c[:3]
        rgb = 0.1 * albedo[:3] * occlusion + diffuse + specular
        want = np.clip(np.append(rgb, albedo[3]), 0, 1) * 255
        got = frame[j, i].astype(np.float64)
        assert np.abs(got - want).max() <= tol, ((i, j), got, want)
        checked += 1
    assert checked > min_checked, checked


def test_fragment_shader_against_float64_restatement(oracle):
    """VoxelConeTracing.fs main() (:165-229) restated in float64 for pixels of the Cornell box: TBN = inverse(transpose(
    mat3(T, B, N))) with the un-normalised world-space frame (length 0.05), cone start offset Normal_world * voxel size,
    PCF gain 0.111 (range [0, 2.775]), six weighted diffuse cones + one specular cone, specColor.rrra for single-channel
    maps, ambient 0.1; compared with the oracle's frame to 1 LSB."""
    _check_fragment_shader(oracle, scenes.cornell(), 150)


def test_fragment_shader_with_textures_and_bump_mapping(oracle):
    """The same with multi-texel albedo / specular / height maps on every surface: bilinear REPEAT fetches, the three-tap
    CalcBumpNormal (:110-128) pushed through the TBN, RGB specular maps used as they are.  Only magnified pixels are
    compared (implicit LOD <= 0 from forward differences of the interpolated uv)."""
    sc = scenes.cornell()
    rng = np.random.default_rng(8)
    tex = [rng.integers(40, 256, (8, 8, 3), dtype=np.uint8) for _ in range(3)]          # albedo per material
    spec = rng.integers(0, 256, (4, 8, 3), dtype=np.uint8)
    height = rng.integers(0, 256, (8, 4, 1), dtype=np.uint8)
    sc.textures = tex + [spec, height]
    sc.materials = [(0, 3, 4, 20.0), (1, 3, 4, 20.0), (2, 3, 4, 20.0)]
    _check_fragment_shader(oracle, sc, 100)


def test_fragment_shader_with_minified_textures_and_implicit_lod(oracle):
    """32x32 maps on a 48x40 frame: most pixels minify.  The implicit LOD (GL 4.3 8.14: log2 of the longer of the two
    texel-space forward differences of the interpolated uv, per texture size) selects two box-filtered mip levels."""
    sc = scenes.cornell()
    rng = np.random.default_rng(9)
    smooth = lambda c: np.clip(rng.integers(60, 200, (32, 32, c)) + rng.integers(-40, 40, (32, 32, c)), 0, 255).astype(np.uint8)
    sc.textures = [smooth(3), smooth(3), smooth(3), smooth(3), smooth(1)]
    sc.materials = [(0, 3, 4, 20.0), (1, 3, 4, 20.0), (2, 3, 4, 20.0)]
    _check_fragment_shader(oracle, sc, 100, use_lod=True, tol=2.0)


# ------------------------------------------------------------------------------- voxelisation light injection
def test_light_injection_of_a_floor_under_an_occluder(oracle):
    """Voxelization.{vs,gs,fs}: a floor quad (normal +y => projected along Y, Voxelization.gs:36) partly shadowed by a
    smaller quad above it.  Every floor voxel gets one fragment at its pixel centre (centre coverage); its value is
    unorm8(albedo * lit_taps / 25) with the taps of Voxelization.fs:18-52 evaluated in float64 on the oracle's depth map,
    stored at voxel (x, y, V-1-j) per the un-swizzle of Voxelization.fs:77-82."""
    V, S = 32, 512
    u = setup(oracle, V=V, coverage="center", shadow_map_size=S)
    oracle.upload_texture(0, np.array([[[200, 100, 50]]], dtype=np.uint8))
    y_floor, y_occ = -20.3, 11.1
    v1, i1 = quad_mesh((-60, y_floor, -60), (-60, y_floor, 60), (60, y_floor, 60), (60, y_floor, -60))
    v2, i2 = quad_mesh((-22, y_occ, -17), (-22, y_occ, 23), (18, y_occ, 23), (18, y_occ, -17))
    oracle.upload_mesh(np.concatenate([v1, v2]), np.concatenate([i1, i2 + 4]))
    oracle.draw_depth(); oracle.draw_voxels()
    g, c = oracle.grid(0), oracle.counts()
    tex = oracle.depth().astype(np.float64) / 16777215.0
    DMVP = np.asarray(u["DepthModelViewProjectionMatrix"], dtype=np.float64).reshape(4, 4).T
    yv = int(np.floor((y_floor / G + 0.5) * V))
    albedo = np.array([200, 100, 50]) / 255.0
    checked = shadowed = partial = 0
    for j in range(V):
        for i in range(V):
            xw = ((i + 0.5) / V * 2 - 1) * 75.0                  # ProjY: x_ndc = x_w / 75, y_ndc = -z_w / 75 (SURVEY A.1)
            zw = -((j + 0.5) / V * 2 - 1) * 75.0
            inside = abs(xw) < 60 - 1e-6 and abs(zw) < 60 - 1e-6
            voxel = (V - 1 - j, yv, i)                           # [z][y][x]
            if not inside:
                if abs(abs(xw) - 60) > 1e-3 and abs(abs(zw) - 60) > 1e-3:
                    assert c[voxel] == 0
                continue
            assert c[voxel] == 1, (i, j)
            dc = DMVP @ np.array([xw * 20.0, y_floor * 20.0, zw * 20.0, 1.0])
            dc[:3] = dc[:3] * 0.5 + 0.5                          # Voxelization.vs:19-20
            lit, safe = pcf_lit_taps(tex, S, dc)
            if not safe:
                continue
            val = albedo * (lit / 25.0) * 255.0
            if np.any(np.abs(val - np.floor(val) - 0.5) < 1e-3):
                continue
            assert np.array_equal(g[voxel][:3], np.rint(val).astype(np.uint8)), ((i, j), lit, g[voxel])
            assert g[voxel][3] == 255
            checked += 1; shadowed += lit == 0; partial += 0 < lit < 25
    assert checked > 500 and shadowed > 20 and partial > 5


# ------------------------------------------------------------------------------------------------ shadow map
def test_shadow_map_depths_of_a_tilted_plane(oracle):
    """DrawDepthTexture (Voxel_Cone_Tracing.h:192-211, Shadow.vs): the ortho light projection is affine, so the window
    depth over a tilted quad is a plane in texel coordinates; every covered texel must hold rint(z * (2^24 - 1)) of that
    plane at the texel centre (float32 interpolation: +-2 units), uncovered texels the clear value."""
    S = 128
    u = setup(oracle, V=32, shadow_map_size=S)
    p00, e1, e2 = np.array([-50.4, -30.0, -40.1]), np.array([6.0, 35.0, 92.0]), np.array([96.0, 9.0, -8.0])
    quad = [tuple(p00), tuple(p00 + e1), tuple(p00 + e1 + e2), tuple(p00 + e2)]   # planar; cross(e1, e2) faces the light
    v, idx = quad_mesh(*quad)
    oracle.upload_mesh(v, idx)
    oracle.draw_depth()
    d = oracle.depth().astype(np.int64)
    DMVP = np.asarray(u["DepthModelViewProjectionMatrix"], dtype=np.float64).reshape(4, 4).T
    win = []
    for p in quad:
        c = DMVP @ np.array([p[0] * 20.0, p[1] * 20.0, p[2] * 20.0, 1.0])
        win.append(((c[0] * 0.5 + 0.5) * S, (c[1] * 0.5 + 0.5) * S, c[2] * 0.5 + 0.5))
    win = np.array(win)
    # vertex positions are snapped to 1/256 texel before set-up and attributes are interpolated over the snapped
    # triangle (GL 4.3 14.6.1 allows it; DESIGN.md defines 8 sub-pixel bits): up to 1/512 texel * slope = ~200 units here
    assert np.abs(win[:, :2] * 256 - np.rint(win[:, :2] * 256)).max() < 0.49
    win[:, :2] = np.rint(win[:, :2] * 256) / 256
    A = np.column_stack([win[:3, 0], win[:3, 1], np.ones(3)])
    coef = np.linalg.solve(A, win[:3, 2])                       # z = a x + b y + c through three corners
    assert abs(coef @ np.array([win[3, 0], win[3, 1], 1.0]) - win[3, 2]) < 2e-5   # planar up to the snap
    covered = d < 0xFFFFFF
    assert covered.sum() > 1500
    jj, ii = np.nonzero(covered)
    want = np.rint((coef[0] * (ii + 0.5) + coef[1] * (jj + 0.5) + coef[2]) * 16777215.0)
    # the second triangle's plane differs from the first's by the snap of the fourth corner: compare each texel with
    # the nearer of the two planes
    A2 = np.column_stack([win[[0, 2, 3], 0], win[[0, 2, 3], 1], np.ones(3)])
    coef2 = np.linalg.solve(A2, win[[0, 2, 3], 2])
    want2 = np.rint((coef2[0] * (ii + 0.5) + coef2[1] * (jj + 0.5) + coef2[2]) * 16777215.0)
    assert np.minimum(np.abs(d[jj, ii] - want), np.abs(d[jj, ii] - want2)).max() <= 3
    # coverage: texel centres strictly inside the projected quad are covered, those outside are not
    def side(a, b, px, py):
        return (b[0] - a[0]) * (py - a[1]) - (b[1] - a[1]) * (px - a[0])
    X, Y = np.meshgrid(np.arange(S) + 0.5, np.arange(S) + 0.5)
    e = np.stack([side(win[k], win[(k + 1) % 4], X, Y) for k in range(4)])
    if e[:, S // 2, S // 2].sum() < 0:
        e = -e
    inside, outside = (e > 1e-3).all(0), (e < -1e-3).any(0)
    assert covered[inside].all() and not covered[outside].any()


# ------------------------------------------------------------------------------- other coverage policies
def _random_lattice_triangle(rng, V, sub=256, min_area=None):
    while True:
        q = rng.integers(2 * sub, (V - 2) * sub, (3, 2))
        t = [tuple(int(x) for x in p) for p in q]
        a = edge(t[0], t[1], t[2])
        if abs(a) > (min_area or sub * sub):
            return t


def _voxelise_window_triangle(oracle, V, tri, rng, sub=256):
    z_world = 75.0 - (rng.integers(0, V) + 0.5) * G / V
    verts = np.zeros((3, 14), dtype=np.float32)
    verts[:, :3] = np.array([(p[0] / sub * G / V - 75.0, p[1] / sub * G / V - 75.0, z_world) for p in tri]) * 20.0
    verts[:, 3:6] = (0, 0, 1); verts[:, 8:11] = (1, 0, 0); verts[:, 11:14] = (0, 1, 0)
    oracle.upload_mesh(verts, np.array([[0, 1, 2]], dtype=np.uint32))
    oracle.draw_depth(); oracle.draw_voxels()
    c = oracle.counts()
    zs = np.nonzero(c.sum((1, 2)))[0]
    assert len(zs) == 1
    return c[zs[0]]


def test_conservative_coverage_is_exact_open_square_overlap(oracle):
    """CoveragePolicy 2 (the policy of every BASELINE config): a pixel yields a fragment iff the OPEN pixel square and the
    OPEN triangle intersect.  Exact separating-axis test in integers (axes: the square's two and the triangle's three)."""
    V, sub = 32, 256
    rng = np.random.default_rng(17)
    for trial in range(20):
        setup(oracle, V=V, coverage="conservative")
        tri = _random_lattice_triangle(rng, V)
        if trial % 4 == 0:                                     # vertices on pixel corners: touching squares do not count
            tri = [((p[0] // sub) * sub, (p[1] // sub) * sub) for p in tri]
            if edge(*tri) == 0:
                continue
        cov = _voxelise_window_triangle(oracle, V, tri, rng)
        axes = [(1, 0), (0, 1)] + [(-(tri[(k + 1) % 3][1] - tri[k][1]), tri[(k + 1) % 3][0] - tri[k][0]) for k in range(3)]
        for j in range(V):
            for i in range(V):
                sq = [(i * sub, j * sub), ((i + 1) * sub, j * sub), ((i + 1) * sub, (j + 1) * sub), (i * sub, (j + 1) * sub)]
                overlap = True
                for ax in axes:
                    pt = [ax[0] * p[0] + ax[1] * p[1] for p in tri]
                    ps = [ax[0] * p[0] + ax[1] * p[1] for p in sq]
                    if not (max(pt) > min(ps) and max(ps) > min(pt)):
                        overlap = False
                        break
                assert int(cov[j, i]) == int(overlap), (trial, i, j, tri)


def test_msaa4_any_coverage_against_sample_classification(oracle):
    """CoveragePolicy 1 (the reference's 4x MSAA window, main.cpp:30): fragment iff any of the four samples of the D3D
    pattern (+-1/8, +-3/8 rotated grid) is covered.  A sample strictly inside forces a fragment; all four strictly
    outside forbid it; samples exactly on an edge are left to the fill rule."""
    V, sub = 32, 256
    rng = np.random.default_rng(23)
    offs = [(-2, -6), (6, -2), (-6, 2), (2, 6)]                 # 1/16 pixel units
    seen_partial = 0
    for trial in range(20):
        setup(oracle, V=V, coverage="msaa4")
        tri = _random_lattice_triangle(rng, V)
        cov = _voxelise_window_triangle(oracle, V, tri, rng)
        for j in range(V):
            for i in range(V):
                ks = [classify(tri, (i * sub + sub // 2 + ox * sub // 16, j * sub + sub // 2 + oy * sub // 16)) for ox, oy in offs]
                if max(ks) == 1:
                    assert cov[j, i] == 1, (trial, i, j)
                    seen_partial += min(ks) == -1
                elif max(ks) == -1:
                    assert cov[j, i] == 0, (trial, i, j)
                else:
                    assert cov[j, i] in (0, 1)
    assert seen_partial > 50


# ------------------------------------------------------------------- dominant-axis projection of tilted triangles
def test_tilted_triangles_land_in_the_voxels_of_their_world_positions(oracle):
    """Voxelization.gs:34-47 + Voxelization.fs:58-86 for general triangles: whatever axis is chosen and however the
    fragment coordinates are un-swizzled, a fragment generated at a pixel centre must be stored in the voxel that
    contains its world-space position, floor((world / 150 + 0.5) * V) per component (SURVEY.md A.3).  Float64 plane
    intersection per pixel centre of the dominant-axis projection; centres near edges or slice boundaries are skipped."""
    V = 32
    rng = np.random.default_rng(29)
    per_axis = [0, 0, 0]
    for trial in range(45):
        setup(oracle, V=V, coverage="center")
        while True:
            w = rng.uniform(-60, 60, (3, 3))
            n = np.cross(w[1] - w[0], w[2] - w[0])
            an = np.abs(n)
            axis = int(np.argmax(an))
            if np.linalg.norm(n) > 800 and an[axis] > 1.3 * np.sort(an)[1] and axis == trial % 3:
                break
        verts = np.zeros((3, 14), dtype=np.float32)
        verts[:, :3] = w * 20.0
        verts[:, 3:6] = n / np.linalg.norm(n); verts[:, 8:11] = (1, 0, 0); verts[:, 11:14] = (0, 1, 0)
        w = verts[:, :3].astype(np.float64) * np.float64(np.float32(0.05))      # what the shader sees after ModelMatrix
        oracle.upload_mesh(verts, np.array([[0, 1, 2]], dtype=np.uint32))
        oracle.draw_depth(); oracle.draw_voxels()
        c = oracle.counts()
        # the two in-plane world axes of each projection as (component, sign): window x, window y   (SURVEY.md A.1)
        plane = {0: ((2, -1), (1, 1)), 1: ((0, 1), (2, -1)), 2: ((0, 1), (1, 1))}[axis]
        (cx, sx), (cy, sy) = plane
        win = np.stack([(sx * w[:, cx] / 75 * 0.5 + 0.5) * V, (sy * w[:, cy] / 75 * 0.5 + 0.5) * V], 1)
        d = n @ w[0]
        expected = set()
        for j in range(V):
            for i in range(V):
                p = np.array([i + 0.5, j + 0.5])
                e = np.array([(win[(k + 1) % 3, 0] - win[k, 0]) * (p[1] - win[k, 1]) - (win[(k + 1) % 3, 1] - win[k, 1]) * (p[0] - win[k, 0])
                              for k in range(3)])
                if e.sum() < 0:
                    e = -e
                if e.min() < 0.02 * abs(e.sum()):
                    continue                                    # outside, or too close to an edge to call
                pos = np.zeros(3)
                pos[cx] = sx * ((i + 0.5) / V * 2 - 1) * 75.0
                pos[cy] = sy * ((j + 0.5) / V * 2 - 1) * 75.0
                pos[axis] = (d - n[cx] * pos[cx] - n[cy] * pos[cy]) / n[axis]
                f = (pos / G + 0.5) * V
                if abs(f[axis] - np.rint(f[axis])) < 2e-3:
                    continue                                    # on a slice boundary
                vx, vy, vz = np.floor(f).astype(int)
                assert c[vz, vy, vx] >= 1, (trial, axis, (i, j), (vx, vy, vz))
                expected.add((vz, vy, vx))
        assert len(expected) > 5
        per_axis[axis] += 1
        # nothing far from the triangle: every occupied voxel lies within one voxel of its world-space bounding box
        zz, yy, xx = np.nonzero(c)
        lo = np.floor((w.min(0) / G + 0.5) * V) - 1
        hi = np.floor((w.max(0) / G + 0.5) * V) + 1
        assert np.all(xx >= lo[0]) and np.all(xx <= hi[0]) and np.all(yy >= lo[1]) and np.all(yy <= hi[1])
        assert np.all(zz >= lo[2]) and np.all(zz <= hi[2])
    assert per_axis == [15, 15, 15]


# ------------------------------------------------------------------------------------------- alpha cut-outs
def test_alpha_discard_reveals_the_surface_behind(oracle):
    """VoxelConeTracing.fs:167-172: fragments whose albedo alpha is below 0.5 are discarded before the depth write, so
    the nearest OPAQUE fragment wins.  A card with a 4x4 alpha pattern in front of a wall: per pixel, the bilinear alpha
    at the ray's hit point decides whether the card or the wall is visible."""
    rng = np.random.default_rng(31)
    W, H = 64, 48
    card_tex = np.zeros((4, 4, 4), dtype=np.uint8)
    card_tex[..., :3] = 180
    card_tex[..., 3] = np.where(rng.random((4, 4)) < 0.5, 0, 255)
    assert 3 < (card_tex[..., 3] == 0).sum() < 13
    wall_tex = np.array([[[90, 120, 200]]], dtype=np.uint8)
    flat = np.array([[[128]]], dtype=np.uint8)
    cv, ci = quad_mesh((-30, -25, 20), (30, -25, 20), (30, 25, 20), (-30, 25, 20))        # card, normal +z
    wv, wi = quad_mesh((-70, -60, -40), (70, -60, -40), (70, 60, -40), (-70, 60, -40))    # wall behind it
    sc = scenes.Scene("card", np.concatenate([cv, wv]), np.concatenate([ci, wi + 4]).astype(np.uint32),
                      np.array([0, 0, 1, 1], dtype=np.uint16), [card_tex, wall_tex, flat],
                      [(0, 2, 2, 20.0), (1, 2, 2, 20.0)], camera_pos=(6.0, 3.0, 140.0), yaw=-92.0, pitch=-1.0)
    u = uniforms.scene_uniforms(sc, V=32, width=W, height=H, shadow_map_size=256)
    u["FilterMode"] = 0
    oracle.set_uniforms(u); oracle.load_scene(sc); oracle.draw_depth(); oracle.draw_voxels(); oracle.render()
    vis, frame = oracle.visibility(), oracle.frame()
    col = lambda name: np.asarray(u[name], dtype=np.float64).reshape(4, 4).T
    inv = np.linalg.inv(col("ProjectionMatrix") @ col("ModelViewMatrix"))
    seen = {"card": 0, "hole": 0}
    for j in range(H):
        for i in range(W):
            ndc = np.array([(i + 0.5) / W * 2 - 1, (j + 0.5) / H * 2 - 1])
            a, b = inv @ np.array([*ndc, -1.0, 1.0]), inv @ np.array([*ndc, 1.0, 1.0])
            o, d = a[:3] / a[3], b[:3] / b[3] - a[:3] / a[3]
            hits = []
            for t_id in range(4):
                p0, p1, p2 = sc.verts[sc.idx[t_id].astype(int), :3].astype(np.float64)
                e1, e2 = p1 - p0, p2 - p0
                pv = np.cross(d, e2); det = e1 @ pv
                tv = o - p0; bu = (tv @ pv) / det; qv = np.cross(tv, e1); bv = (qv @ d) / det
                bary = np.array([1 - bu - bv, bu, bv])
                hits.append((t_id, bary, (qv @ e2) / det))
            if any(-0.03 < h[1].min() < 0.03 for h in hits):
                continue                                        # near an edge or a diagonal of either quad
            want = 0xFFFFFFFF
            for t_id, bary, _ in sorted((h for h in hits if h[1].min() > 0), key=lambda h: h[2]):
                if t_id < 2:
                    uv = bary @ sc.verts[sc.idx[t_id].astype(int), 6:8].astype(np.float64)
                    alpha = bilinear_repeat(card_tex, *uv)[3]
                    if abs(alpha - 0.5) < 0.03:
                        want = None
                        break
                    if alpha < 0.5:
                        seen["hole"] += 1
                        continue                                # discarded: look further along the ray
                    seen["card"] += 1
                want = t_id
                break
            if want is None:
                continue
            assert int(vis[j, i]) == want, ((i, j), int(vis[j, i]), want)
            if want == 0xFFFFFFFF:
                assert tuple(frame[j, i]) == (128, 128, 128, 255)      # glClearColor 0.5 grey, Voxel_Cone_Tracing.h:156-159
    assert seen["card"] > 100 and seen["hole"] > 100


# ------------------------------------------------------------------------------- Bounces >= 3 (extension)
def test_reinjection_bounce_against_float64_gather(oracle):
    """Bounces = 3 (DESIGN.md "Bounces"; the reference only claims it, README.md:14): every occupied voxel gathers one
    diffuse-aperture cone along each of +-X, +-Y, +-Z from one voxel outside its centre through the pyramid of the
    previous bounce, averages them, and stores min(old + gathered * old, 1); alpha is untouched."""
    V = 16
    rng = np.random.default_rng(41)
    u = setup(oracle, V=V)
    u["FilterMode"] = 0
    oracle.set_uniforms(u)
    counts = (rng.random((V, V, V)) < 0.06).astype(np.uint32) * rng.integers(1, 4, (V, V, V)).astype(np.uint32)
    sums = (rng.integers(20, 256, (V, V, V, 3)) * counts[..., None]).astype(np.uint32)
    oracle.set_accum(counts, sums); oracle.resolve_and_mip()
    g2 = oracle.grid(0).copy()
    levels = mip_chain(g2)
    u["Bounces"] = 3
    oracle.set_uniforms(u)
    oracle.set_accum(counts, sums); oracle.resolve_and_mip()
    g3 = oracle.grid(0)
    assert np.array_equal(g3[..., 3], g2[..., 3])
    vws = G / V
    checked = brighter = 0
    for z, y, x in zip(*np.nonzero(counts)):
        centre = (np.array([x, y, z]) + 0.5) * vws - G / 2
        acc, margin = np.zeros(3), 1.0
        for axis in range(3):
            for sign in (1.0, -1.0):
                d = np.zeros(3); d[axis] = sign
                c4, _, m = cone(levels, V, centre + d * vws, d, 0.577)
                acc += c4[:3] / 6.0; margin = min(margin, m)
        if margin < 1e-4:
            continue
        base = g2[z, y, x, :3].astype(np.float64) / 255.0
        val = np.minimum(base + acc * base, 1.0) * 255.0
        if np.any(np.abs(val - np.floor(val) - 0.5) < 2e-3):
            continue
        assert np.array_equal(g3[z, y, x, :3], np.rint(val).astype(np.uint8)), ((x, y, z), g3[z, y, x], val)
        checked += 1; brighter += bool((g3[z, y, x, :3] > g2[z, y, x, :3]).any())
    assert checked > 150 and brighter > 50
