"""Voxel view (vct_render_voxels, DESIGN.md section 3 "Voxel view") on the CPU: hand-derived known answers on the C++
reference (tests/voxel_view_ref.cpp, fed with the oracle's parameters and mip pyramid), an independent numpy float32
restatement of the rule that must agree with it in every byte, index and step count, and the flythrough tool's --voxels
option.  The device is held to the reference in
tests/test_gpu_voxel_view.py."""
import importlib.util
import os

import numpy as np
import pytest

from vct_b200 import glmath as gm
from vct_b200 import uniforms
from voxel_view_ref import render_voxels as ref_view

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
MISS = 0xFFFFFFFF


# ------------------------------------------------------------------------------------------ numpy restatement
def _mat_mul(A, B):
    """column-major 4x4 product in double, glm's operator* order"""
    return [((A[0 * 4 + i] * B[j * 4 + 0] + A[1 * 4 + i] * B[j * 4 + 1]) + A[2 * 4 + i] * B[j * 4 + 2]) + A[3 * 4 + i] * B[j * 4 + 3]
            for j in range(4) for i in range(4)]


def _inverse_glm(a):
    """glm::inverse(mat4) in double, operation for operation (compute_inverse<4, 4>)"""
    m = lambda c, r: a[c * 4 + r]
    c00 = m(2, 2) * m(3, 3) - m(3, 2) * m(2, 3); c02 = m(1, 2) * m(3, 3) - m(3, 2) * m(1, 3); c03 = m(1, 2) * m(2, 3) - m(2, 2) * m(1, 3)
    c04 = m(2, 1) * m(3, 3) - m(3, 1) * m(2, 3); c06 = m(1, 1) * m(3, 3) - m(3, 1) * m(1, 3); c07 = m(1, 1) * m(2, 3) - m(2, 1) * m(1, 3)
    c08 = m(2, 1) * m(3, 2) - m(3, 1) * m(2, 2); c10 = m(1, 1) * m(3, 2) - m(3, 1) * m(1, 2); c11 = m(1, 1) * m(2, 2) - m(2, 1) * m(1, 2)
    c12 = m(2, 0) * m(3, 3) - m(3, 0) * m(2, 3); c14 = m(1, 0) * m(3, 3) - m(3, 0) * m(1, 3); c15 = m(1, 0) * m(2, 3) - m(2, 0) * m(1, 3)
    c16 = m(2, 0) * m(3, 2) - m(3, 0) * m(2, 2); c18 = m(1, 0) * m(3, 2) - m(3, 0) * m(1, 2); c19 = m(1, 0) * m(2, 2) - m(2, 0) * m(1, 2)
    c20 = m(2, 0) * m(3, 1) - m(3, 0) * m(2, 1); c22 = m(1, 0) * m(3, 1) - m(3, 0) * m(1, 1); c23 = m(1, 0) * m(2, 1) - m(2, 0) * m(1, 1)
    F = [(c00, c00, c02, c03), (c04, c04, c06, c07), (c08, c08, c10, c11), (c12, c12, c14, c15), (c16, c16, c18, c19), (c20, c20, c22, c23)]
    Vv = [(m(1, r), m(0, r), m(0, r), m(0, r)) for r in range(4)]
    sa, sb = (1.0, -1.0, 1.0, -1.0), (-1.0, 1.0, -1.0, 1.0)
    inv = [0.0] * 16
    for k in range(4):
        inv[0 + k] = ((Vv[1][k] * F[0][k] - Vv[2][k] * F[1][k]) + Vv[3][k] * F[2][k]) * sa[k]
        inv[4 + k] = ((Vv[0][k] * F[0][k] - Vv[2][k] * F[3][k]) + Vv[3][k] * F[4][k]) * sb[k]
        inv[8 + k] = ((Vv[0][k] * F[1][k] - Vv[1][k] * F[3][k]) + Vv[3][k] * F[5][k]) * sa[k]
        inv[12 + k] = ((Vv[0][k] * F[2][k] - Vv[1][k] * F[4][k]) + Vv[2][k] * F[5][k]) * sb[k]
    d = [m(0, 0) * inv[0], m(0, 1) * inv[4], m(0, 2) * inv[8], m(0, 3) * inv[12]]
    one_over_det = 1.0 / ((d[0] + d[1]) + (d[2] + d[3]))
    return [v * one_over_det for v in inv]


def inv_vp(u):
    """rule 1: ModelMatrix * inverse(ProjectionMatrix * ModelViewMatrix), double from the float uniforms, rounded once"""
    dbl = lambda k: [float(x) for x in np.asarray(u[k], np.float32).reshape(16)]
    r = _mat_mul(dbl("ModelMatrix"), _inverse_glm(_mat_mul(dbl("ProjectionMatrix"), dbl("ModelViewMatrix"))))
    return np.array(r, dtype=np.float32)


def _mul_mat_vec(m, x, y, z, w):
    return [((m[0 + r] * x + m[4 + r] * y) + m[8 + r] * z) + m[12 + r] * w for r in range(4)]


def _unorm8(x):
    x = np.fmin(np.fmax(x, f32(0)), f32(1))
    return np.rint(np.where(np.isnan(x), f32(0), x) * f32(255)).astype(np.uint32)


def view_np(u, tex, level, details=False):
    """rules 2-6 in numpy float32, every operation rounded to binary32 as the kernel does.  tex: the level's texels,
    (N, N, N, 4) uint8 or float16 indexed [z, y, x].  -> rgba (H, W, 4), voxel (H, W), steps (and the rays if details)"""
    W, H, N = int(u["screen_width"]), int(u["screen_height"]), int(u["VoxelDimensions"]) >> level
    G, fN = f32(u["VoxelGridWorldSize"]), f32(N)
    m = inv_vp(u)
    x = (np.arange(W, dtype=np.int64) * 2 + 1).astype(f32) / f32(W) - f32(1)
    y = (np.arange(H, dtype=np.int64) * 2 + 1).astype(f32) / f32(H) - f32(1)
    X, Y = np.meshgrid(x, y)
    with np.errstate(all="ignore"):
        n = _mul_mat_vec(m, X, Y, f32(-1), f32(1))
        fr = _mul_mat_vec(m, X, Y, f32(1), f32(1))
        o = [(n[a] / n[3] / G + f32(0.5)) * fN for a in range(3)]
        e = [(fr[a] / fr[3] / G + f32(0.5)) * fN for a in range(3)]
        d = [e[a] - o[a] for a in range(3)]
        t_in, t_out = np.zeros((H, W), f32), np.ones((H, W), f32)
        face = np.zeros((H, W), np.int64)
        inside = np.ones((H, W), bool)
        iv = []
        for a in range(3):
            fin = np.isfinite(o[a]) & np.isfinite(d[a])
            par = d[a] == 0
            inside &= fin & ~(par & ~((o[a] >= 0) & (o[a] <= fN)))
            ia = np.where(par | ~fin, f32(0), f32(1) / np.where(par, f32(1), d[a]))
            iv.append(ia)
            t0, t1 = (f32(0) - o[a]) * ia, (fN - o[a]) * ia
            lo, hi = np.where(t1 < t0, t1, t0), np.where(t0 < t1, t1, t0)
            lim = fin & ~par
            up = lim & (lo > t_in)
            t_in, face = np.where(up, lo, t_in), np.where(up, a + 1, face)
            t_out = np.where(lim & (hi < t_out), hi, t_out)
        act = inside & (t_in < t_out)
        v = [np.clip(np.floor(o[a] + t_in * d[a]), f32(0), f32(N - 1)).astype(np.int64) for a in range(3)]
        st = [np.sign(d[a]).astype(np.int64) for a in range(3)]
        tm = [np.where(d[a] == 0, f32(np.inf), ((v[a] + (st[a] > 0)).astype(f32) - o[a]) * iv[a]) for a in range(3)]
        td = [np.abs(iv[a]) for a in range(3)]
    bg = int(_unorm8(f32(0.5) if float(u["ambientFactor"]) < 0.5 else f32(1)))
    rgba = np.full((H, W, 4), bg, np.uint8)
    rgba[..., 3] = 255
    vox = np.full((H, W), MISS, np.uint32)
    steps = 0
    shade = np.array([256, 218, 256, 179], np.uint32)
    while act.any():
        steps += int(act.sum())
        jj, ii = np.nonzero(act)
        vx, vy, vz = v[0][jj, ii], v[1][jj, ii], v[2][jj, ii]
        t = tex[vz, vy, vx]
        if t.dtype == np.float16:
            a_ = t[:, 3].astype(f32)
            occ = a_ > 0
            with np.errstate(all="ignore"):
                c = np.stack([_unorm8(t[:, k].astype(f32) / a_) for k in range(3)], 1)
        else:
            al = t[:, 3].astype(np.uint32)
            occ = al > 0
            c = np.minimum(255, (t[:, :3].astype(np.uint32) * 255 + (al // 2)[:, None]) // np.maximum(al, 1)[:, None])
        s = shade[face[jj, ii]][:, None]
        hj, hi_ = jj[occ], ii[occ]
        rgba[hj, hi_, :3] = ((c[occ] * s[occ] + 128) >> 8).astype(np.uint8)
        vox[hj, hi_] = ((vz[occ] * N + vy[occ]) * N + vx[occ]).astype(np.uint32)
        act[hj, hi_] = False
        jj, ii = np.nonzero(act)
        T = [tm[a][jj, ii] for a in range(3)]
        ax = np.where((T[0] <= T[1]) & (T[0] <= T[2]), 0, np.where(T[1] <= T[2], 1, 2))
        for a in range(3):
            sel = ax == a
            sj, si = jj[sel], ii[sel]
            stop = tm[a][sj, si] >= t_out[sj, si]
            nv = v[a][sj, si] + st[a][sj, si]
            stop |= (nv < 0) | (nv >= N)
            act[sj[stop], si[stop]] = False
            gj, gi = sj[~stop], si[~stop]
            v[a][gj, gi] = nv[~stop]
            tm[a][gj, gi] = tm[a][gj, gi] + td[a][gj, gi]
            face[gj, gi] = a + 1
    if details:
        return rgba, vox, steps, {"o": o, "d": d}
    return rgba, vox, steps


# ------------------------------------------------------------------------------------------ scenes for the KATs
def cam_uniforms(V, eye, center, up=(0, 1, 0), size=(65, 65), G=None, far=1000.0, fov=45.0, fmt=0):
    w, h = size
    u = uniforms.reference_uniforms(V=V, width=w, height=h, grid_world=float(G or V), grid_format=fmt)
    u["ModelMatrix"] = gm.colmajor(np.eye(4, dtype=np.float32))
    u["ModelViewMatrix"] = gm.colmajor(gm.look_at(eye, center, up))
    u["ProjectionMatrix"] = gm.colmajor(gm.perspective(gm.radians(fov), np.float32(w) / np.float32(h), 0.1, far))
    return u


def one_voxel_grid(V=16, at=(8, 8, 8), rgb=(200, 100, 50)):
    g = np.zeros((V, V, V, 4), np.uint8)
    x, y, z = at
    g[z, y, x] = (*rgb, 255)
    return g


def reference_view(oracle, u, grid0, level):
    oracle.set_uniforms(u)
    oracle.set_grid_level0(grid0)
    return ref_view(oracle, level)


def shaded(rgb, s):
    return tuple((c * s + 128) >> 8 for c in rgb)


# ------------------------------------------------------------------------------------------ known answers
# voxel (8, 8, 8) of a V = 16 grid with G = 16 covers world [0, 1]^3; the camera looks at its centre along an axis
LEVEL_KAT = [(0, (200, 100, 50, 255), (200, 100, 50)),
             (1, (25, 13, 6, 32), (199, 104, 48)),
             (2, (3, 2, 1, 4), (191, 128, 64)),
             (3, (0, 0, 0, 1), (0, 0, 0))]


@pytest.mark.parametrize("level,texel,shown", LEVEL_KAT)
def test_one_voxel_at_every_level(oracle, level, texel, shown):
    g = one_voxel_grid()
    n = 16 >> level
    t = 8 >> level
    for eye, up, s in (((0.5, 30.0, 0.5), (0, 0, -1), 256), ((0.5, 0.5, 30.0), (0, 1, 0), 179), ((30.0, 0.5, 0.5), (0, 1, 0), 218)):
        u = cam_uniforms(16, eye, (0.5, 0.5, 0.5), up)
        rgba, vox, steps = reference_view(oracle, u, g, level)
        assert tuple(oracle.grid(level)[t, t, t]) == texel
        assert tuple(rgba[32, 32]) == (*shaded(shown, s), 255), (eye, level)
        assert vox[32, 32] == (t * n + t) * n + t
        assert steps > 0


def test_one_voxel_vanishes_at_the_last_level(oracle):
    u = cam_uniforms(16, (0.5, 0.5, 30.0), (0.5, 0.5, 0.5))
    rgba, vox, steps = reference_view(oracle, u, one_voxel_grid(), 4)
    assert tuple(oracle.grid(4)[0, 0, 0]) == (0, 0, 0, 0)
    assert (rgba[..., :3] == 128).all() and (rgba[..., 3] == 255).all() and (vox == MISS).all()
    assert steps > 0     # the rays still visit the one texel


def test_front_face_covers_exactly_the_expected_pixels(oracle):
    """camera 10 units in front of the voxel's +z face on its axis, fov 45 deg, 65 x 65: the face spans NDC
    |x|, |y| < 0.5 / (10 tan 22.5 deg) = 0.1207; pixel centres sit at multiples of 2/65, so the 7 x 7 pixels around the
    centre see the face (|ndc| <= 0.0923) and the next ring (0.1231) does not"""
    u = cam_uniforms(16, (0.5, 0.5, 11.0), (0.5, 0.5, 0.0))
    rgba, vox, _ = reference_view(oracle, u, one_voxel_grid(), 0)
    want = np.zeros((65, 65), bool)
    want[29:36, 29:36] = True
    assert np.array_equal(vox != MISS, want)
    assert (vox[want] == (8 * 16 + 8) * 16 + 8).all()
    assert (rgba[want][:, :3] == shaded((200, 100, 50), 179)).all()
    assert (rgba[~want][:, :3] == 128).all()


def test_exactly_axis_parallel_rays(oracle):
    """the camera on the grid's centre lines x = y = 8 (world 0): the centre pixel's ray has d_x = d_y = 0 exactly and
    runs along the voxel boundary x = y = 8, which floor() assigns to voxel 8"""
    u = cam_uniforms(16, (0.0, 0.0, 30.0), (0.0, 0.0, 0.0))
    _, _, _, ray = view_np(u, one_voxel_grid(), 0, details=True)
    assert ray["d"][0][32, 32] == 0 and ray["d"][1][32, 32] == 0 and ray["o"][0][32, 32] == 8 and ray["o"][1][32, 32] == 8
    rgba, vox, _ = reference_view(oracle, u, one_voxel_grid(at=(8, 8, 8)), 0)
    assert vox[32, 32] == (8 * 16 + 8) * 16 + 8 and tuple(rgba[32, 32, :3]) == shaded((200, 100, 50), 179)
    rgba, vox, _ = reference_view(oracle, u, one_voxel_grid(at=(7, 7, 8)), 0)
    assert vox[32, 32] == MISS                       # the voxel on the other side of the boundary is not on the ray
    u = cam_uniforms(16, (0.0, 0.0, -30.0), (0.0, 0.0, 0.0))   # looking along +z: o_z < 0, parallel in x and y
    rgba, vox, _ = reference_view(oracle, u, one_voxel_grid(at=(8, 8, 8)), 0)
    assert vox[32, 32] == (8 * 16 + 8) * 16 + 8


def test_camera_inside_an_occupied_voxel_sees_it_unshaded(oracle):
    u = cam_uniforms(16, (0.5, 0.5, 0.5), (0.5, 0.5, -1.0), size=(24, 16))
    rgba, vox, steps = reference_view(oracle, u, one_voxel_grid(), 0)
    assert (vox == (8 * 16 + 8) * 16 + 8).all()
    assert (rgba.reshape(-1, 4) == (200, 100, 50, 255)).all()     # face "none": no shading
    assert steps == 24 * 16                                        # one texel per pixel


def test_camera_inside_an_empty_voxel(oracle):
    u = cam_uniforms(16, (0.5, 0.5, 3.5), (0.5, 0.5, 0.0))        # in voxel (8, 8, 11), three empty voxels from the hit
    rgba, vox, _ = reference_view(oracle, u, one_voxel_grid(), 0)
    assert vox[32, 32] == (8 * 16 + 8) * 16 + 8 and tuple(rgba[32, 32, :3]) == shaded((200, 100, 50), 179)
    u1 = dict(u, screen_width=1, screen_height=1, ProjectionMatrix=gm.colmajor(gm.perspective(gm.radians(45.0), 1.0, 0.1, 1000.0)))
    _, vox1, steps1 = reference_view(oracle, u1, one_voxel_grid(), 0)
    assert vox1[0, 0] == (8 * 16 + 8) * 16 + 8 and steps1 == 4    # voxels z = 11, 10, 9, 8


def test_camera_outside_looking_away_sees_background(oracle):
    u = cam_uniforms(16, (0.0, 0.0, 30.0), (0.0, 0.0, 60.0))
    g = one_voxel_grid()
    for level in range(5):
        rgba, vox, steps = reference_view(oracle, u, g, level)
        assert (rgba.reshape(-1, 4) == (128, 128, 128, 255)).all() and (vox == MISS).all() and steps == 0
    u["ambientFactor"] = 0.7
    rgba, _, _ = reference_view(oracle, u, g, 0)
    assert (rgba.reshape(-1, 4) == 255).all()


def test_far_plane_cuts_a_voxel_off(oracle):
    g = one_voxel_grid()
    near = cam_uniforms(16, (0.5, 0.5, 30.0), (0.5, 0.5, 0.0), far=35.0)
    cut = cam_uniforms(16, (0.5, 0.5, 30.0), (0.5, 0.5, 0.0), far=29.5)    # the face at z = 1 is 29 away, the voxel
    assert reference_view(oracle, near, g, 0)[1][32, 32] != MISS             # spans 29..30: the plane cuts through it
    assert reference_view(oracle, cut, g, 0)[1][32, 32] != MISS
    gone = cam_uniforms(16, (0.5, 0.5, 30.0), (0.5, 0.5, 0.0), far=28.5)
    rgba, vox, _ = reference_view(oracle, gone, g, 0)
    assert (vox == MISS).all() and (rgba[..., :3] == 128).all()


def test_bad_level_is_rejected(oracle):
    oracle.set_uniforms(cam_uniforms(16, (0.5, 0.5, 30.0), (0.5, 0.5, 0.0)))
    for level in (-1, 5):
        with pytest.raises(ValueError):
            ref_view(oracle, level)


# ------------------------------------------------------------------------------------------ numpy == reference
def sparse_grid(V, seed, fmt, density=0.03):
    rng = np.random.default_rng(seed)
    occ = rng.random((V, V, V)) < density
    if fmt == 1:
        g = np.zeros((V, V, V, 4), np.float16)
        g[..., :3] = rng.random((V, V, V, 3)).astype(np.float16)
        g[..., 3] = 1.0
    else:
        g = rng.integers(0, 256, (V, V, V, 4), dtype=np.uint8)
        g[..., 3] = 255
    g[~occ] = 0
    return g


CAMERAS = {   # world units: V = 32 voxels over G = 24, the grid spans [-12, 12]^3
    "outside": dict(eye=(30.0, 17.0, 41.0), center=(0.0, 0.0, 0.0)),
    "inside": dict(eye=(1.3, -2.1, 3.7), center=(-9.0, 4.0, -20.0)),
    "axis": dict(eye=(0.0, 0.0, 40.0), center=(0.0, 0.0, 0.0)),
    "down": dict(eye=(0.1, 50.0, 0.2), center=(0.1, 0.0, 0.2), up=(0, 0, -1)),
}


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("cam", sorted(CAMERAS))
def test_numpy_restatement_equals_the_reference(oracle, fmt, cam):
    V = 32
    u = cam_uniforms(V, size=(53, 37), G=24.0, fmt=fmt, **CAMERAS[cam])
    g = sparse_grid(V, seed=len(cam) * 7 + fmt, fmt=fmt)
    oracle.set_uniforms(u)
    oracle.set_grid_level0(g)
    hits = 0
    for level in range(6):
        rgba, vox, steps = ref_view(oracle, level)
        nr, nv, ns = view_np(u, oracle.grid(level), level)
        assert np.array_equal(rgba, nr), f"{cam} level {level}: rgba differs"
        assert np.array_equal(vox, nv), f"{cam} level {level}: voxel indices differ"
        assert steps == ns, f"{cam} level {level}: steps {steps} vs {ns}"
        hits += int((vox != MISS).sum())
    assert hits > 0


def test_inverse_view_projection_matrix():
    u = cam_uniforms(32, **CAMERAS["outside"])
    m = lambda k: np.asarray(u[k], np.float64).reshape(4, 4).T
    want = m("ModelMatrix") @ np.linalg.inv(m("ProjectionMatrix") @ m("ModelViewMatrix"))
    np.testing.assert_allclose(inv_vp(u).reshape(4, 4).T, want, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------ flythrough --voxels
def _flythrough():
    spec = importlib.util.spec_from_file_location("flythrough", os.path.join(ROOT, "tools", "flythrough.py"))
    fly = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fly)
    return fly


def test_flythrough_voxels_option(capsys):
    fly = _flythrough()
    a = fly.main(["--script", "W*3 M(900,0)", "--dry-run"])
    plain = capsys.readouterr().out
    b = fly.main(["--script", "W*3 M(900,0)", "--dry-run", "--voxels", "2"])
    assert capsys.readouterr().out == plain               # --dry-run prints the same camera path
    assert np.array_equal(a.position, b.position) and a.Yaw == b.Yaw
    with pytest.raises(SystemExit):
        fly.main(["--dry-run", "--voxels", "two"])
