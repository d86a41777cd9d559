"""Ray casts (vct_cast_rays, DESIGN.md section 3 "Ray casts") on the CPU: hand-derived known answers on the C++ reference
(tests/raycast_ref.cpp, fed with the oracle's parameters and mip pyramid), an independent numpy float32 restatement of
the rule that must agree with it in every output, and the view as a special case: segments built from the view's
per-pixel near and far points give the texels, step count and (shaded) pixels of the view's own reference
(tests/voxel_view_ref.cpp), which shares no code with the cast reference.  The device is held to the
reference in tests/test_gpu_raycast.py."""
import numpy as np
import pytest

from test_voxel_view import (MISS, _mul_mat_vec, _unorm8, cam_uniforms, inv_vp, one_voxel_grid, reference_view,
                             sparse_grid)
from raycast_ref import cast_rays as ref_cast

f32 = np.float32
PX, NX, PY, NY, PZ, NZ = 1, 2, 3, 4, 5, 6
SHADE = np.array([256, 218, 256, 179], np.uint32)      # by entry axis: none, X, Y, Z (the view's face shading)


def seg(a, b):
    return np.array([[*a, *b]], np.float32)


def one_voxel_oracle(oracle, V=16, fmt=0):
    """voxel (8, 8, 8) of (200, 100, 50) in a V = 16 grid with G = 16: world x maps to texel x + 8"""
    oracle.set_uniforms(cam_uniforms(V, (0.5, 0.5, 30.0), (0.5, 0.5, 0.5), fmt=fmt))
    oracle.set_grid_level0(one_voxel_grid(V))
    return oracle


def cast1(oracle, level, a, b):
    voxel, t, face, rgba, steps = ref_cast(oracle, level, seg(a, b))
    return int(voxel[0]), float(t[0]), int(face[0]), tuple(int(x) for x in rgba[0]), int(steps[0])


# ------------------------------------------------------------------------------------------ known answers
HIT = (8 * 16 + 8) * 16 + 8


def test_segment_along_x_enters_the_voxel_half_way(oracle):
    one_voxel_oracle(oracle)
    assert cast1(oracle, 0, (-8, .5, .5), (8, .5, .5)) == (HIT, 0.5, NX, (200, 100, 50, 255), 9)
    voxel, t, face, rgba, steps = cast1(oracle, 0, (8, .5, .5), (-8, .5, .5))
    assert (voxel, face, rgba) == (HIT, PX, (200, 100, 50, 255))
    assert t == 7 / 16 and steps == 8                    # texels x = 15 .. 8, entered through the plane x = 9


@pytest.mark.parametrize("level,rgb,alpha", [(1, (199, 104, 48), 32), (2, (191, 128, 64), 4), (3, (0, 0, 0), 1)])
def test_coarse_levels_hit_the_parent_texel(oracle, level, rgb, alpha):
    one_voxel_oracle(oracle)
    n, p = 16 >> level, 8 >> level
    voxel, t, face, rgba, steps = cast1(oracle, level, (-8, .5, .5), (8, .5, .5))
    assert voxel == (p * n + p) * n + p and face == NX and rgba == (*rgb, alpha)
    assert t == p / n and steps == p + 1


def test_the_voxel_vanishes_at_the_last_level(oracle):
    one_voxel_oracle(oracle)
    assert cast1(oracle, 4, (-8, .5, .5), (8, .5, .5)) == (MISS, np.inf, 0, (0, 0, 0, 0), 1)


@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("sign", [1, -1])
def test_axis_parallel_segments_give_the_matching_face(oracle, axis, sign):
    one_voxel_oracle(oracle)
    a, b = [.5, .5, .5], [.5, .5, .5]
    a[axis], b[axis] = -sign * 8.0, sign * 8.0
    voxel, t, face, rgba, steps = cast1(oracle, 0, a, b)
    assert voxel == HIT and rgba == (200, 100, 50, 255)
    assert face == 2 * axis + (2 if sign > 0 else 1)     # moving +axis enters through the -axis face
    assert t == (0.5 if sign > 0 else 7 / 16)


def test_segment_starting_inside_the_voxel(oracle):
    one_voxel_oracle(oracle)
    assert cast1(oracle, 0, (.5, .5, .5), (7.0, -3.0, 2.0)) == (HIT, 0.0, 0, (200, 100, 50, 255), 1)


def test_segment_ending_on_the_entry_plane_misses(oracle):
    one_voxel_oracle(oracle)
    voxel, t, face, rgba, steps = cast1(oracle, 0, (-8, .5, .5), (0, .5, .5))
    assert (voxel, t, face, rgba) == (MISS, np.inf, 0, (0, 0, 0, 0)) and steps == 8
    assert cast1(oracle, 0, (-8, .5, .5), (0.001, .5, .5))[0] == HIT


def test_point_queries(oracle):
    one_voxel_oracle(oracle)
    for p in ((.5, .5, .5), (0.0, 0.0, 0.0), (.999, .25, .75)):
        assert cast1(oracle, 0, p, p) == (HIT, 0.0, 0, (200, 100, 50, 255), 1)
    for p in ((1.5, .5, .5), (-3.0, 2.0, 6.5), (7.9, 7.9, 7.9)):
        assert cast1(oracle, 0, p, p) == (MISS, np.inf, 0, (0, 0, 0, 0), 1)


def test_segments_outside_the_grid_and_non_finite_miss_without_a_step(oracle):
    one_voxel_oracle(oracle)
    for a, b in (((-20, .5, .5), (-9, .5, .5)), ((9, 9, 9), (30, 40, 50)), ((-30, 30, 0), (30, 30, 0)),
                 ((8.5, 0, 0), (8.5, 0, 0)), ((np.nan, .5, .5), (8, .5, .5)), ((-8, .5, .5), (np.inf, .5, .5)),
                 ((-8, -np.inf, .5), (8, .5, .5))):
        assert cast1(oracle, 0, a, b) == (MISS, np.inf, 0, (0, 0, 0, 0), 0), (a, b)


# ------------------------------------------------------------------------------------------ numpy restatement
def cast_np(tex, G, seg):
    """the rule in numpy float32, every operation rounded to binary32 as the kernel does.  tex: the level's texels,
    (N, N, N, 4) uint8 or float16 indexed [z, y, x].  -> voxel, t, face, rgba, steps"""
    N = tex.shape[0]
    G, fN = f32(G), f32(N)
    s = np.asarray(seg, f32).reshape(-1, 6)
    n = s.shape[0]
    with np.errstate(all="ignore"):
        o = [(s[:, a] / G + f32(0.5)) * fN for a in range(3)]
        e = [(s[:, 3 + a] / G + f32(0.5)) * fN for a in range(3)]
        d = [e[a] - o[a] for a in range(3)]
        t_in, t_out = np.zeros(n, f32), np.ones(n, f32)
        axis = np.zeros(n, np.int64)
        ok = np.ones(n, bool)
        iv = []
        for a in range(3):
            fin = np.isfinite(o[a]) & np.isfinite(d[a])
            par = d[a] == 0
            ok &= fin & ~(par & ~((o[a] >= 0) & (o[a] <= fN)))
            ia = np.where(par | ~fin, f32(0), f32(1) / np.where(par, f32(1), d[a]))
            iv.append(ia)
            t0, t1 = (f32(0) - o[a]) * ia, (fN - o[a]) * ia
            lo, hi = np.where(t1 < t0, t1, t0), np.where(t0 < t1, t1, t0)
            lim = fin & ~par
            up = lim & (lo > t_in)
            t_in, axis = np.where(up, lo, t_in), np.where(up, a + 1, axis)
            t_out = np.where(lim & (hi < t_out), hi, t_out)
        act = ok & (t_in < t_out)
        v = [np.clip(np.floor(np.where(act, o[a] + t_in * d[a], 0)), f32(0), f32(N - 1)).astype(np.int64) for a in range(3)]
        st = [np.sign(np.where(act, d[a], 0)).astype(np.int64) for a in range(3)]
        tm = [np.where(d[a] == 0, f32(np.inf), ((v[a] + (st[a] > 0)).astype(f32) - o[a]) * iv[a]) for a in range(3)]
        td = [np.abs(iv[a]) for a in range(3)]
    t_enter = t_in.copy()
    voxel, t = np.full(n, MISS, np.uint32), np.full(n, np.inf, f32)
    face, rgba, steps = np.zeros(n, np.uint8), np.zeros((n, 4), np.uint8), np.zeros(n, np.uint32)
    while act.any():
        k = np.nonzero(act)[0]
        steps[k] += 1
        tx = tex[v[2][k], v[1][k], v[0][k]]
        if tx.dtype == np.float16:
            al = tx[:, 3].astype(f32)
            occ = al > 0
            with np.errstate(all="ignore"):
                c = np.stack([_unorm8(tx[:, j].astype(f32) / al) for j in range(3)] + [_unorm8(al)], 1)
        else:
            al = tx[:, 3].astype(np.uint32)
            occ = al > 0
            c = np.minimum(255, (tx[:, :3].astype(np.uint32) * 255 + (al // 2)[:, None]) // np.maximum(al, 1)[:, None])
            c = np.concatenate([c, al[:, None]], 1)
        h = k[occ]
        voxel[h] = ((v[2][h] * N + v[1][h]) * N + v[0][h]).astype(np.uint32)
        t[h] = t_enter[h]
        rgba[h] = c[occ].astype(np.uint8)
        ax = axis[h]
        dh = np.choose(np.maximum(ax - 1, 0), [d[0][h], d[1][h], d[2][h]])
        face[h] = np.where(ax == 0, 0, 2 * ax - np.where(dh > 0, 0, 1))
        act[h] = False
        k = np.nonzero(act)[0]
        T = [tm[a][k] for a in range(3)]
        nxt = np.where((T[0] <= T[1]) & (T[0] <= T[2]), 0, np.where(T[1] <= T[2], 1, 2))
        for a in range(3):
            q = k[nxt == a]
            nv = v[a][q] + st[a][q]
            stop = (tm[a][q] >= t_out[q]) | (nv < 0) | (nv >= N)
            act[q[stop]] = False
            g = q[~stop]
            v[a][g] = nv[~stop]
            t_enter[g] = tm[a][g]
            tm[a][g] = tm[a][g] + td[a][g]
            axis[g] = a + 1
    return voxel, t, face, rgba, steps


def segment_mix(V, G, seed, n=4000):
    """crossing the grid, starting inside it, axis-parallel (on texel boundaries too), degenerate, non-finite, and lying
    wholly outside it, shuffled"""
    rng = np.random.default_rng(seed)
    h = f32(G) / 2
    u = lambda lo, hi, k: rng.uniform(lo, hi, (k, 3)).astype(f32)
    parts = [np.concatenate([u(-1.6 * h, 1.6 * h, n), u(-1.6 * h, 1.6 * h, n)], 1),       # crossing (most of them)
             np.concatenate([u(-h, h, n), u(-2 * h, 2 * h, n)], 1)]                         # starting inside
    cell = f32(G) / f32(V)
    a = (rng.integers(-V // 2 - 2, V // 2 + 3, (n, 3)).astype(f32) * cell)                 # texel corners ...
    a[: n // 2] += u(-h / V, h / V, n // 2)                                                 # ... and anywhere
    b = a.copy()
    ax = rng.integers(0, 3, n)
    b[np.arange(n), ax] = rng.uniform(-1.5 * h, 1.5 * h, n).astype(f32)
    two = rng.random(n) < 0.3                                                               # some move along two axes
    b[np.nonzero(two)[0], (ax[two] + 1) % 3] = rng.uniform(-1.5 * h, 1.5 * h, int(two.sum())).astype(f32)
    parts.append(np.concatenate([a, b], 1))
    p = u(-1.1 * h, 1.1 * h, n // 2)
    parts.append(np.concatenate([p, p], 1))                                                 # degenerate: point queries
    bad = np.concatenate([u(-h, h, n // 4), u(-h, h, n // 4)], 1)
    bad[np.arange(n // 4), rng.integers(0, 6, n // 4)] = rng.choice(np.array([np.nan, np.inf, -np.inf], f32), n // 4)
    parts.append(bad)                                                                       # non-finite
    out = np.concatenate([u(1.05 * h, 3 * h, n // 4), u(1.05 * h, 3 * h, n // 4)], 1)
    out[:, [1, 4]] *= -1
    parts.append(out)                                                                       # outside, same side
    s = np.concatenate(parts)
    return s[rng.permutation(s.shape[0])]


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("V", [16, 64])
def test_numpy_restatement_equals_the_reference(oracle, V, fmt):
    G = 24.0
    oracle.set_uniforms(cam_uniforms(V, (30.0, 17.0, 41.0), (0.0, 0.0, 0.0), G=G, fmt=fmt))
    oracle.set_grid_level0(sparse_grid(V, seed=V * 3 + fmt, fmt=fmt, density=0.02))
    segs = segment_mix(V, G, seed=V + 10 * fmt)
    hits, faces = 0, set()
    for level in range(V.bit_length()):
        got = ref_cast(oracle, level, segs)
        want = cast_np(oracle.grid(level), G, segs)
        for name, g, w in zip(("voxel", "t", "face", "rgba", "steps"), got, want):
            assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), \
                f"V={V} fmt={fmt} level {level}: {name} differs on {int((g != w).reshape(len(segs), -1).any(1).sum())}"
        hits += int((got[0] != MISS).sum())
        faces |= set(got[2].tolist())
    assert hits > 1000 and faces == set(range(7))              # every face and "none"


# ------------------------------------------------------------------------------------------ the view as a special case
def pixel_segments(u):
    """each pixel's near and far points, n.xyz / n.w and f.xyz / f.w in float32 as the view computes them"""
    W, H = int(u["screen_width"]), int(u["screen_height"])
    m = inv_vp(u)
    x = (np.arange(W, dtype=np.int64) * 2 + 1).astype(f32) / f32(W) - f32(1)
    y = (np.arange(H, dtype=np.int64) * 2 + 1).astype(f32) / f32(H) - f32(1)
    X, Y = np.meshgrid(x, y)
    n, fr = _mul_mat_vec(m, X, Y, f32(-1), f32(1)), _mul_mat_vec(m, X, Y, f32(1), f32(1))
    with np.errstate(all="ignore"):
        return np.stack([n[0] / n[3], n[1] / n[3], n[2] / n[3], fr[0] / fr[3], fr[1] / fr[3], fr[2] / fr[3]], -1).reshape(-1, 6)


def shaded_pixels(face, rgba):
    s = SHADE[(face.astype(np.int64) + 1) // 2][:, None]
    return ((rgba[:, :3].astype(np.uint32) * s + 128) >> 8).astype(np.uint8)


def assert_view_equivalence(oracle, u, grid0, level):
    vrgba, vvox, vsteps = reference_view(oracle, u, grid0, level)
    voxel, t, face, rgba, steps = ref_cast(oracle, level, pixel_segments(u))
    assert np.array_equal(voxel, vvox.reshape(-1)), f"level {level}: texel maps differ"
    assert int(steps.astype(np.int64).sum()) == vsteps
    hit = voxel != MISS
    assert np.array_equal(shaded_pixels(face[hit], rgba[hit]), vrgba.reshape(-1, 4)[hit, :3])
    assert (rgba[~hit] == 0).all() and (face[~hit] == 0).all() and np.isinf(t[~hit]).all()
    assert ((t[hit] >= 0) & (t[hit] <= 1)).all()
    return int(hit.sum())


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("cam", ["outside", "inside", "axis", "down"])
def test_pixel_segments_reproduce_the_view(oracle, fmt, cam):
    from test_voxel_view import CAMERAS
    V = 32
    u = cam_uniforms(V, size=(53, 37), G=24.0, fmt=fmt, **CAMERAS[cam])
    g = sparse_grid(V, seed=len(cam) * 7 + fmt, fmt=fmt)
    assert sum(assert_view_equivalence(oracle, u, g, level) for level in range(6)) > 0


def test_one_voxel_view_through_pixel_segments(oracle):
    u = cam_uniforms(16, (0.5, 0.5, 11.0), (0.5, 0.5, 0.0))
    assert assert_view_equivalence(oracle, u, one_voxel_grid(), 0) == 49     # the 7 x 7 pixels that see the face
