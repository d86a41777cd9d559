"""Irradiance probes (DESIGN.md section 3 "Irradiance probes"): the face basis, and the CPU reference
(tests/probe_ref.py, composed from the oracle's cone march) against hand-derived answers on uniform and empty grids and
against the float64 cone loop of test_oracle_independent.py."""
import numpy as np
import pytest

from probe_ref import FACES, PROBES_KAT, bake_probes, face_directions, rotated_unnormalised
from test_oracle_independent import G, cone, mip_chain, random_grid
from test_oracle_kat import setup
from vct_b200 import uniforms

CONE_SETS = ("6+1", "5+1", "9+1")


def test_face_basis_is_orthonormal_right_handed_and_in_axis_order():
    axes = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], dtype=np.float32)
    for f in range(6):
        T, B, N = FACES[f].astype(np.float64)
        assert np.array_equal(N, axes[f])
        assert np.array_equal(FACES[f].astype(np.float64) @ FACES[f].T.astype(np.float64), np.eye(3))
        assert np.array_equal(np.cross(T, B), N)


@pytest.mark.parametrize("cones", CONE_SETS)
def test_rotated_directions_are_signed_permutations_of_the_table(cones):
    dirs, _ = uniforms.cone_set(cones)
    v = rotated_unnormalised(dirs)
    for f in range(6):
        M = FACES[f].T.astype(np.float64)                    # columns T, B, N: v = M d, a signed permutation
        assert np.array_equal(v[f].astype(np.float64), dirs.astype(np.float64) @ M.T)
        assert np.array_equal(np.sort(np.abs(v[f]), axis=1), np.sort(np.abs(dirs), axis=1))
    fd = face_directions(dirs)
    np.testing.assert_allclose(np.linalg.norm(fd.astype(np.float64), axis=-1), 1.0, atol=1e-6)
    # +Z is the identity basis: the frame's cones for a surface facing +Z with T = +X, B = +Y
    d64 = dirs.astype(np.float64)
    np.testing.assert_allclose(fd[4], d64 / np.linalg.norm(d64, axis=1, keepdims=True), atol=1e-7)


@pytest.mark.parametrize("V,cones", [(128, "6+1"), (128, "5+1"), (128, "9+1"), (256, "6+1")])
def test_uniform_grid_known_answer(oracle, V, cones):
    setup(oracle, V=V, cones=cones)
    g = np.empty((V, V, V, 4), dtype=np.uint8)
    g[..., :3] = 153
    g[..., 3] = 255
    oracle.set_grid_level0(g)
    out, steps = bake_probes(oracle, PROBES_KAT)
    vws = G / V
    occlusion = 1.0 - 1.0 / (1.0 + 0.03 * max(vws, 2 * 0.577 * vws))
    assert abs(occlusion - {128: 0.038989, 256: 0.019882}[V]) < 1e-6
    np.testing.assert_allclose(out[..., :3], 153 / 255.0, atol=1e-6)
    np.testing.assert_allclose(out[..., 3], occlusion, atol=1e-6)
    n_cones = len(uniforms.cone_set(cones)[1])
    assert np.all(steps == n_cones)                          # alpha reaches 1 at the first sample of every cone


@pytest.mark.parametrize("V,per_cone", [(128, 6), (256, 7)])
def test_empty_grid_known_answer(oracle, V, per_cone):
    setup(oracle, V=V)
    oracle.set_grid_level0(np.zeros((V, V, V, 4), dtype=np.uint8))
    out, steps = bake_probes(oracle, PROBES_KAT)
    assert np.all(out[..., :3] == 0.0) and np.all(out[..., 3] == 1.0)
    assert np.all(steps == 6 * per_cone)                     # SURVEY.md A.5: diffuse cone steps on an empty grid


def test_non_finite_probe_gives_nan_and_no_steps(oracle):
    setup(oracle, V=32)
    oracle.set_grid_level0(random_grid(32, np.random.default_rng(2)))
    xyz = np.array([[1.0, 2.0, 3.0], [np.nan, 0.0, 0.0], [0.0, np.inf, 0.0], [1.0, 2.0, 3.0]], dtype=np.float32)
    out, steps = bake_probes(oracle, xyz)
    assert np.all(np.isnan(out[1:3])) and np.all(steps[1:3] == 0)
    assert np.array_equal(out[0], out[3]) and np.all(np.isfinite(out[0])) and np.all(steps[0] > 0)


@pytest.mark.parametrize("cones", CONE_SETS)
def test_reference_against_float64_cone_loop(oracle, cones):
    """FilterMode 0 (fp32 filter weights) on a random 32^3 grid; the bounds of test_cone_march_against_float64_loop"""
    V = 32
    rng = np.random.default_rng(7 + len(cones))
    u = setup(oracle, V=V, cones=cones)
    u["FilterMode"] = 0
    oracle.set_uniforms(u)
    g = random_grid(V, rng, fill=0.02)
    oracle.set_grid_level0(g)
    levels = mip_chain(g)
    dirs, weights = uniforms.cone_set(cones)
    fd = face_directions(dirs)
    xyz = rng.uniform(-90, 90, (24, 3)).astype(np.float32)        # beyond +-75 the grid repeats
    out, steps = bake_probes(oracle, xyz)
    vws = G / V
    checked = 0
    for i in range(xyz.shape[0]):
        for f in range(6):
            start = xyz[i].astype(np.float64) + FACES[f, 2].astype(np.float64) * vws
            want, n_want, margin = np.zeros(4), 0, 1.0
            for c in range(len(weights)):
                r, n, m = cone(levels, V, start, fd[f, c].astype(np.float64), 0.577)
                want += float(weights[c]) * r
                n_want += n
                margin = min(margin, m)
            if margin < 1e-4:                # a float32/float64 difference could add or drop a whole step here
                continue
            want[3] = 1.0 - want[3]
            assert steps[i, f] == n_want
            assert np.abs(out[i, f] - want).max() < 2e-5 * max(1, n_want), (i, f, out[i, f], want)
            checked += 1
    assert checked > 100
