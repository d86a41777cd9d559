"""CPU reference of the irradiance probes (vct_bake_probes, DESIGN.md section 3 "Irradiance probes"), composed from the
oracle's single-cone march: for a probe p and each face f of +X, -X, +Y, -Y, +Z, -Z, every cone of the table is turned
by the face's basis (T, B, N), starts at p + N * vws and is marched with DiffuseTanHalfAngle; the face's value is the
weighted sum in cone order, (ind.rgb, 1 - ind.a).  The directions, starts and the sum are float32 operations in the
order the device performs them, so the same composition over vct_trace_cones reproduces the device bit for bit."""
import numpy as np

# (T, B, N) per face, in the order +X, -X, +Y, -Y, +Z, -Z; each row right-handed (T x B = N) and orthonormal
FACES = np.array([
    [[0, 0, -1], [0, 1, 0], [1, 0, 0]],
    [[0, 0, 1], [0, 1, 0], [-1, 0, 0]],
    [[1, 0, 0], [0, 0, -1], [0, 1, 0]],
    [[1, 0, 0], [0, 0, 1], [0, -1, 0]],
    [[1, 0, 0], [0, 1, 0], [0, 0, 1]],
    [[-1, 0, 0], [0, 1, 0], [0, 0, -1]],
], dtype=np.float32)

# probes for the known-answer tests: the centre, inside, near the boundary and outside the grid (where it repeats)
PROBES_KAT = np.array([[0.0, 0.0, 0.0], [13.5, -40.25, 70.0], [-74.9, 74.9, 3.0], [120.0, -200.0, 5.5]], dtype=np.float32)


def rotated_unnormalised(cone_dirs):
    """(6, n, 3) float32: d.x T + d.y B + d.z N per face and cone, summed as ((x T + y B) + z N)"""
    d = np.asarray(cone_dirs, dtype=np.float32).reshape(-1, 3)
    T, B, N = FACES[:, None, 0], FACES[:, None, 1], FACES[:, None, 2]
    return (d[None, :, 0:1] * T + d[None, :, 1:2] * B) + d[None, :, 2:3] * N


def face_directions(cone_dirs):
    """(6, n, 3) float32 cone directions per face: IEEE normalize, sqrt((x*x + y*y) + z*z) then three divisions"""
    v = rotated_unnormalised(cone_dirs)
    length = np.sqrt((v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1]) + v[..., 2] * v[..., 2])
    return v / length[..., None]


def face_starts(xyz, grid_world, V):
    """(n, 6, 3) float32 cone start points p + N * vws, vws = VoxelGridWorldSize / VoxelDimensions"""
    vws = np.float32(grid_world) / np.float32(V)
    p = np.asarray(xyz, dtype=np.float32).reshape(-1, 3)
    return p[:, None, :] + FACES[None, :, 2] * vws


def combine(r, weights):
    """r (..., n_cones, 4) single-cone results (rgb, occ) -> (..., 4) (ind.rgb, 1 - ind.a), float32, cone order"""
    w = np.asarray(weights, dtype=np.float32)
    ind = np.zeros(r.shape[:-2] + (4,), dtype=np.float32)
    for c in range(w.shape[0]):
        ind = ind + w[c] * r[..., c, :]
    ind[..., 3] = np.float32(1.0) - ind[..., 3]
    return ind


def oracle_cones(oracle):
    p = oracle.p
    n = p.NumDiffuseCones
    dirs = np.array(p.ConeDirections[:3 * n], dtype=np.float32).reshape(n, 3)
    return dirs, np.array(p.ConeWeights[:n], dtype=np.float32)


def bake_probes(oracle, xyz):
    """(n, 6, 4) float32 values and (n, 6) int64 steps of the probes at xyz, on the oracle's pyramid and uniforms"""
    p = oracle.p
    dirs, weights = oracle_cones(oracle)
    fdirs = face_directions(dirs)
    xyz = np.asarray(xyz, dtype=np.float32).reshape(-1, 3)
    starts = face_starts(xyz, p.VoxelGridWorldSize, p.VoxelDimensions)
    tan = float(np.float32(p.DiffuseTanHalfAngle))
    out = np.full((xyz.shape[0], 6, 4), np.nan, dtype=np.float32)
    steps = np.zeros((xyz.shape[0], 6), dtype=np.int64)
    r = np.zeros((6, dirs.shape[0], 4), dtype=np.float32)
    for i in range(xyz.shape[0]):
        if not np.all(np.isfinite(xyz[i])):
            continue
        for f in range(6):
            for c in range(dirs.shape[0]):
                r[f, c], n = oracle.cone(starts[i, f], fdirs[f, c], tan)
                steps[i, f] += n
        out[i] = combine(r, weights)
    return out, steps
