"""Uniform values exactly as the reference's host code computes them.

Follows /root/reference/Voxel_Cone_Tracing_Final/Voxel_Cone_Tracing.h:
  :84-86   DepthViewProjectionMatrix = ortho(-120,120,-120,120,-100,100) * lookAt(lightDirection, 0, +Y)
  :128-134 ProjX/Y/Z = ortho(-G/2, G/2, -G/2, G/2, G/2, 3G/2) * lookAt(G*axis, 0, up)
  :161-162 view = camera.GetViewMatrix(); proj = perspective(radians(Zoom), w/h, 0.1, 1000)
  :183     ModelMatrix = scale(0.05)
Keys are the GLSL uniform names the reference passes to Shader::set* (Shader.h:362-417); extra keys
(cone table, apertures, ...) are the constants the reference hard-codes in VoxelConeTracing.fs:43-57.
"""
from __future__ import annotations

import numpy as np

from . import glmath as gm

COVERAGE = {"center": 0, "msaa4": 1, "conservative": 2}

# VoxelConeTracing.fs:48-57
REFERENCE_CONE_DIRECTIONS = np.array([
    [0.0, 0.0, 1.0], [0.0, 0.866025, 0.5], [0.823639, 0.267617, 0.5],
    [0.509037, -0.700629, 0.5], [-0.509037, -0.700629, 0.5], [-0.823639, 0.267617, 0.5]], dtype=np.float32)
REFERENCE_CONE_WEIGHTS = np.array([0.25, 0.15, 0.15, 0.15, 0.15, 0.15], dtype=np.float32)


def cone_set(kind="6+1"):
    """'6+1' = the reference's table; '5+1' = BASELINE config 2 wording (the five 60-degree cones,
    weights renormalised to 1); '9+1' = config 3 extension (normal + 8 at 60 degrees); '16+1' = the largest
    table the library takes (normal at 0.1 + 15 at 60 degrees at 0.06 each)."""
    if kind == "6+1":
        return REFERENCE_CONE_DIRECTIONS.copy(), REFERENCE_CONE_WEIGHTS.copy()
    if kind == "5+1":
        return REFERENCE_CONE_DIRECTIONS[1:].copy(), np.full(5, 0.2, dtype=np.float32)
    ring = {"9+1": (8, 0.2, 0.1), "16+1": (15, 0.1, 0.06)}
    if kind in ring:
        n, w0, w1 = ring[kind]
        a = np.arange(n) * (2 * np.pi / n)
        d = np.concatenate([[[0, 0, 1]], np.stack([0.866025 * np.cos(a), 0.866025 * np.sin(a), np.full(n, 0.5)], 1)])
        w = np.concatenate([[w0], np.full(n, w1)])
        return d.astype(np.float32), w.astype(np.float32)
    raise ValueError(kind)


def reference_uniforms(V=128, width=1280, height=720, shadow_map_size=4096, grid_world=150.0,
                       light_direction=(0.0, 1.0, 0.25), camera_pos=(0.0, 4.0, 0.0), yaw=-90.0, pitch=0.0,
                       fov_deg=45.0, model_scale=0.05, ambient=0.1, cones="6+1", coverage="msaa4",
                       bounces=2, grid_format=0):
    G = np.float32(grid_world)
    model = gm.scale(model_scale)
    light = np.asarray(light_direction, dtype=np.float32)
    depth_vp = gm.ortho(-120, 120, -120, 120, -100, 100) @ gm.look_at(light, (0, 0, 0), (0, 1, 0))
    vp = gm.ortho(-G * 0.5, G * 0.5, -G * 0.5, G * 0.5, G * 0.5, G * 1.5)
    projx = vp @ gm.look_at((G, 0, 0), (0, 0, 0), (0, 1, 0))
    projy = vp @ gm.look_at((0, G, 0), (0, 0, 0), (0, 0, -1))
    projz = vp @ gm.look_at((0, 0, G), (0, 0, 0), (0, 1, 0))
    view = gm.view_matrix(camera_pos, yaw, pitch)
    proj = gm.perspective(gm.radians(fov_deg), np.float32(width) / np.float32(height), 0.1, 1000.0)
    dirs, wts = cone_set(cones)
    f32 = lambda m: np.asarray(m, dtype=np.float32)
    return {
        "VoxelDimensions": int(V), "VoxelGridWorldSize": float(G), "ShadowMapSize": int(shadow_map_size),
        "screen_width": int(width), "screen_height": int(height),
        "ModelMatrix": gm.colmajor(model), "ModelViewMatrix": gm.colmajor(f32(view @ model)),
        "ProjectionMatrix": gm.colmajor(proj),
        "DepthModelViewProjectionMatrix": gm.colmajor(f32(depth_vp @ model)),
        "ProjX": gm.colmajor(projx), "ProjY": gm.colmajor(projy), "ProjZ": gm.colmajor(projz),
        "CameraPosition": f32(camera_pos), "LightDirection": light, "ambientFactor": float(ambient),
        "ConeDirections": dirs, "ConeWeights": wts,
        "DiffuseTanHalfAngle": 0.577, "SpecularTanHalfAngle": 0.07, "StepMultiplier": 1.0,
        "MaxDistance": 75.0, "MaxAlpha": 0.95, "PcfRadius": 2, "ShadowBias": 0.002,
        "CoveragePolicy": COVERAGE[coverage] if isinstance(coverage, str) else int(coverage),
        "Bounces": int(bounces), "GridFormat": int(grid_format),
    }


def scene_uniforms(scene, **kw):
    kw.setdefault("camera_pos", scene.camera_pos)
    kw.setdefault("yaw", scene.yaw)
    kw.setdefault("pitch", scene.pitch)
    kw.setdefault("fov_deg", scene.fov_deg)
    return reference_uniforms(**kw)
