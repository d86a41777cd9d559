"""Python mirror of the reference's `struct Voxel_Cone_Tracing`
(/root/reference/Voxel_Cone_Tracing_Final/Voxel_Cone_Tracing.h:11-252): same field and method names, the
GL calls replaced by calls through the C ABI (include/vct_c_api.h).  The C++ twin is host/Voxel_Cone_Tracing.h.
"""
from __future__ import annotations

import numpy as np

from . import glmath as gm
from . import uniforms as un
from .capi import Context


FORWARD, BACKWARD, LEFT, RIGHT, UP, DOWN = range(6)     # enum Camera_Direction, Camera.h:11-19


class Camera:
    """Camera.h: the LearnOpenGL fly camera the reference steers with W/A/S/D + mouse (main.cpp:100-150).  position,
    Yaw = -90, Pitch = 0, Zoom = 45, MovementSpeed = SPEED = 2.6, MouseSensitivity = SENSITIVITY = 0.1 (Camera.h:21-25,
    50-60); Front / Right / Up from yaw and pitch (UpdateCamera, :131-144)."""

    def __init__(self, position=(0.0, 4.0, 0.0), yaw=-90.0, pitch=0.0, zoom=45.0):
        self.position = np.asarray(position, dtype=np.float32)
        self.WorldUp = np.array([0.0, 1.0, 0.0], dtype=np.float32)
        self.Yaw, self.Pitch, self.Zoom = float(yaw), float(pitch), float(zoom)
        self.MovementSpeed, self.MouseSensitivity = 2.6, 0.1
        self.UpdateCamera()

    def UpdateCamera(self):
        y, p = np.radians(np.float32(self.Yaw)), np.radians(np.float32(self.Pitch))
        front = np.array([np.cos(y) * np.cos(p), np.sin(p), np.sin(y) * np.cos(p)], dtype=np.float32)
        self.Front = front / np.linalg.norm(front)
        right = np.cross(self.Front, self.WorldUp)
        self.Right = (right / np.linalg.norm(right)).astype(np.float32)
        up = np.cross(self.Right, self.Front)
        self.Up = (up / np.linalg.norm(up)).astype(np.float32)

    def GetViewMatrix(self):
        return gm.view_matrix(self.position, self.Yaw, self.Pitch)

    def ProcessKeyBoard(self, direction, deltaTime):
        """Camera.h:80-101 (W / S / A / D in main.cpp:136-143; UP and DOWN exist in the enum but no key is bound to them):
        move by MovementSpeed * deltaTime"""
        step = np.float32(self.MovementSpeed * deltaTime)
        axis, sign = {FORWARD: (self.Front, 1), BACKWARD: (self.Front, -1), LEFT: (self.Right, -1), RIGHT: (self.Right, 1),
                      UP: (self.WorldUp, 1), DOWN: (self.WorldUp, -1)}[direction]
        self.position = (self.position + sign * step * axis).astype(np.float32)

    def ProcessMouseMovement(self, xOffset, yOffset, constrainPitch=True):
        """Camera.h:103-119: offsets scaled by MouseSensitivity; pitch kept inside +-89 degrees"""
        self.Yaw += xOffset * self.MouseSensitivity
        self.Pitch += yOffset * self.MouseSensitivity
        if constrainPitch:
            self.Pitch = min(max(self.Pitch, -89.0), 89.0)
        self.UpdateCamera()

    def ProcessMouseScroll(self, yOffset):
        """Camera.h:121-129: Zoom (the field of view, in degrees) kept inside [1, 45]"""
        self.Zoom = min(max(self.Zoom - float(yOffset), 1.0), 45.0)


class Voxel_Cone_Tracing:
    def __init__(self, screen_width=1280, screen_height=720, window=None, device=0, VoxelDimensions=128,
                 camera=None):
        # Global Properties (Voxel_Cone_Tracing.h:14-17)
        self.lightDirection = np.array([0.0, 1.0, 0.25], dtype=np.float32)
        self.VoxelDimensions = int(VoxelDimensions)      # const int 128 in the reference; runtime here
        self.VoxelGridWorldSize = 150.0
        self.window = window                             # ignored: headless
        self.screen_width, self.screen_height = int(screen_width), int(screen_height)
        self.ShadowMapSize = 4096                        # :35
        self.AmbientFactor = 0.1                         # :53
        self.CoveragePolicy = "msaa4"                    # 4x MSAA window, main.cpp:30
        self.ConeSet = "6+1"
        self.Bounces = 2
        self.camera = camera or Camera()                 # global `camera`, :8
        self.model = None                                # Model model, :48
        self.ctx = Context(device)                       # opaque device handle replaces the GL object ids
        self.DepthViewProjectionMatrix = self.ProjX = self.ProjY = self.ProjZ = None

    # Voxel_Cone_Tracing.h:67-140
    def init_voxel_cone_tracing(self, model):
        """`model` is a scenes.Scene (replaces Model("...sponza.obj"), :77)."""
        self.model = model
        c = self.ctx
        c.set_i("ShadowMapSize", self.ShadowMapSize)
        c.set_i("VoxelDimensions", self.VoxelDimensions)
        c.set_f("VoxelGridWorldSize", self.VoxelGridWorldSize)
        light = self.lightDirection
        self.DepthViewProjectionMatrix = gm.ortho(-120, 120, -120, 120, -100, 100) @ gm.look_at(light, (0, 0, 0), (0, 1, 0))
        size = np.float32(self.VoxelGridWorldSize)
        vp = gm.ortho(-size * 0.5, size * 0.5, -size * 0.5, size * 0.5, size * 0.5, size * 1.5)
        self.ProjX = vp @ gm.look_at((size, 0, 0), (0, 0, 0), (0, 1, 0))
        self.ProjY = vp @ gm.look_at((0, size, 0), (0, 0, 0), (0, 0, -1))
        self.ProjZ = vp @ gm.look_at((0, 0, size), (0, 0, 0), (0, 1, 0))
        c.load_scene(model)
        self.DrawDepthTexture()
        self.DrawVoxelTexture()

    def _model_matrix(self):
        return gm.scale(0.05)      # :183, :204, :240

    # Voxel_Cone_Tracing.h:192-211
    def DrawDepthTexture(self):
        c = self.ctx
        mMat = self._model_matrix()
        c.set_mat4("DepthModelViewProjectionMatrix", gm.colmajor((self.DepthViewProjectionMatrix @ mMat).astype(np.float32)))
        c.draw_depth()

    # Voxel_Cone_Tracing.h:213-250
    def DrawVoxelTexture(self):
        c = self.ctx
        c.set_i("VoxelDimensions", self.VoxelDimensions)
        c.set_mat4("ProjX", gm.colmajor(self.ProjX))
        c.set_mat4("ProjY", gm.colmajor(self.ProjY))
        c.set_mat4("ProjZ", gm.colmajor(self.ProjZ))
        c.set_i("ShadowMap", 5)
        c.set_i("VoxelTexture", 6)
        mMat = self._model_matrix()
        c.set_mat4("ModelMatrix", gm.colmajor(mMat))
        c.set_mat4("DepthModelViewProjectionMatrix", gm.colmajor((self.DepthViewProjectionMatrix @ mMat).astype(np.float32)))
        c.set_i("ShadowMapSize", self.ShadowMapSize)
        c.set_i("CoveragePolicy", un.COVERAGE[self.CoveragePolicy])
        c.set_i("Bounces", self.Bounces)
        c.draw_voxels()

    def _set_render_uniforms(self):
        c = self.ctx
        c.set_i("screen_width", self.screen_width)
        c.set_i("screen_height", self.screen_height)
        vMat = self.camera.GetViewMatrix()
        pMat = gm.perspective(gm.radians(self.camera.Zoom), np.float32(self.screen_width) / np.float32(self.screen_height), 0.1, 1000.0)
        c.set_3f("CameraPosition", self.camera.position)
        c.set_3f("LightDirection", self.lightDirection)
        c.set_f("VoxelGridWorldSize", self.VoxelGridWorldSize)
        c.set_i("VoxelDimensions", self.VoxelDimensions)
        c.set_f("ambientFactor", self.AmbientFactor)
        c.set_i("ShadowMapSize", self.ShadowMapSize)
        c.set_i("ShadowMap", 5)
        c.set_i("VoxelTexture", 6)
        mMat = self._model_matrix()
        c.set_mat4("ModelMatrix", gm.colmajor(mMat))
        c.set_mat4("ModelViewMatrix", gm.colmajor((vMat @ mMat).astype(np.float32)))
        c.set_mat4("ProjectionMatrix", gm.colmajor(pMat))
        c.set_mat4("DepthModelViewProjectionMatrix", gm.colmajor((self.DepthViewProjectionMatrix @ mMat).astype(np.float32)))
        dirs, wts = un.cone_set(self.ConeSet)
        c.set_cones(dirs, wts)

    # Voxel_Cone_Tracing.h:146-190.  `out`: optional host buffer (numpy / pinned torch tensor) for the frame.
    def Render(self, out=None):
        self._set_render_uniforms()
        self.ctx.render(out)

    def RenderVoxels(self, level, out=None):
        """Voxel view (no reference counterpart): mip `level` of the current pyramid drawn as cubes from the camera of
        Render, into the frame buffer and, if given, `out`."""
        self._set_render_uniforms()
        self.ctx.render_voxels(level, out)

    def BakeProbes(self, xyz):
        """Irradiance probes (no reference counterpart): indirect light and occlusion of the current pyramid at the
        (n, 3) world points `xyz` for a surface facing +X, -X, +Y, -Y, +Z, -Z, with the cone table of Render.  Returns
        (n, 6, 4) float32 (r, g, b, occlusion) and (n, 6) uint32 textureLod calls."""
        self._set_render_uniforms()
        return self.ctx.bake_probes(xyz)

    def CastRays(self, level, a, b):
        """Ray casts (no reference counterpart): the first occupied texel of mip `level` of the current pyramid along each
        world-space segment a[i] -> b[i] ((n, 3) each).  Returns (voxel, t, face, rgba, steps) as Context.cast_rays."""
        self._set_render_uniforms()   # VoxelGridWorldSize; the camera uniforms it also sets have no effect on a cast
        seg = np.concatenate([np.asarray(a, np.float32).reshape(-1, 3), np.asarray(b, np.float32).reshape(-1, 3)], 1)
        return self.ctx.cast_rays(level, seg)

    def Frame(self, out=None):
        """DrawVoxelTexture + Render in one call (what 'full frames/s' times)."""
        self._set_render_uniforms()
        self.ctx.frame(out)
