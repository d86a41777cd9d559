"""ctypes binding of include/vct_c_api.h (libvct_b200.so).  No CPU fallback: if the library is missing
or no CUDA device is present, calls raise."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libvct_b200.so")

PASSES = {"depth": 0, "vox_clear": 1, "vox_cover": 2, "vox_shade": 3, "resolve": 4, "mip": 5,
          "visibility": 6, "cone": 7, "frame": 8, "reinject": 9, "exchange_push": 10, "exchange_merge": 11,
          "voxel_view": 12, "probes": 13, "rays": 14}

# every symbol include/vct_c_api.h declares (tests check the library exports all of them)
SYMBOLS = [
    "vct_create", "vct_destroy", "vct_last_error", "vct_version", "vct_set_i", "vct_set_f", "vct_set_3f",
    "vct_set_mat4", "vct_get_i", "vct_get_f", "vct_set_cones", "vct_upload_texture", "vct_set_material",
    "vct_upload_mesh", "vct_update_positions", "vct_draw_depth", "vct_draw_voxels", "vct_render", "vct_frame", "vct_frame_async", "vct_frame_wait",
    "vct_render_voxels",
    "vct_voxelize_range", "vct_accum_buffer", "vct_resolve_and_mip", "vct_shared_accum_bytes", "vct_set_shared_accum",
    "vct_voxelize_shared", "vct_resolve_shared", "vct_frame_shared_begin", "vct_exchange_stream", "vct_frame_shared_end", "vct_readback_depth", "vct_readback_counts",
    "vct_readback_sums", "vct_readback_grid", "vct_upload_grid_level0", "vct_build_mips", "vct_readback_visibility",
    "vct_readback_frame", "vct_frame_buffer", "vct_cone_samples", "vct_fragment_count", "vct_occupied_voxels", "vct_debug_counter",
    "vct_trace_cones", "vct_bake_probes", "vct_cast_rays", "vct_sample_voxels", "vct_set_stream", "vct_use_own_stream", "vct_sync", "vct_pass_time_us", "vct_kernel_launches", "vct_bench_tex3d",
    "vct_bench_tex3d_format", "vct_bench_atomics", "vct_pass_timeline",
    "vct_comm_init", "vct_comm_destroy", "vct_comm_info", "vct_comm_barrier", "vct_frame_sharded", "vct_frame_sharded_wait",
    "vct_comm_frame_buffer", "vct_create_multi", "vct_comm_init_multi", "vct_frame_sharded_multi",
]

COMM_NO_MULTICAST, COMM_KEEP_SHARES, COMM_ROW_BANDS = 1, 2, 4


class VctError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"vct error {code}: {msg}")
        self.code = code


_lib = None


def load_library(path=None):
    """Loads libvct_b200.so (built by build.py).  Raises if it is missing -- there is no fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(f"{p} not found: run `python voxel-cone-tracing_b200/build.py` (the CUDA "
                                "extension is mandatory, there is no CPU fallback)")
    L = C.CDLL(p)
    L.vct_last_error.restype = C.c_char_p
    L.vct_last_error.argtypes = [C.c_void_p]
    L.vct_version.restype = C.c_char_p
    L.vct_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    vp, i, f, sz, cp = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_char_p
    sig = {
        "vct_destroy": [vp], "vct_set_i": [vp, cp, i], "vct_set_f": [vp, cp, f], "vct_set_3f": [vp, cp, f, f, f],
        "vct_set_mat4": [vp, cp, vp], "vct_get_i": [vp, cp, C.POINTER(i)], "vct_get_f": [vp, cp, C.POINTER(f)],
        "vct_set_cones": [vp, i, vp, vp], "vct_upload_texture": [vp, i, i, i, i, vp],
        "vct_set_material": [vp, i, i, i, i, f], "vct_upload_mesh": [vp, vp, sz, vp, sz, vp],
        "vct_update_positions": [vp, vp, sz, i], "vct_draw_depth": [vp], "vct_draw_voxels": [vp],
        "vct_render": [vp, vp], "vct_render_voxels": [vp, i, vp, vp], "vct_frame": [vp, vp], "vct_frame_async": [vp, vp], "vct_frame_wait": [vp], "vct_voxelize_range": [vp, sz, sz, i],
        "vct_accum_buffer": [vp, C.POINTER(vp), C.POINTER(sz)], "vct_resolve_and_mip": [vp],
        "vct_shared_accum_bytes": [vp, C.POINTER(sz)], "vct_set_shared_accum": [vp, vp, vp],
        "vct_voxelize_shared": [vp, sz, sz], "vct_resolve_shared": [vp],
        "vct_frame_shared_begin": [vp, sz, sz], "vct_exchange_stream": [vp, C.POINTER(C.c_void_p)],
        "vct_frame_shared_end": [vp, C.c_void_p],
        "vct_readback_depth": [vp, vp], "vct_readback_counts": [vp, vp], "vct_readback_sums": [vp, vp],
        "vct_readback_grid": [vp, i, vp], "vct_upload_grid_level0": [vp, vp], "vct_build_mips": [vp],
        "vct_readback_visibility": [vp, vp], "vct_readback_frame": [vp, vp],
        "vct_frame_buffer": [vp, C.POINTER(vp), C.POINTER(sz)], "vct_cone_samples": [vp, C.POINTER(C.c_uint64)],
        "vct_fragment_count": [vp, C.POINTER(C.c_uint64)], "vct_occupied_voxels": [vp, C.POINTER(C.c_uint64)], "vct_debug_counter": [vp, i, C.POINTER(C.c_uint64)],
        "vct_trace_cones": [vp, sz, vp, vp, vp, vp, vp], "vct_bake_probes": [vp, sz, vp, vp, vp, i], "vct_cast_rays": [vp, i, sz, vp, vp, vp, vp, vp, vp, i], "vct_sample_voxels": [vp, sz, vp, vp, vp], "vct_set_stream": [vp, vp], "vct_use_own_stream": [vp], "vct_sync": [vp], "vct_pass_time_us": [vp, i, C.POINTER(f)],
        "vct_kernel_launches": [vp, C.POINTER(C.c_uint64)],
        "vct_bench_tex3d": [vp, i, C.c_uint64, i, f, i, C.POINTER(f)],
        "vct_bench_tex3d_format": [vp, i, i, C.c_uint64, i, f, i, C.POINTER(f)],
        "vct_bench_atomics": [vp, C.c_uint64, i, C.POINTER(f)],
        "vct_pass_timeline": [vp, i, i, C.POINTER(f), C.POINTER(f)],
        "vct_comm_init": [vp, i, i, cp, i], "vct_comm_destroy": [vp],
        "vct_comm_info": [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(sz)], "vct_comm_barrier": [vp],
        "vct_frame_sharded": [vp, vp], "vct_frame_sharded_wait": [vp],
        "vct_comm_frame_buffer": [vp, C.POINTER(vp), C.POINTER(sz)],
        "vct_create_multi": [C.POINTER(i), i, C.POINTER(vp)], "vct_comm_init_multi": [C.POINTER(vp), i, i],
        "vct_frame_sharded_multi": [C.POINTER(vp), i, vp],
    }
    for name, argtypes in sig.items():
        fn = getattr(L, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    if path is None:
        _lib = L
    return L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """Thin object wrapper over a vct_handle."""

    def __init__(self, device=0, handle=None):
        self.L = load_library()
        if handle is not None:          # adopt a handle made by vct_create_multi
            self.h, self.device = handle, device
            return
        h = C.c_void_p()
        rc = self.L.vct_create(int(device), C.byref(h))
        if rc:
            raise VctError(rc, self.L.vct_last_error(None).decode())
        self.h = h
        self.device = device

    def _ck(self, rc):
        if rc:
            raise VctError(rc, self.L.vct_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.vct_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- uniforms
    def set_i(self, name, v):
        self._ck(self.L.vct_set_i(self.h, name.encode(), int(v)))

    def set_f(self, name, v):
        self._ck(self.L.vct_set_f(self.h, name.encode(), float(v)))

    def set_3f(self, name, v):
        self._ck(self.L.vct_set_3f(self.h, name.encode(), float(v[0]), float(v[1]), float(v[2])))

    def set_mat4(self, name, m16):
        a = np.ascontiguousarray(m16, dtype=np.float32).reshape(16)
        self._ck(self.L.vct_set_mat4(self.h, name.encode(), _ptr(a)))

    def get_i(self, name):
        v = C.c_int()
        self._ck(self.L.vct_get_i(self.h, name.encode(), C.byref(v)))
        return v.value

    def get_f(self, name):
        v = C.c_float()
        self._ck(self.L.vct_get_f(self.h, name.encode(), C.byref(v)))
        return v.value

    def set_cones(self, dirs, weights):
        d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        w = np.ascontiguousarray(weights, dtype=np.float32).reshape(-1)
        assert d.shape[0] == w.shape[0]
        self._ck(self.L.vct_set_cones(self.h, d.shape[0], _ptr(d), _ptr(w)))

    _INT = {"VoxelDimensions", "ShadowMapSize", "screen_width", "screen_height", "PcfRadius", "CoveragePolicy",
            "Bounces", "GridFormat", "MaxFragments", "MaxTileItems", "DenseResolve", "Profile", "RowBegin", "RowEnd",
            "RowInterleave", "RowPhase"}
    _VEC3 = {"CameraPosition", "LightDirection"}
    _MAT4 = {"ModelMatrix", "ModelViewMatrix", "ProjectionMatrix", "DepthModelViewProjectionMatrix", "ProjX",
             "ProjY", "ProjZ"}

    def set_uniforms(self, u: dict):
        """dict keyed by the GLSL uniform names (see uniforms.reference_uniforms)."""
        if "ConeDirections" in u:
            self.set_cones(u["ConeDirections"], u["ConeWeights"])
        for k, v in u.items():
            if k in ("ConeDirections", "ConeWeights"):
                continue
            if k in self._INT:
                self.set_i(k, v)
            elif k in self._VEC3:
                self.set_3f(k, v)
            elif k in self._MAT4:
                self.set_mat4(k, v)
            else:
                self.set_f(k, v)

    # ---- scene
    def upload_texture(self, tex_id, t):
        t = np.ascontiguousarray(t, dtype=np.uint8)
        h, w = t.shape[:2]
        ch = 1 if t.ndim == 2 else t.shape[2]
        self._ck(self.L.vct_upload_texture(self.h, int(tex_id), w, h, ch, _ptr(t)))

    def set_material(self, mat, diffuse, specular, height, shininess=20.0):
        self._ck(self.L.vct_set_material(self.h, int(mat), int(diffuse), int(specular), int(height), float(shininess)))

    def upload_mesh(self, verts14, idx, tri_material=None):
        v = np.ascontiguousarray(verts14, dtype=np.float32).reshape(-1, 14)
        ix = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 3)
        tm = None if tri_material is None else np.ascontiguousarray(tri_material, dtype=np.uint16)
        self._ck(self.L.vct_upload_mesh(self.h, _ptr(v), v.shape[0], _ptr(ix), ix.shape[0],
                                        None if tm is None else _ptr(tm)))

    def load_scene(self, scene):
        for i, t in enumerate(scene.textures):
            self.upload_texture(i, t)
        for i, m in enumerate(scene.materials):
            self.set_material(i, *m)
        self.upload_mesh(scene.verts, scene.idx, scene.tri_material)

    def update_positions(self, xyz=None, n_verts=None, device_ptr=None):
        if device_ptr is not None:
            self._ck(self.L.vct_update_positions(self.h, C.c_void_p(int(device_ptr)), int(n_verts), 1))
        else:
            a = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
            self._ck(self.L.vct_update_positions(self.h, _ptr(a), a.shape[0], 0))

    # ---- passes
    def draw_depth(self):
        self._ck(self.L.vct_draw_depth(self.h))

    def draw_voxels(self):
        self._ck(self.L.vct_draw_voxels(self.h))

    def render(self, out=None):
        self._ck(self.L.vct_render(self.h, None if out is None else _host_ptr(out)))

    def frame(self, out=None):
        self._ck(self.L.vct_frame(self.h, None if out is None else _host_ptr(out)))

    def render_voxels(self, level, out=None, voxel=None):
        """Voxel view of mip `level` from the render camera into the frame buffer.  `out`: optional host buffer for the
        (H, W, 4) uint8 view, `voxel`: optional host buffer for the (H, W) uint32 texel indices (0xFFFFFFFF = miss);
        with neither the call stays on the device and is asynchronous."""
        self._ck(self.L.vct_render_voxels(self.h, int(level), None if out is None else _host_ptr(out),
                                          None if voxel is None else _host_ptr(voxel)))

    def frame_async(self, out):
        """Pipelined frame: renders and queues the copy into `out` (pinned host buffer); see frame_wait()."""
        self._ck(self.L.vct_frame_async(self.h, _host_ptr(out)))

    def frame_wait(self):
        self._ck(self.L.vct_frame_wait(self.h))

    def voxelize_range(self, tb, te, clear_first=True):
        self._ck(self.L.vct_voxelize_range(self.h, int(tb), int(te), int(bool(clear_first))))

    def accum_buffer(self):
        p, n = C.c_void_p(), C.c_size_t()
        self._ck(self.L.vct_accum_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def resolve_and_mip(self):
        self._ck(self.L.vct_resolve_and_mip(self.h))

    # fused sharded voxelisation over a symmetric (optionally multicast-mapped) accumulator
    def shared_accum_bytes(self):
        n = C.c_size_t()
        self._ck(self.L.vct_shared_accum_bytes(self.h, C.byref(n)))
        return n.value

    def set_shared_accum(self, local_ptr, multicast_ptr=0):
        self._ck(self.L.vct_set_shared_accum(self.h, C.c_void_p(int(local_ptr)), C.c_void_p(int(multicast_ptr)) if multicast_ptr else None))

    def voxelize_shared(self, tb, te):
        self._ck(self.L.vct_voxelize_shared(self.h, int(tb), int(te)))

    def resolve_shared(self):
        self._ck(self.L.vct_resolve_shared(self.h))

    def frame_shared_begin(self, tb, te):
        self._ck(self.L.vct_frame_shared_begin(self.h, int(tb), int(te)))

    def exchange_stream(self):
        s = C.c_void_p()
        self._ck(self.L.vct_exchange_stream(self.h, C.byref(s)))
        return int(s.value or 0)

    def frame_shared_end(self, host_rgba=None):
        self._ck(self.L.vct_frame_shared_end(self.h, None if host_rgba is None else _host_ptr(host_rgba)))

    # ---- multi-GPU owned by the library (vct_comm.cu)
    def comm_init(self, rank, world, session, flags=0):
        self._ck(self.L.vct_comm_init(self.h, int(rank), int(world), str(session).encode(), int(flags)))

    def comm_destroy(self):
        self._ck(self.L.vct_comm_destroy(self.h))

    def comm_info(self):
        r, w, m, n = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
        self._ck(self.L.vct_comm_info(self.h, C.byref(r), C.byref(w), C.byref(m), C.byref(n)))
        return {"rank": r.value, "world": w.value, "multicast": bool(m.value), "segment_bytes": n.value}

    def comm_barrier(self):
        self._ck(self.L.vct_comm_barrier(self.h))

    def frame_sharded(self, host_rgba=None):
        self._ck(self.L.vct_frame_sharded(self.h, None if host_rgba is None else _host_ptr(host_rgba)))

    def frame_sharded_wait(self):
        self._ck(self.L.vct_frame_sharded_wait(self.h))

    def comm_frame_buffer(self):
        p, n = C.c_void_p(), C.c_size_t()
        self._ck(self.L.vct_comm_frame_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    # ---- read-back
    def depth(self):
        S = self.get_i("ShadowMapSize")
        a = np.empty((S, S), dtype=np.uint32)
        self._ck(self.L.vct_readback_depth(self.h, _ptr(a)))
        return a

    def counts(self):
        V = self.get_i("VoxelDimensions")
        a = np.empty((V, V, V), dtype=np.uint32)
        self._ck(self.L.vct_readback_counts(self.h, _ptr(a)))
        return a

    def sums(self):
        V = self.get_i("VoxelDimensions")
        a = np.empty((V, V, V, 3), dtype=np.uint32)
        self._ck(self.L.vct_readback_sums(self.h, _ptr(a)))
        return a

    def grid(self, level=0):
        n = self.get_i("VoxelDimensions") >> level
        a = np.empty((n, n, n, 4), dtype=np.float16 if self.get_i("GridFormat") == 1 else np.uint8)
        self._ck(self.L.vct_readback_grid(self.h, int(level), _ptr(a)))
        return a

    def upload_grid_level0(self, rgba, build_mips=True):
        a = np.ascontiguousarray(rgba, dtype=np.float16 if self.get_i("GridFormat") == 1 else np.uint8)
        V = self.get_i("VoxelDimensions")
        assert a.size == V ** 3 * 4
        self._ck(self.L.vct_upload_grid_level0(self.h, _ptr(a)))
        if build_mips:
            self._ck(self.L.vct_build_mips(self.h))

    def build_mips(self):
        self._ck(self.L.vct_build_mips(self.h))

    def visibility(self):
        a = np.empty((self.get_i("screen_height"), self.get_i("screen_width")), dtype=np.uint32)
        self._ck(self.L.vct_readback_visibility(self.h, _ptr(a)))
        return a

    def read_frame(self):
        a = np.empty((self.get_i("screen_height"), self.get_i("screen_width"), 4), dtype=np.uint8)
        self._ck(self.L.vct_readback_frame(self.h, _ptr(a)))
        return a

    def frame_buffer(self):
        p, n = C.c_void_p(), C.c_size_t()
        self._ck(self.L.vct_frame_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def _u64(self, fn):
        v = C.c_uint64()
        self._ck(fn(self.h, C.byref(v)))
        return v.value

    def cone_samples(self):
        return self._u64(self.L.vct_cone_samples)

    def fragment_count(self):
        return self._u64(self.L.vct_fragment_count)

    def occupied_voxels(self):
        return self._u64(self.L.vct_occupied_voxels)

    def debug_counter(self, which=0):
        v = C.c_uint64()
        self._ck(self.L.vct_debug_counter(self.h, int(which), C.byref(v)))
        return v.value

    def kernel_launches(self):
        return self._u64(self.L.vct_kernel_launches)

    def trace_cones(self, starts, dirs, tan_half):
        s = np.ascontiguousarray(starts, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(np.broadcast_to(np.asarray(tan_half, dtype=np.float32), (s.shape[0],)))
        out = np.empty((s.shape[0], 4), dtype=np.float32)
        steps = np.empty(s.shape[0], dtype=np.uint32)
        self._ck(self.L.vct_trace_cones(self.h, s.shape[0], _ptr(s), _ptr(d), _ptr(t), _ptr(out), _ptr(steps)))
        return out, steps

    def bake_probes(self, xyz=None, out=None, steps=None, n=None, device_xyz=None, device_out=None, device_steps=None):
        """Irradiance probes: indirect light and occlusion at each point for a surface facing +X, -X, +Y, -Y, +Z, -Z.

        Host form: `xyz` (n, 3) float32; returns `out` (n, 6, 4) float32 = (r, g, b, occlusion) per face and `steps`
        (n, 6) uint32 textureLod calls per face (both allocated unless given).  Device form: `n` probes at the device
        pointers `device_xyz` (n*3 float32), `device_out` (n*24 float32) and optionally `device_steps` (n*6 uint32), e.g.
        torch CUDA tensors' data_ptr(); asynchronous on the context's stream, returns None."""
        if device_xyz is not None or device_out is not None:
            ptr = lambda p: None if p is None else C.c_void_p(int(p))
            self._ck(self.L.vct_bake_probes(self.h, int(n), ptr(device_xyz), ptr(device_out), ptr(device_steps), 1))
            return None
        x = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        k = x.shape[0]
        if out is None:
            out = np.empty((k, 6, 4), dtype=np.float32)
        if steps is None:
            steps = np.empty((k, 6), dtype=np.uint32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == k * 24
        assert steps.dtype == np.uint32 and steps.flags.c_contiguous and steps.size == k * 6
        self._ck(self.L.vct_bake_probes(self.h, k, _ptr(x), _ptr(out), _ptr(steps), 0))
        return out, steps

    def cast_rays(self, level, segments=None, n=None, device_segments=None, device_voxel=None, device_t=None,
                  device_face=None, device_rgba=None, device_steps=None):
        """Ray casts: the first occupied texel of mip `level` along each world-space segment a -> b.

        Host form: `segments` (n, 6) float32 (a.xyz, b.xyz); returns (voxel, t, face, rgba, steps): (n,) uint32 texel
        indices (z*N + y)*N + x (0xFFFFFFFF = miss), (n,) float32 segment parameter where the walk entered the texel
        (+inf = miss), (n,) uint8 entry-face normal 1..6 = +X, -X, +Y, -Y, +Z, -Z (0 = started inside it or missed),
        (n, 4) uint8 un-premultiplied colour and alpha (0 = miss), (n,) uint32 texels visited.  Device form: `n`
        segments at the device pointers `device_segments` (n*6 float32) and `device_voxel` (n uint32), optionally
        `device_t`, `device_face`, `device_rgba` (n*4 bytes, 4-byte aligned) and `device_steps`, e.g. torch CUDA
        tensors' data_ptr(); asynchronous on the context's stream, returns None."""
        if device_segments is not None or device_voxel is not None:
            ptr = lambda p: None if p is None else C.c_void_p(int(p))
            self._ck(self.L.vct_cast_rays(self.h, int(level), int(n), ptr(device_segments), ptr(device_voxel), ptr(device_t),
                                          ptr(device_face), ptr(device_rgba), ptr(device_steps), 1))
            return None
        s = np.ascontiguousarray(segments, dtype=np.float32).reshape(-1, 6)
        k = s.shape[0]
        voxel, t, face = np.empty(k, np.uint32), np.empty(k, np.float32), np.empty(k, np.uint8)
        rgba, steps = np.empty((k, 4), np.uint8), np.empty(k, np.uint32)
        self._ck(self.L.vct_cast_rays(self.h, int(level), k, _ptr(s), _ptr(voxel), _ptr(t), _ptr(face), _ptr(rgba),
                                      _ptr(steps), 0))
        return voxel, t, face, rgba, steps

    # ---- execution control
    def set_stream(self, cuda_stream_ptr):
        """Run on the given CUDA stream handle (0 / None = the CUDA default stream)."""
        self._ck(self.L.vct_set_stream(self.h, C.c_void_p(int(cuda_stream_ptr)) if cuda_stream_ptr else None))

    def use_own_stream(self):
        self._ck(self.L.vct_use_own_stream(self.h))

    def sample_voxels(self, pos, lod):
        p = np.ascontiguousarray(pos, dtype=np.float32).reshape(-1, 3)
        l = np.ascontiguousarray(np.broadcast_to(np.asarray(lod, dtype=np.float32), (p.shape[0],)))
        out = np.empty((p.shape[0], 4), dtype=np.float32)
        self._ck(self.L.vct_sample_voxels(self.h, p.shape[0], _ptr(p), _ptr(l), _ptr(out)))
        return out

    def sync(self):
        self._ck(self.L.vct_sync(self.h))

    def pass_time_us(self, name):
        v = C.c_float()
        self._ck(self.L.vct_pass_time_us(self.h, PASSES[name] if isinstance(name, str) else int(name), C.byref(v)))
        return v.value

    def pass_timeline(self, frames_back, name):
        a, b = C.c_float(), C.c_float()
        self._ck(self.L.vct_pass_timeline(self.h, int(frames_back), PASSES[name], C.byref(a), C.byref(b)))
        return a.value, b.value

    def bench_tex3d(self, V=256, n_samples=1 << 28, pattern=0, lod=0.5, iters=5, grid_format=0):
        v = C.c_float()
        self._ck(self.L.vct_bench_tex3d_format(self.h, int(V), int(grid_format), int(n_samples), int(pattern), float(lod),
                                               int(iters), C.byref(v)))
        return v.value

    def bench_atomics(self, n_fragments, iters=5):
        v = C.c_float()
        self._ck(self.L.vct_bench_atomics(self.h, int(n_fragments), int(iters), C.byref(v)))
        return v.value


def _host_ptr(out):
    """numpy array, torch CPU tensor (pinned or not) or raw int address."""
    if isinstance(out, int):
        return C.c_void_p(out)
    if hasattr(out, "data_ptr"):
        return C.c_void_p(out.data_ptr())
    return _ptr(out)



class MultiContext:
    """One process driving n devices (vct_create_multi / vct_comm_init_multi / vct_frame_sharded_multi)."""

    def __init__(self, devices):
        self.L = load_library()
        n = len(devices)
        self._arr = (C.c_void_p * n)()
        rc = self.L.vct_create_multi((C.c_int * n)(*[int(d) for d in devices]), n, self._arr)
        if rc:
            raise VctError(rc, self.L.vct_last_error(None).decode())
        self.ctx = [Context(int(d), handle=C.c_void_p(self._arr[k])) for k, d in enumerate(devices)]

    def __len__(self):
        return len(self.ctx)

    def each(self, fn):
        return [fn(c) for c in self.ctx]

    def comm_init(self, flags=0):
        rc = self.L.vct_comm_init_multi(self._arr, len(self.ctx), int(flags))
        if rc:
            raise VctError(rc, self.L.vct_last_error(self.ctx[0].h).decode())

    def frame_sharded(self, host_rgba=None):
        rc = self.L.vct_frame_sharded_multi(self._arr, len(self.ctx), None if host_rgba is None else _host_ptr(host_rgba))
        if rc:
            for c in self.ctx:
                c._ck(rc)

    def wait(self):
        for c in self.ctx:
            c.frame_sharded_wait()

    def close(self):
        for c in self.ctx:
            c.close()
