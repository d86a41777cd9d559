"""ctypes binding of tests/voxel_view_ref.cpp, the CPU reference of the voxel view (test infrastructure).  The source is
compiled on first use into a temporary directory (the repository tree may be read-only), keyed by its content hash.
render_voxels(oracle, level) views mip `level` of the oracle's pyramid with the oracle's parameters."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "voxel_view_ref.cpp")
_lib = None


class VVParams(C.Structure):
    _fields_ = [("VoxelDimensions", C.c_int32), ("GridFormat", C.c_int32), ("screen_width", C.c_int32),
                ("screen_height", C.c_int32), ("VoxelGridWorldSize", C.c_float), ("ambientFactor", C.c_float),
                ("ModelMatrix", C.c_float * 16), ("ModelViewMatrix", C.c_float * 16), ("ProjectionMatrix", C.c_float * 16)]


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        out_dir = os.path.join(tempfile.gettempdir(), f"vct_voxel_view_ref_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, hashlib.sha256(src).hexdigest()[:16] + ".so")
        if not os.path.exists(so):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared",
                            "-o", tmp, _SRC], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.vv_render_voxels.argtypes = [C.POINTER(VVParams), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
        L.vv_render_voxels.restype = C.c_int
        _lib = L
    return _lib


def render_voxels(oracle, level):
    """-> (H, W, 4) uint8 rgba (row 0 = bottom), (H, W) uint32 texel indices (0xFFFFFFFF = miss), texels visited"""
    p = oracle.p
    if not 0 <= level < p.VoxelDimensions.bit_length():
        raise ValueError(f"level {level} outside the pyramid")
    q = VVParams()
    for name, _ in VVParams._fields_:
        v = getattr(p, name)
        if isinstance(v, (int, float)):
            setattr(q, name, v)
        else:
            getattr(q, name)[:] = v[:]
    tex = np.ascontiguousarray(oracle.grid(level))
    H, W = p.screen_height, p.screen_width
    rgba, vox, steps = np.empty((H, W, 4), np.uint8), np.empty((H, W), np.uint32), C.c_uint64(0)
    rc = lib().vv_render_voxels(C.byref(q), int(level), tex.ctypes.data_as(C.c_void_p), rgba.ctypes.data_as(C.c_void_p),
                                vox.ctypes.data_as(C.c_void_p), C.byref(steps))
    if rc:
        raise ValueError(f"level {level} outside the pyramid")
    return rgba, vox, int(steps.value)
