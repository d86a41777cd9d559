"""ctypes binding of tests/raycast_ref.cpp, the CPU reference of ray casts (test infrastructure).  The source is compiled
on first use into a temporary directory (the repository tree may be read-only), keyed by its content hash.
cast_rays(oracle, level, segments) casts world-space segments through mip `level` of the oracle's pyramid with the
oracle's parameters."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "raycast_ref.cpp")
_lib = None


class RCParams(C.Structure):
    _fields_ = [("VoxelDimensions", C.c_int32), ("GridFormat", C.c_int32), ("VoxelGridWorldSize", C.c_float)]


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        out_dir = os.path.join(tempfile.gettempdir(), f"vct_raycast_ref_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, hashlib.sha256(src).hexdigest()[:16] + ".so")
        if not os.path.exists(so):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared",
                            "-o", tmp, _SRC], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.rc_cast_rays.argtypes = [C.POINTER(RCParams), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
        L.rc_cast_rays.restype = C.c_int
        _lib = L
    return _lib


def cast_rays(oracle, level, segments):
    """segments (n, 6) float32 world-space a.xyz, b.xyz -> voxel (n,) uint32 (0xFFFFFFFF = miss), t (n,) float32 (+inf =
    miss), face (n,) uint8 (1..6 = +X, -X, +Y, -Y, +Z, -Z, 0 = none), rgba (n, 4) uint8, steps (n,) uint32"""
    p = oracle.p
    if not 0 <= level < p.VoxelDimensions.bit_length():
        raise ValueError(f"level {level} outside the pyramid")
    q = RCParams(p.VoxelDimensions, p.GridFormat, p.VoxelGridWorldSize)
    seg = np.ascontiguousarray(segments, dtype=np.float32).reshape(-1, 6)
    n = seg.shape[0]
    tex = np.ascontiguousarray(oracle.grid(level))
    voxel, t, face = np.empty(n, np.uint32), np.empty(n, np.float32), np.empty(n, np.uint8)
    rgba, steps = np.empty((n, 4), np.uint8), np.empty(n, np.uint32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib().rc_cast_rays(C.byref(q), int(level), ptr(tex), n, ptr(seg), ptr(voxel), ptr(t), ptr(face), ptr(rgba), ptr(steps))
    if rc:
        raise ValueError(f"level {level} outside the pyramid")
    return voxel, t, face, rgba, steps
