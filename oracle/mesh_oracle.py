"""TEST INFRASTRUCTURE ONLY -- numpy front-end of oracle/mesh_oracle.c, the serial restatement of the marching-cubes export
(include/inerf_b200.h "mesh export").  Built with gcc into oracle/_build/libmesh_oracle.so on first use, with the flags of
oracle/Makefile, against the same table header as the CUDA kernels."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "mesh_oracle.c")
_INC = os.path.join(os.path.dirname(_HERE), "instance_nerf_b200", "csrc")
_SO = os.path.join(_HERE, "_build", "libmesh_oracle.so")
CFLAGS = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-Werror"]
_lib = None


def build():
    os.makedirs(os.path.dirname(_SO), exist_ok=True)
    tmp = f"{_SO}.{os.getpid()}"
    r = subprocess.run(["gcc", *CFLAGS, "-I", _INC, _SRC, "-o", tmp, "-lm"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building the mesh oracle failed:\n" + r.stdout + r.stderr)
    os.replace(tmp, _SO)
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = ctypes.CDLL(_SO)
        _lib.oracle_mesh.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_float,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib.oracle_mesh.restype = ctypes.c_int
    return _lib


def mesh(v, bbox, iso):
    """v float32 [X, Y, Z] -> (verts float32 [V, 3], faces int32 [F, 3]) in the order of the CUDA kernels."""
    v = np.ascontiguousarray(v, dtype=np.float32)
    bb = np.ascontiguousarray(bbox, dtype=np.float32).reshape(6)
    X, Y, Z = v.shape
    counts = np.zeros(2, np.int32)
    args = (v.ctypes.data, X, Y, Z, bb.ctypes.data, ctypes.c_float(iso), counts.ctypes.data)
    if lib().oracle_mesh(*args, None, None) != 0:
        raise MemoryError("oracle_mesh")
    verts = np.empty((int(counts[0]), 3), np.float32)
    faces = np.empty((int(counts[1]), 3), np.int32)
    if lib().oracle_mesh(*args, verts.ctypes.data, faces.ctypes.data) != 0:
        raise MemoryError("oracle_mesh")
    return verts, faces
