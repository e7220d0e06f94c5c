"""TEST INFRASTRUCTURE — ctypes loader of the CPU port of fi_marching_cubes (tests/mc_port.cpp), the sequential
restatement the kernels are compared with bit for bit.  Never imported by the product."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "mc_port.cpp")
TABLE = os.path.join(HERE, "..", "field_interpolation_b200", "csrc", "mc_table.cuh")

_cache = {}


def build(out_dir: str | None = None) -> str:
    """Compiles the port (once per source change) into out_dir, by default tests/_build."""
    out_dir = out_dir or os.path.join(HERE, "_build")
    out = os.path.join(out_dir, "libmc_port.so")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(SRC), os.path.getmtime(TABLE)):
        os.makedirs(out_dir, exist_ok=True)
        cmd = [os.environ.get("CXX", "g++"), "-std=c++14", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", out, SRC]
        subprocess.run(cmd, check=True)
    return out


class Port:
    def __init__(self, path):
        self.dll = C.CDLL(path)
        fn = self.dll.mcp_marching_cubes
        pf, pi32, pi64 = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int64)
        fn.restype, fn.argtypes = None, [pi32, pf, C.c_float, pf, pf, pi32, pi64, pi64]

    def marching_cubes(self, values, iso: float = 0.0, want_normals: bool = False):
        """Same arguments and results as field_interpolation_b200.marching_cubes on a (nz, ny, nx) host array."""
        a = np.ascontiguousarray(values, dtype=np.float32)
        assert a.ndim == 3
        sizes = np.array([a.shape[2], a.shape[1], a.shape[0]], np.int32)
        pf, pi32 = C.POINTER(C.c_float), C.POINTER(C.c_int32)
        nv, nt = C.c_int64(0), C.c_int64(0)
        fn = self.dll.mcp_marching_cubes
        fn(sizes.ctypes.data_as(pi32), a.ctypes.data_as(pf), float(iso), None, None, None, C.byref(nv), C.byref(nt))
        verts, tris = np.empty((nv.value, 3), np.float32), np.empty((nt.value, 3), np.int32)
        nrms = np.empty((nv.value, 3), np.float32)
        fn(sizes.ctypes.data_as(pi32), a.ctypes.data_as(pf), float(iso), verts.ctypes.data_as(pf),
           nrms.ctypes.data_as(pf) if want_normals else None, tris.ctypes.data_as(pi32), C.byref(nv), C.byref(nt))
        return (verts, tris, nrms) if want_normals else (verts, tris)


def port(out_dir: str | None = None) -> Port:
    if "port" not in _cache:
        _cache["port"] = Port(build(out_dir))
    return _cache["port"]
