"""TEST INFRASTRUCTURE: ctypes wrapper around tests/oracle_rays.cpp, the CPU oracle's RayTracer#trace_sync and
World#intersect on caller-supplied rays.  The library is compiled with the oracle's flags into a temporary directory
(keyed by the sources' hash), so the test tree itself is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from raytracing_rb_b200 import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = (os.path.join(HERE, "oracle_rays.cpp"), os.path.join(ROOT, "oracle", "rtrb_oracle.cpp"),
           os.path.join(ROOT, "include", "rtrb_b200.h"))

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "rtrb_oracle_rays_%s_%d.so" % (h, os.getuid()))
        if not os.path.isfile(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread",
                                   "-o", tmp, SOURCES[0]])
            os.replace(tmp, so)
        L = C.CDLL(so)
        P = C.POINTER
        L.rtrb_oracle_scene_create.restype = C.c_void_p
        L.rtrb_oracle_scene_create.argtypes = [P(_abi.SceneDesc)]
        L.rtrb_oracle_scene_destroy.argtypes = [C.c_void_p]
        L.rtrb_oracle_trace_rays.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, P(_abi.Stats)]
        L.rtrb_oracle_world_intersect_full.argtypes = [C.c_void_p, P(C.c_double), P(C.c_double), P(C.c_double),
                                                       P(C.c_int), P(C.c_int)]
        _lib = L
    return _lib


class RayOracle:
    def __init__(self, scene_holder):
        self._holder = scene_holder
        self._h = lib().rtrb_oracle_scene_create(C.byref(scene_holder.desc))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().rtrb_oracle_scene_destroy(self._h)
            self._h = None

    def trace_rays(self, rays, trace_depth=1, mc=0, seed=1, keys=None):
        """-> (rgb [n, 3], hit [n], stats dict, status code), as Renderer.trace_rays."""
        rays = np.ascontiguousarray(rays, np.float64).reshape(-1, 6)
        n = rays.shape[0]
        if keys is not None:
            keys = np.ascontiguousarray(keys, np.uint32).reshape(-1, 2)
        rgb = np.zeros((n, 3), np.float64)
        hit = np.zeros(n, np.int32)
        st = _abi.Stats()
        code = lib().rtrb_oracle_trace_rays(self._h, trace_depth, mc, seed, n, rays.ctypes.data,
                                            keys.ctypes.data if keys is not None else None, rgb.ctypes.data,
                                            hit.ctypes.data, C.byref(st))
        return rgb, hit, st.as_dict(), code

    def intersect_rays(self, rays):
        """-> structured array of RAY_HIT_DTYPE, as Renderer.intersect_rays."""
        from raytracing_rb_b200 import RAY_HIT_DTYPE
        rays = np.ascontiguousarray(rays, np.float64).reshape(-1, 6)
        out = np.zeros(rays.shape[0], RAY_HIT_DTYPE)
        o7, din, face = (C.c_double * 7)(), C.c_int(), C.c_int()
        for i, r in enumerate(rays):
            idx = lib().rtrb_oracle_world_intersect_full(self._h, (C.c_double * 3)(*r[:3]), (C.c_double * 3)(*r[3:]), o7,
                                                         C.byref(din), C.byref(face))
            out[i]["object"], out[i]["direction"], out[i]["face"] = idx, din.value, face.value
            out[i]["distance"] = o7[0]
            out[i]["intersection"] = o7[1:4]
            out[i]["delta"] = o7[4:7]
        return out
