"""ctypes bindings for the CPU reference of rt_world_hit (tests/world_hit_oracle.cpp).

TEST INFRASTRUCTURE ONLY, like oracle/orc.py.  The library is the oracle plus one entry point; it is compiled on first use
with the oracle's flags into a directory under the system's temporary directory (keyed by the sources' digest), so the
repository tree is never written.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from transmittance_oracle import CXXFLAGS

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "world_hit_oracle.cpp"), os.path.join(ROOT, "oracle", "oracle.cpp"),
           os.path.join(ROOT, "include", "rt2025.h"), os.path.join(ROOT, "include", "rt2025_rng.h")]
# rt_hit_record of include/rt2025.h (rt2025.rt_hit_record_dtype; restated so that the oracle does not load the product)
hit_record_dtype = np.dtype([("t", "<f8"), ("p", "<f8", (3,)), ("normal", "<f8", (3,)), ("u", "<f8"), ("v", "<f8"), ("kind", "<u4"),
                             ("front_face", "<u4"), ("prim_id", "<u4"), ("inst_id", "<u4"), ("material", "<u4"), ("reserved", "<u4")])
assert hit_record_dtype.itemsize == 96

_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in SOURCES:
            h.update(open(p, "rb").read())
        h.update(" ".join(CXXFLAGS).encode())
        out_dir = os.path.join(tempfile.gettempdir(), f"rt2025_world_hit_oracle_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        path = os.path.join(out_dir, h.hexdigest()[:16] + ".so")
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=out_dir)
            os.close(fd)
            subprocess.check_call(["/usr/bin/g++", *CXXFLAGS, "-shared", "-o", tmp, SOURCES[0]])
            os.replace(tmp, path)  # atomic: concurrent first uses each build, one wins
        L = C.CDLL(path)
        L.orc_last_error.restype = C.c_char_p
        L.orc_scene_create.restype = C.c_void_p
        L.orc_scene_create.argtypes = [C.c_void_p]
        L.orc_scene_destroy.argtypes = [C.c_void_p]
        L.orc_world_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint64, C.c_uint32,
                                    C.c_void_p]
        _lib = L
    return _lib


class WorldHitOracle:
    """The oracle's scene for `host_scene` (an rt2025 host scene) with the world-hit reference."""

    def __init__(self, host_scene):
        self.L = lib()
        self.host = host_scene
        self.h = self.L.orc_scene_create(C.cast(host_scene.desc, C.c_void_p))
        if not self.h:
            raise RuntimeError("oracle: " + self.L.orc_last_error().decode())

    def __del__(self):
        try:
            if self.h:
                self.L.orc_scene_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def world_hit(self, rays, t_min=1e-8, t_max=float("inf"), seed=0, segment=0):
        """The record world.hit(ray, [t_min, t_max]) returns with the addressed draws of (seed, ray index, 0, segment).  `t_max`
        is a scalar or one value per ray."""
        ray_dtype = np.dtype([("origin", "<f8", (3,)), ("direction", "<f8", (3,)), ("time", "<f8")])  # rt_ray
        rays = np.ascontiguousarray(rays).view(ray_dtype)
        out = np.empty(len(rays), dtype=hit_record_dtype)
        per_ray = None
        if np.ndim(t_max) != 0:
            per_ray = np.ascontiguousarray(t_max, dtype=np.float64)
            assert per_ray.shape == (len(rays),)
            t_max = float("inf")
        self.L.orc_world_hit(self.h, rays.ctypes.data, None if per_ray is None else per_ray.ctypes.data, len(rays), t_min, t_max, seed,
                             segment, out.ctypes.data)
        return out
