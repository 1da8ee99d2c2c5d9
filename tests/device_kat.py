"""ctypes bindings for the device shading harness (tests/device_kat.cu).

TEST INFRASTRUCTURE ONLY, like oracle/orc.py.  The library is the harness plus the product's scene compiler (csrc/compile.cpp,
csrc/bvh_build.cpp), built with the Makefile's NVCC and NVCCFLAGS - the product's own compiler and flags, sm_100a - on first use, into a
directory under the system's temporary directory keyed by the digest of every source and the flags, so the repository tree is never
written.  kat_light_table needs no device; everything else runs one thin kernel per call.
"""
import ctypes as C
import glob
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "raytracer-2025_b200", "csrc")
HARNESS = os.path.join(HERE, "device_kat.cu")
LINKED = [os.path.join(CSRC, "compile.cpp"), os.path.join(CSRC, "bvh_build.cpp")]
RT_NONE = 0xFFFFFFFF
RAY_DTYPE = np.dtype([("origin", "<f8", (3,)), ("direction", "<f8", (3,)), ("time", "<f8")])  # rt_ray

_lib = None


def make_flags():
    """[NVCC, *NVCCFLAGS] as the Makefile defines them (read through make itself, so the two cannot drift apart)."""
    out = subprocess.check_output(["make", "-s", "--no-print-directory", "-C", ROOT, "--eval",
                                   "_kat_flags:\n\t@echo $(NVCC) $(NVCCFLAGS)", "_kat_flags"], text=True)
    return out.split()


def sources():
    return sorted([HARNESS, os.path.join(ROOT, "Makefile")] + glob.glob(os.path.join(CSRC, "*")) + glob.glob(os.path.join(ROOT, "include", "*.h")))


def lib_path():
    flags = make_flags()
    h = hashlib.sha256()
    for p in sources():
        h.update(os.path.basename(p).encode())
        h.update(open(p, "rb").read())
    h.update(" ".join(flags).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"rt2025_device_kat_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, h.hexdigest()[:16] + ".so")
    if not os.path.exists(path):
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=out_dir)
        os.close(fd)
        # the relative include paths of NVCCFLAGS are the Makefile's: compile from the repository root
        try:
            subprocess.check_call([*flags, "-shared", "-o", tmp, HARNESS, *LINKED, "-Xlinker", "-lgomp"], cwd=ROOT)
        except BaseException:
            os.unlink(tmp)
            raise
        os.replace(tmp, path)  # atomic: concurrent first uses each build, one wins
    return path


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(lib_path())
        P = C.c_void_p
        L.kat_last_error.restype = C.c_char_p
        L.kat_scene_create.restype = P
        L.kat_scene_create.argtypes = [P]
        L.kat_scene_destroy.argtypes = [P]
        L.kat_scene_info.argtypes = [P, P]
        L.kat_prim_of_object.argtypes = [P, P, C.c_uint32]
        L.kat_light_table.argtypes = [P, P, P, P, P, C.c_uint32]
        L.kat_disney_evaluate.argtypes = [P, C.c_int, P, P, P, C.c_int, P]
        L.kat_disney_generate.argtypes = [P, C.c_int, P, P, P, P, C.c_int, P]
        L.kat_texture_value.argtypes = [P, P, P, C.c_int, P]
        L.kat_background_value.argtypes = [P, C.c_uint32, P, C.c_int, P]
        L.kat_surface_hit_info.argtypes = [P, P, P, P, C.c_int, P]
        L.kat_remap_record.argtypes = [P, P, P, C.c_int, P]
        L.kat_lights_pdf.argtypes = [P, C.c_int, P, P, C.c_int, P]
        L.kat_lights_random.argtypes = [P, C.c_int, P, P, C.c_int, P]
        L.kat_material_emitted.argtypes = [P, P, P, C.c_int, P]
        L.kat_slab.argtypes = [P, P, C.c_int, P]
        L.kat_medium_free_flight.argtypes = [P, C.c_int, P]
        L.kat_free_flight_overshoots.argtypes = [P, C.c_int, P]
        L.kat_scene_lean_info.argtypes = [P, P]
        L.kat_prim_class.argtypes = [P, P, C.c_uint32]
        L.kat_media.argtypes = [P, P, P, P, C.c_uint32]
        L.kat_shade_step.argtypes = [P, P, C.c_uint32, C.c_int, P, P, P, P, C.c_int, P]
        L.kat_camera_ray.argtypes = [P, C.c_uint64, P, C.c_int, P]
        _lib = L
    return _lib


# Every array handed to the library is bound to a name first: `_u32(x).ctypes.data` alone would leave only an address to a temporary
# that may be freed before the call reads it.
def _f64(a, cols=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if cols is None else a.reshape(-1, cols)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _check(rc):
    if rc != 0:
        raise RuntimeError("device_kat: " + lib().kat_last_error().decode())


def light_table(host_scene):
    """Every light leaf of the compiled scene: dict of kind, xform (RT_NONE: none), weight, cdf arrays.  Needs no device."""
    L = lib()
    cap = 4096
    kind, xform = np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
    weight, cdf = np.zeros(cap), np.zeros(cap)
    n = L.kat_light_table(C.cast(host_scene.desc, C.c_void_p), kind.ctypes.data, xform.ctypes.data, weight.ctypes.data, cdf.ctypes.data, cap)
    if n < 0:
        raise RuntimeError("device_kat: " + L.kat_last_error().decode())
    assert n <= cap
    return dict(kind=kind[:n], xform=xform[:n], weight=weight[:n], cdf=cdf[:n])


def disney_evaluate(params15, thin, v_out, v_in, front_face):
    """-> (reflectance (n, 3), forward pdf (n,), error (n,) bool) of disney::evaluate_disney, one call per row."""
    v_out, v_in = _f64(v_out, 3), _f64(v_in, 3)
    ff = np.ascontiguousarray(np.broadcast_to(np.asarray(front_face, dtype=np.int32), (len(v_out),)))
    out, params = np.zeros((len(v_out), 5)), _f64(params15)
    _check(lib().kat_disney_evaluate(params.ctypes.data, int(bool(thin)), v_out.ctypes.data, v_in.ctypes.data, ff.ctypes.data, len(v_out),
                                     out.ctypes.data))
    return out[:, :3], out[:, 3], out[:, 4] != 0.0


def disney_generate(params15, thin, v_out, front_face, pick, u):
    """-> (direction (n, 3), rc (n,)): disney::generate_local then the unit_vector of shade_one; rc 1 Some, 0 None, -1 panic."""
    v_out = _f64(v_out, 3)
    ff = np.ascontiguousarray(np.broadcast_to(np.asarray(front_face, dtype=np.int32), (len(v_out),)))
    out, params, pick, u = np.zeros((len(v_out), 4)), _f64(params15), _f64(pick, 2), _f64(u, 2)
    _check(lib().kat_disney_generate(params.ctypes.data, int(bool(thin)), v_out.ctypes.data, ff.ctypes.data, pick.ctypes.data, u.ctypes.data,
                                     len(v_out), out.ctypes.data))
    return out[:, :3], out[:, 3].astype(np.int64)


def slab(o, d, t_min, t_max, lo, hi):
    """make_rayf + slab of the traversal, one call per row: o, d (n, 3) binary64, t_min / t_max (n,) binary64 (rounded to binary32
    down / up as the traversal does), lo / hi (n, 3) binary32 boxes -> (n,) bool, True when the box is kept."""
    inp = np.ascontiguousarray(np.column_stack([_f64(o, 3), _f64(d, 3), _f64(t_min), _f64(t_max)]))
    box = np.ascontiguousarray(np.column_stack([np.asarray(lo, np.float32).reshape(-1, 3), np.asarray(hi, np.float32).reshape(-1, 3)]))
    n = len(inp)
    out = np.zeros(n, np.uint8)
    _check(lib().kat_slab(inp.ctypes.data, box.ctypes.data, n, out.ctypes.data))
    return out != 0


def medium_free_flight(t1, t2, d, neg_inv_density, xi):
    """medium_free_flight of one medium per row -> (ok (n,) bool, tm (n,))."""
    d = _f64(d, 3)
    n = len(d)
    inp = np.ascontiguousarray(np.column_stack([np.broadcast_to(t1, n), np.broadcast_to(t2, n), d, np.broadcast_to(neg_inv_density, n),
                                                np.broadcast_to(xi, n)]))
    out = np.zeros((n, 2))
    _check(lib().kat_medium_free_flight(inp.ctypes.data, n, out.ctypes.data))
    return out[:, 0] != 0.0, out[:, 1]


def free_flight_overshoots(neg_inv_density, xi, t, d):
    """free_flight_overshoots per row -> (n,) bool."""
    d = _f64(d, 3)
    n = len(d)
    inp = np.ascontiguousarray(np.column_stack([np.broadcast_to(neg_inv_density, n), np.broadcast_to(xi, n), np.broadcast_to(t, n), d]))
    out = np.zeros(n, np.uint8)
    _check(lib().kat_free_flight_overshoots(inp.ctypes.data, n, out.ctypes.data))
    return out != 0


def camera_ray(camera, seed, i, j, sidx):
    """k_generate's camera_ray for every row (i, j, sidx broadcast together) -> rt_ray records."""
    inp = np.ascontiguousarray(np.column_stack(np.broadcast_arrays(np.asarray(i), np.asarray(j), np.asarray(sidx))), dtype=np.uint32)
    n = len(inp)
    out = np.zeros(n, dtype=RAY_DTYPE)
    _check(lib().kat_camera_ray(C.addressof(camera), int(seed), inp.ctypes.data, n, out.ctypes.data))
    return out


class DeviceScene:
    """The product's compiled tables of `host_scene` on the device, for the shading wrappers."""

    def __init__(self, host_scene):
        self.L = lib()
        self.host = host_scene
        self.h = self.L.kat_scene_create(C.cast(host_scene.desc, C.c_void_p))
        if not self.h:
            raise RuntimeError("device_kat: " + self.L.kat_last_error().decode())
        info = np.zeros(5, np.uint32)
        self.L.kat_scene_info(self.h, info.ctypes.data)
        self.n_lights, self.lights_flat, self.has_lean, self.n_lean, self.n_prims = (int(x) for x in info)
        n_obj = host_scene.desc.contents.n_objects
        self.prim_of_object = np.zeros(n_obj, np.uint32)
        self.L.kat_prim_of_object(self.h, self.prim_of_object.ctypes.data, n_obj)
        lean = np.zeros(4, np.uint32)
        self.L.kat_scene_lean_info(self.h, lean.ctypes.data)
        self.shade_lean_mask, self.has_walk_lean, self.walk_thick, n_media = (int(x) for x in lean)
        self.prim_class = np.zeros(self.n_prims, np.uint32)
        self.L.kat_prim_class(self.h, self.prim_class.ctypes.data, self.n_prims)
        self.medium_object, self.medium_flags, self.medium_xform = (np.zeros(n_media, np.uint32) for _ in range(3))
        self.L.kat_media(self.h, self.medium_object.ctypes.data, self.medium_flags.ctypes.data, self.medium_xform.ctypes.data, n_media)

    def __del__(self):
        try:
            if self.h:
                self.L.kat_scene_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def texture_value(self, tex, u, v, p):
        """texture_value for every row: tex (n,) or scalar, u (n,), v (n,), p (n, 3) -> (n, 3)."""
        p = _f64(p, 3)
        n = len(p)
        inp = np.ascontiguousarray(np.column_stack([np.broadcast_to(u, n), np.broadcast_to(v, n), p]))
        tex = _u32(np.broadcast_to(tex, n))
        out = np.zeros((n, 3))
        _check(self.L.kat_texture_value(self.h, tex.ctypes.data, inp.ctypes.data, n, out.ctypes.data))
        return out

    def background_value(self, tex, dirs):
        dirs = _f64(dirs, 3)
        out = np.zeros((len(dirs), 4))
        _check(self.L.kat_background_value(self.h, tex, dirs.ctypes.data, len(dirs), out.ctypes.data))
        return out[:, :3], out[:, 3] != 0.0

    @staticmethod
    def _hits(out):
        return dict(p=out[:, 0:3], normal=out[:, 3:6], u=out[:, 6], v=out[:, 7], front_face=out[:, 8] != 0.0, ok=out[:, 9] != 0.0,
                    material=out[:, 10].astype(np.uint32))

    def surface_hit_info(self, prim, t, rays):
        """surface_hit_info(want_uv = true) of device primitive prim[i] at t[i] on rays[i] (rt_ray records)."""
        rays = np.ascontiguousarray(rays)
        n = len(rays)
        out, prim, t = np.zeros((n, 11)), _u32(prim), _f64(t)
        _check(self.L.kat_surface_hit_info(self.h, prim.ctypes.data, t.ctypes.data, rays.ctypes.data, n, out.ctypes.data))
        return self._hits(out)

    def remap_record(self, remap, hit):
        """remap_record of remaps[remap[i]] on the hit records of `hit` (a dict as surface_hit_info returns)."""
        inp = np.ascontiguousarray(np.column_stack([hit["p"], hit["normal"], hit["u"], hit["v"], np.asarray(hit["front_face"], np.float64)]))
        n = len(inp)
        out, remap = np.zeros((n, 11)), _u32(remap)
        _check(self.L.kat_remap_record(self.h, remap.ctypes.data, inp.ctypes.data, n, out.ctypes.data))
        return self._hits(out)

    def lights_pdf(self, origin, direction, lean=False):
        origin, direction = _f64(origin, 3), _f64(direction, 3)
        out = np.zeros(len(origin))
        _check(self.L.kat_lights_pdf(self.h, int(lean), origin.ctypes.data, direction.ctypes.data, len(origin), out.ctypes.data))
        return out

    def lights_random(self, origin, pick, r1, r2, lean=False):
        origin = _f64(origin, 3)
        n = len(origin)
        inp = np.ascontiguousarray(np.column_stack([np.broadcast_to(pick, n), np.broadcast_to(r1, n), np.broadcast_to(r2, n)]))
        out = np.zeros((n, 4))
        _check(self.L.kat_lights_random(self.h, int(lean), origin.ctypes.data, inp.ctypes.data, n, out.ctypes.data))
        return out[:, :3], out[:, 3] != 0.0

    def material_emitted(self, mat, u, v, p):
        p = _f64(p, 3)
        n = len(p)
        inp = np.ascontiguousarray(np.column_stack([np.broadcast_to(u, n), np.broadcast_to(v, n), p]))
        out, mat = np.zeros((n, 3)), _u32(np.broadcast_to(mat, n))
        _check(self.L.kat_material_emitted(self.h, mat.ctypes.data, inp.ctypes.data, n, out.ctypes.data))
        return out

    def shade_step(self, camera, cls, lean, rays, beta, t, ids6, seeds):
        """One path segment per row (shade_step.cuh): shade_one<cls> (lean 0), the lean shade kernels' code (lean 1) or the lean walk's
        lean_isotropic_scatter (lean 2).  rays: rt_ray records; beta (n, 3); t (n,); ids6 (n, 6): pixel, sample, segment, device
        primitive or medium index, hit kind, max_depth; seeds (n,).  -> dict of next o, d, time, nbeta, alive, errors, contribution."""
        rays = np.ascontiguousarray(rays)
        n = len(rays)
        in4 = np.ascontiguousarray(np.column_stack([_f64(beta, 3), _f64(t)]))
        ids6, seeds = _u32(ids6).reshape(n, 6), np.ascontiguousarray(seeds, dtype=np.uint64)
        out = np.zeros((n, 16))
        _check(self.L.kat_shade_step(self.h, C.addressof(camera), int(cls), int(lean), rays.ctypes.data, in4.ctypes.data, ids6.ctypes.data,
                                     seeds.ctypes.data, n, out.ctypes.data))
        return dict(o=out[:, 0:3], d=out[:, 3:6], time=out[:, 6], nbeta=out[:, 7:10], alive=out[:, 10] != 0.0, errors=out[:, 11].astype(np.int64),
                    contribution=out[:, 12:15])
