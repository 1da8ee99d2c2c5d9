"""ctypes bindings for the CPU oracle (oracle/oracle.cpp).

TEST INFRASTRUCTURE ONLY: import this from tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py — never from the product package.
"""
import ctypes as C
import importlib.util
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

_spec = importlib.util.spec_from_file_location("rt2025", os.path.join(ROOT, "raytracer-2025_b200", "rt2025.py"))
rt = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(rt)

_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, "liboracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-s", "-C", ROOT, "oracle"])
        L = C.CDLL(path)
        L.orc_last_error.restype = C.c_char_p
        L.orc_scene_create.restype = C.c_void_p
        L.orc_scene_create.argtypes = [C.c_void_p]
        L.orc_scene_destroy.argtypes = [C.c_void_p]
        L.orc_get_ranks.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.orc_closest_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_int, C.c_void_p]
        L.orc_render.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_tonemap.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
        D = C.POINTER(C.c_double)
        L.orc_kat_aabb_hit.argtypes = [D, D, D, D, C.c_double, C.c_double]
        L.orc_kat_aabb_longest_axis.argtypes = [D, D]
        L.orc_kat_aabb_from_points.argtypes = [D, D, D]
        L.orc_kat_aabb_union.argtypes = [D, D, D]
        L.orc_kat_sphere_uv.argtypes = [D, D]
        L.orc_kat_ray_at.argtypes = [D, D, C.c_double, D]
        L.orc_kat_vec3.argtypes = [D, D, C.c_double, D]
        L.orc_kat_quat_axis_angle_rotate.argtypes = [D, C.c_double, D, D]
        L.orc_kat_quat_mul.argtypes = [D, D, D]
        U = C.POINTER(C.c_uint32)
        L.orc_kat_philox.argtypes = [U, U, U]
        L.orc_kat_draw.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, D]
        L.orc_texture_value.argtypes = [C.c_void_p, C.c_uint32, C.c_double, C.c_double, D, D]
        L.orc_kat_world_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, D, D]
        L.orc_kat_scatter.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, D, D, D]
        L.orc_kat_cosine_pdf.argtypes = [D, D, D, D, D]
        L.orc_kat_disney_evaluate.argtypes = [D, C.c_int, D, D, C.c_int, D]
        L.orc_kat_disney_generate.argtypes = [D, C.c_int, D, C.c_int, D, D, D]
        L.orc_kat_lights_pdf_value.restype = C.c_double
        L.orc_kat_lights_pdf_value.argtypes = [C.c_void_p, D, D]
        L.orc_kat_lights_random.argtypes = [C.c_void_p, D, C.c_uint32, C.c_double, C.c_double, D]
        L.orc_kat_shade_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.orc_kat_shade_record.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.orc_camera_ray.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        _lib = L
    return _lib


def d(*v):
    return (C.c_double * len(v))(*[float(x) for x in v])


class OracleScene:
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

    def ranks(self):
        n = self.host.desc.contents.n_objects
        out = np.empty(n, dtype=np.uint32)
        assert self.L.orc_get_ranks(self.h, out.ctypes.data, n) == 0
        return out

    def closest_hit(self, rays, t_min=1e-8, t_max=float("inf"), mode=0):
        """mode 0: reference container semantics; mode 1: brute force over all leaves."""
        rays = np.ascontiguousarray(rays, dtype=rt.rt_ray_dtype)
        out = np.empty(len(rays), dtype=rt.rt_hit_dtype)
        self.L.orc_closest_hit(self.h, rays.ctypes.data, len(rays), t_min, t_max, mode, out.ctypes.data)
        return out

    def render(self, camera=None, seed=1, part_index=0, part_count=1, sample_begin=0, sample_end=0, threads=0):
        cam = camera if camera is not None else self.host.camera
        o = rt.rt_render_opts()
        o.struct_size = C.sizeof(rt.rt_render_opts)
        o.seed, o.accum_type = seed, rt.RT_ACCUM_F64
        o.part_index, o.part_count, o.sample_begin, o.sample_end = part_index, part_count, sample_begin, sample_end
        img = np.zeros((cam.image_height, cam.image_width, 3), dtype=np.float64)
        st = rt.rt_stats()
        self.L.orc_render(self.h, C.byref(cam), C.byref(o), img.ctypes.data, C.byref(st), threads)
        return img, st

    # ---- known-answer hooks (tests/test_oracle_kat_hand.py) ----
    def world_hit(self, o, dvec, time=0.0, t_min=1e-8, t_max=float("inf"), xi=None):
        """world.hit with every random draw forced to xi (None: media disabled) -> dict or None."""
        ray = rt.make_rays([o], [dvec], [time])
        out = (C.c_double * 12)()
        x = d(*xi) if xi is not None else None
        if not self.L.orc_kat_world_hit(self.h, ray.ctypes.data, t_min, t_max, x, out):
            return None
        o12 = list(out)
        return dict(t=o12[0], p=o12[1:4], normal=o12[4:7], u=o12[7], v=o12[8], front_face=bool(o12[9]), prim_id=int(o12[10]), inst_id=int(o12[11]))

    def scatter(self, mat, o, dvec, p, normal, front_face, u=0.0, v=0.0, xi=(0.5, 0.5), time=0.0):
        """materials[mat].scatter on a hand-made hit record -> (kind, attenuation, direction, error)."""
        ray = rt.make_rays([o], [dvec], [time])
        out = (C.c_double * 7)()
        kind = self.L.orc_kat_scatter(self.h, mat, ray.ctypes.data, d(*p, *normal, u, v, 1.0 if front_face else 0.0), d(*xi), out)
        return kind, list(out)[0:3], list(out)[3:6], bool(out[6])

    def shade_step(self, rays, seeds, ids3, camera=None):
        """One level of ray_color per row (ray_step): world.hit with media, emission, scatter, the mixture pdf and the next ray, the
        draws addressed by (seeds[i]; ids3[i] = pixel, sample, segment).  -> dict of arrays (hit: 0 miss, 1 surface, 2 medium;
        object: the leaf shape or the ConstantMedium; kind: the ScatterKind; goes_on: the recursion continues with the next ray; fuzzed:
        a SCATTER_RAY direction that went through sin / cos)."""
        cam = camera if camera is not None else self.host.camera
        rays = np.ascontiguousarray(rays, dtype=rt.rt_ray_dtype)
        n = len(rays)
        seeds, ids3 = np.ascontiguousarray(seeds, dtype=np.uint64), np.ascontiguousarray(ids3, dtype=np.uint32).reshape(n, 3)
        out = np.zeros((n, 28))
        self.L.orc_kat_shade_step(self.h, C.byref(cam), rays.ctypes.data, seeds.ctypes.data, ids3.ctypes.data, n, out.ctypes.data)
        return _segments(out)

    def shade_record(self, rays, records, seeds, ids3, camera=None):
        """The step rt_shade runs, on given rt_hit_records (shade_record: ray_step after world.hit), with the draws addressed as in
        shade_step.  -> the dict of shade_step; hit is the record's kind, object RT_NONE and t NaN (neither is read)."""
        cam = camera if camera is not None else self.host.camera
        rays = np.ascontiguousarray(rays, dtype=rt.rt_ray_dtype)
        records = np.ascontiguousarray(records, dtype=rt.rt_hit_record_dtype)
        n = len(rays)
        assert len(records) == n
        seeds, ids3 = np.ascontiguousarray(seeds, dtype=np.uint64), np.ascontiguousarray(ids3, dtype=np.uint32).reshape(n, 3)
        out = np.zeros((n, 28))
        self.L.orc_kat_shade_record(self.h, C.byref(cam), rays.ctypes.data, records.ctypes.data, seeds.ctypes.data, ids3.ctypes.data, n,
                                    out.ctypes.data)
        return _segments(out)

    def lights_pdf_value(self, origin, direction):
        return self.L.orc_kat_lights_pdf_value(self.h, d(*origin), d(*direction))

    def lights_random(self, origin, leaf, r1, r2):
        out = (C.c_double * 3)()
        ok = self.L.orc_kat_lights_random(self.h, d(*origin), leaf, r1, r2, out)
        return list(out) if ok else None

    def texture_value(self, tex, u, v, p):
        out = (C.c_double * 3)()
        self.L.orc_texture_value(self.h, tex, u, v, d(*p), out)
        return np.array(out)


def _segments(out):
    """The 28 columns of orc_kat_shade_step / orc_kat_shade_record as named arrays."""
    return dict(hit=out[:, 0].astype(np.int64), object=out[:, 1].astype(np.uint32), t=out[:, 2], background=out[:, 3:6], emission=out[:, 6:9],
                kind=out[:, 9].astype(np.int64), attenuation=out[:, 10:13], albedo_x_pscatter=out[:, 13:16], pdf_val=out[:, 16],
                o=out[:, 17:20], d=out[:, 20:23], time=out[:, 23], goes_on=out[:, 24] != 0.0, generated=out[:, 25] != 0.0,
                error=out[:, 26] != 0.0, fuzzed=out[:, 27] != 0.0)


def disney_evaluate(params15, thin, v_out, v_in, front_face):
    """Disney::evaluate_disney of the oracle on local-space unit vectors -> (reflectance(3), forward pdf) or None where the reference panics."""
    out = (C.c_double * 4)()
    if not lib().orc_kat_disney_evaluate(d(*params15), int(bool(thin)), d(*v_out), d(*v_in), int(bool(front_face)), out):
        return None
    return np.array(out[:3]), out[3]


def disney_generate(params15, thin, v_out, front_face, pick, u):
    """DisneyPDF::generate of the oracle in the local frame with forced draws -> direction, None (the reference's None) or "panic"."""
    out = (C.c_double * 3)()
    rc = lib().orc_kat_disney_generate(d(*params15), int(bool(thin)), d(*v_out), int(bool(front_face)), d(*pick), d(*u), out)
    return np.array(out) if rc == 1 else (None if rc == 0 else "panic")


def camera_rays(camera, seed, pixels_ij, sample):
    """Camera::get_ray for a list of (i, j) pixels at one sample index."""
    L = lib()
    out = np.zeros(len(pixels_ij), dtype=rt.rt_ray_dtype)
    for k, (i, j) in enumerate(pixels_ij):
        L.orc_camera_ray(C.byref(camera), seed, int(i), int(j), int(sample), out[k:k + 1].ctypes.data)
    return out


def cosine_pdf(albedo, normal, direction, xi=(0.5, 0.5)):
    """CosinePDF::new(albedo, normal): (value(direction) -> brdf, pdf), generate() with forced draws; None where it would panic."""
    out = (C.c_double * 7)()
    if not lib().orc_kat_cosine_pdf(d(*albedo), d(*normal), d(*direction), d(*xi), out):
        return None
    o = list(out)
    return o[0:3], o[3], o[4:7]


def tonemap(accum, toon_map=0):
    a = np.ascontiguousarray(accum, dtype=np.float64)
    out = np.empty(a.shape, dtype=np.uint8)
    lib().orc_tonemap(a.ctypes.data, a.size // 3, toon_map, out.ctypes.data)
    return out
