"""ctypes bindings for the C ABI (include/rt2025.h) and the C++ host mirror.

Python is plumbing here: it builds scenes through the host mirror (the reference's constructors,
SURVEY.md §8b), hands the flat description to librt2025.so and moves buffers.  There is no
Python or CPU implementation of the path: every compute call goes through the CUDA library and
raises RtError when it (or a GPU) is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
RT_NONE = 0xFFFFFFFF
RT_OPT_COUNT = 1
RT_OPT_STAGE_TIMES = 2
RT_ACCUM_F32 = 0
RT_ACCUM_F64 = 1
RT_BUILD_NO_REF_RANKS = 1
RT_BUILD_DEVICE_LBVH = 2
RT_HIT_MISS, RT_HIT_SURFACE, RT_HIT_MEDIUM = 0, 1, 2  # rt_hit_record.kind
RT_PATH_ALIVE, RT_PATH_ERROR = 1, 2  # rt_shade path state bits

# every symbol include/rt2025.h declares (tests check that the library exports them all)
ABI_SYMBOLS = [
    "rt_scene_create", "rt_scene_destroy", "rt_closest_hit", "rt_closest_hit_device", "rt_occluded", "rt_occluded_device", "rt_transmittance",
    "rt_transmittance_device", "rt_world_hit", "rt_world_hit_device", "rt_shade", "rt_shade_device",
    "rt_camera_rays", "rt_camera_rays_device", "rt_camera_rays_ids", "rt_camera_rays_ids_device", "rt_world_hit_ids",
    "rt_world_hit_ids_device", "rt_shade_ids", "rt_shade_ids_device", "rt_render",
    "rt_render_device", "rt_render_rgb8", "rt_render_multi", "rt_render_multi_rgb8", "rt_tonemap", "rt_tonemap_device", "rt_scene_get_info", "rt_scene_get_ranks", "rt_last_error",
    "rt_abi_version", "rt_device_count",
]


class RtError(RuntimeError):
    pass


class rt_camera(C.Structure):
    _fields_ = [
        ("image_width", C.c_uint32), ("image_height", C.c_uint32), ("sqrt_spp", C.c_uint32),
        ("max_depth", C.c_uint32), ("background_tex", C.c_uint32), ("toon_map", C.c_uint32),
        ("recip_sqrt_spp", C.c_double), ("pixel_sample_scale", C.c_double),
        ("center", C.c_double * 3), ("pixel00_loc", C.c_double * 3),
        ("pixel_delta_u", C.c_double * 3), ("pixel_delta_v", C.c_double * 3),
        ("defocus_angle_in_degrees", C.c_double),
        ("defocus_disk_u", C.c_double * 3), ("defocus_disk_v", C.c_double * 3),
    ]


class rt_build_opts(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("flags", C.c_uint32), ("device", C.c_int32), ("reserved", C.c_uint32)]


class rt_render_opts(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("flags", C.c_uint32), ("seed", C.c_uint64),
        ("accum_type", C.c_uint32), ("part_index", C.c_uint32), ("part_count", C.c_uint32),
        ("sample_begin", C.c_uint32), ("sample_end", C.c_uint32), ("max_paths_in_flight", C.c_uint32),
        ("reserved", C.c_uint32 * 4),
    ]


class rt_stats(C.Structure):
    _fields_ = [
        ("paths", C.c_uint64), ("segments", C.c_uint64), ("node_visits", C.c_uint64),
        ("prim_tests", C.c_uint64), ("errors", C.c_uint64), ("kernel_launches", C.c_uint64),
        ("ms_total", C.c_double), ("ms_raygen", C.c_double), ("ms_extend", C.c_double),
        ("ms_shade", C.c_double), ("ms_other", C.c_double), ("iterations", C.c_uint64),
        ("reserved", C.c_uint64 * 4),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}

    @property
    def walk_segments(self):
        """of `segments`: evaluated inside the random-walk kernel of an optically thick medium (rt2025.h, reserved[0])"""
        return int(self.reserved[0])

    @property
    def walk_lean_segments(self):
        """of `walk_segments`: evaluated by the lean variant of the random-walk kernel (rt2025.h, reserved[1])"""
        return int(self.reserved[1])

    @property
    def shade_lean_hits(self):
        """hits shaded by the lean variant of a shade-class kernel (rt2025.h, reserved[2])"""
        return int(self.reserved[2])


class rt_scene_info(C.Structure):
    _fields_ = [
        ("n_prims", C.c_uint32), ("n_spheres", C.c_uint32), ("n_planars", C.c_uint32), ("n_nodes", C.c_uint32),
        ("n_media", C.c_uint32), ("n_lights", C.c_uint32), ("n_materials", C.c_uint32), ("n_textures", C.c_uint32),
        ("bvh_depth", C.c_uint32), ("node_bytes", C.c_uint32), ("device_bytes", C.c_uint64),
    ]


class rth_camera_params(C.Structure):
    _fields_ = [
        ("aspect_ratio", C.c_double), ("image_width", C.c_uint32), ("samples_per_pixel", C.c_uint32),
        ("max_depth", C.c_uint32), ("background_tex", C.c_uint32), ("vertical_fov_in_degrees", C.c_double),
        ("look_from", C.c_double * 3), ("look_at", C.c_double * 3), ("vec_up", C.c_double * 3),
        ("defocus_angle_in_degrees", C.c_double), ("focus_distance", C.c_double),
        ("toon_map", C.c_uint32), ("reserved", C.c_uint32),
    ]


# rt_scene_desc header fields (the pointers are only ever dereferenced by native code)
class rt_scene_desc(C.Structure):
    _fields_ = [
        ("version", C.c_uint32), ("struct_size", C.c_uint32), ("world_root", C.c_uint32), ("lights_root", C.c_uint32),
        ("n_objects", C.c_uint32), ("n_children", C.c_uint32), ("n_spheres", C.c_uint32), ("n_planars", C.c_uint32),
        ("n_transforms", C.c_uint32), ("n_media", C.c_uint32), ("n_materials", C.c_uint32), ("n_textures", C.c_uint32),
        ("n_images", C.c_uint32), ("n_perlins", C.c_uint32), ("n_texels", C.c_uint64),
        ("n_remaps", C.c_uint32), ("reserved0", C.c_uint32),
        ("objects", C.c_void_p), ("children", C.c_void_p), ("spheres", C.c_void_p), ("planars", C.c_void_p),
        ("transforms", C.c_void_p), ("media", C.c_void_p), ("materials", C.c_void_p), ("textures", C.c_void_p),
        ("images", C.c_void_p), ("texels", C.c_void_p), ("perlins", C.c_void_p), ("remaps", C.c_void_p),
    ]


rt_object_dtype = np.dtype([("kind", "<u4"), ("material", "<u4"), ("first_child", "<u4"), ("child_count", "<u4"),
                            ("data", "<u4"), ("reserved", "<u4"), ("bbox", "<f8", (6,))])
rt_ray_dtype = np.dtype([("origin", "<f8", (3,)), ("direction", "<f8", (3,)), ("time", "<f8")])
rt_hit_dtype = np.dtype([("t", "<f8"), ("prim_id", "<u4"), ("inst_id", "<u4"), ("u", "<f4"), ("v", "<f4")])
assert rt_ray_dtype.itemsize == 56 and rt_hit_dtype.itemsize == 24 and rt_object_dtype.itemsize == 72
rt_hit_record_dtype = np.dtype([("t", "<f8"), ("p", "<f8", (3,)), ("normal", "<f8", (3,)), ("u", "<f8"), ("v", "<f8"), ("kind", "<u4"),
                                ("front_face", "<u4"), ("prim_id", "<u4"), ("inst_id", "<u4"), ("material", "<u4"), ("reserved", "<u4")])
assert rt_hit_record_dtype.itemsize == 96
# the address of a row's draws in the path-id entries: (pixel j * W + i, stratum, segment); `reserved` is never read or written
rt_path_id_dtype = np.dtype([("pixel", "<u4"), ("sample", "<u4"), ("segment", "<u4"), ("reserved", "<u4")])
assert rt_path_id_dtype.itemsize == 16


def build_native(targets=("product", "host")):
    """Compile the in-tree libraries with make (nvcc -gencode arch=compute_100a,code=sm_100a)."""
    subprocess.check_call(["make", "-s", "-C", ROOT, *targets])


_host = None
_product = None


def host_lib():
    """librt2025_host.so: the C++ mirror of the reference's scene-construction API."""
    global _host
    if _host is None:
        path = os.path.join(PKG_DIR, "librt2025_host.so")
        if not os.path.exists(path):
            build_native(("host",))
        L = C.CDLL(path)
        L.rth_last_error.restype = C.c_char_p
        L.rth_scene_named.restype = C.c_void_p
        L.rth_scene_named.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(C.c_double), C.c_int]
        L.rth_scene_desc.restype = C.POINTER(rt_scene_desc)
        L.rth_scene_desc.argtypes = [C.c_void_p]
        L.rth_scene_camera.restype = C.POINTER(rt_camera)
        L.rth_scene_camera.argtypes = [C.c_void_p]
        L.rth_scene_free.argtypes = [C.c_void_p]
        L.rth_builder_new.restype = C.c_void_p
        L.rth_builder_new.argtypes = [C.c_uint64]
        L.rth_builder_free.argtypes = [C.c_void_p]
        L.rth_builder_finish.restype = C.c_void_p
        L.rth_builder_finish.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(rth_camera_params)]
        D3 = C.POINTER(C.c_double)
        sig = {
            "rth_tex_solid": [C.c_void_p, C.c_double, C.c_double, C.c_double],
            "rth_tex_checker": [C.c_void_p, C.c_double, C.c_uint32, C.c_uint32],
            "rth_tex_noise": [C.c_void_p, C.c_double],
            "rth_tex_image_missing": [C.c_void_p],
            "rth_tex_image": [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_int],
            "rth_tex_gradient": [C.c_void_p, D3, D3],
            "rth_mat_empty": [C.c_void_p],
            "rth_mat_lambertian": [C.c_void_p, C.c_uint32],
            "rth_mat_metal": [C.c_void_p, D3, C.c_double],
            "rth_mat_dielectric": [C.c_void_p, C.c_uint32, C.c_double],
            "rth_mat_diffuse_light": [C.c_void_p, C.c_uint32, C.c_uint32],
            "rth_mat_isotropic": [C.c_void_p, C.c_uint32],
            "rth_mat_transparent": [C.c_void_p],
            "rth_mat_mix": [C.c_void_p, C.c_uint32, C.c_uint32, C.c_double],
            "rth_mat_mix_image": [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32],
            "rth_mat_portal": [C.c_void_p, D3, D3, D3],
            "rth_mat_disney": [C.c_void_p, D3, C.c_uint32, D3],
            "rth_mat_remapped": [C.c_void_p, C.c_uint32, D3, D3, D3, C.c_uint32],
            "rth_sphere": [C.c_void_p, D3, C.c_double, C.c_uint32],
            "rth_sphere_moving": [C.c_void_p, D3, D3, C.c_double, C.c_uint32],
            "rth_quad": [C.c_void_p, D3, D3, D3, C.c_uint32],
            "rth_triangle": [C.c_void_p, D3, D3, D3, C.c_uint32],
            "rth_box": [C.c_void_p, D3, D3, C.c_uint32],
            "rth_list": [C.c_void_p, C.POINTER(C.c_uint32), C.c_uint32, C.c_int],
            "rth_bvh": [C.c_void_p, C.POINTER(C.c_uint32), C.c_uint32],
            "rth_transform": [C.c_void_p, C.c_uint32, D3, D3, D3],
            "rth_medium": [C.c_void_p, C.c_uint32, C.c_double, C.c_uint32],
        }
        for name, args in sig.items():
            f = getattr(L, name)
            f.restype = C.c_uint32
            f.argtypes = args
        L.rth_quat_from_axis_angle.argtypes = [D3, C.c_double, D3]
        _host = L
    return _host


def product_lib(required=True):
    """librt2025.so: the CUDA core.  Fails loudly when it is missing — there is no fallback."""
    global _product
    if _product is None:
        # RT2025_LIB selects another build of the same library (kernel-variant experiments)
        path = os.environ.get("RT2025_LIB") or os.path.join(PKG_DIR, "librt2025.so")
        if not os.path.exists(path):
            if required:
                raise RtError(f"{path} is missing: run `make product` (or __graft_entry__.build()); "
                              "this package has no CPU or Python fallback")
            return None
        L = C.CDLL(path)
        L.rt_last_error.restype = C.c_char_p
        L.rt_abi_version.restype = C.c_uint32
        L.rt_scene_create.argtypes = [C.POINTER(rt_scene_desc), C.POINTER(rt_build_opts), C.POINTER(C.c_void_p)]
        L.rt_scene_destroy.argtypes = [C.c_void_p]
        L.rt_closest_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                     C.c_void_p, C.POINTER(rt_stats)]
        L.rt_closest_hit_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                            C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
        if hasattr(L, "rt_occluded"):  # absent from older builds selected with RT2025_LIB for A/B runs
            L.rt_occluded.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                      C.c_void_p, C.POINTER(rt_stats)]
            L.rt_occluded_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                             C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
        if hasattr(L, "rt_transmittance"):  # absent from older builds selected with RT2025_LIB for A/B runs
            L.rt_transmittance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                           C.c_void_p, C.POINTER(rt_stats)]
            L.rt_transmittance_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                                  C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
        if hasattr(L, "rt_world_hit"):  # absent from older builds selected with RT2025_LIB for A/B runs
            L.rt_world_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint64, C.c_uint32,
                                       C.c_uint32, C.c_void_p, C.POINTER(rt_stats)]
            L.rt_world_hit_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint64,
                                              C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
        if hasattr(L, "rt_shade"):  # absent from older builds selected with RT2025_LIB for A/B runs
            L.rt_shade.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
            L.rt_shade_device.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
            L.rt_camera_rays.argtypes = [C.POINTER(rt_camera), C.c_uint64, C.c_uint32, C.c_void_p]
            L.rt_camera_rays_device.argtypes = [C.POINTER(rt_camera), C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]
        if hasattr(L, "rt_shade_ids"):  # absent from older builds selected with RT2025_LIB for A/B runs
            L.rt_camera_rays_ids.argtypes = [C.POINTER(rt_camera), C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]
            L.rt_camera_rays_ids_device.argtypes = [C.POINTER(rt_camera), C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
            L.rt_world_hit_ids.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint64,
                                           C.c_uint32, C.c_void_p, C.POINTER(rt_stats)]
            L.rt_world_hit_ids_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double,
                                                  C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
            L.rt_shade_ids.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
            L.rt_shade_ids_device.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
        L.rt_render.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.POINTER(rt_render_opts), C.c_void_p,
                                C.POINTER(rt_stats)]
        L.rt_render_device.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.POINTER(rt_render_opts), C.c_void_p,
                                       C.c_void_p, C.POINTER(rt_stats)]
        L.rt_render_rgb8.argtypes = [C.c_void_p, C.POINTER(rt_camera), C.POINTER(rt_render_opts), C.c_void_p, C.POINTER(rt_stats)]
        L.rt_render_multi.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(rt_camera), C.POINTER(rt_render_opts), C.c_void_p,
                                      C.POINTER(rt_stats)]
        if hasattr(L, "rt_render_multi_rgb8"):  # absent from older builds selected with RT2025_LIB for A/B runs
            L.rt_render_multi_rgb8.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(rt_camera), C.POINTER(rt_render_opts), C.c_void_p,
                                               C.POINTER(rt_stats)]
        L.rt_tonemap.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p]
        L.rt_tonemap_device.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]
        L.rt_scene_get_info.argtypes = [C.c_void_p, C.POINTER(rt_scene_info)]
        L.rt_scene_get_ranks.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        _product = L
    return _product


def _d3(v):
    return (C.c_double * len(v))(*[float(x) for x in v])


class HostScene:
    """A flattened scene + camera produced by the host mirror (owns the native memory)."""

    def __init__(self, handle):
        if not handle:
            raise RtError("host: " + host_lib().rth_last_error().decode())
        self._h = handle
        self.desc = host_lib().rth_scene_desc(handle)
        self.camera = host_lib().rth_scene_camera(handle).contents

    def objects(self):
        d = self.desc.contents
        buf = (C.c_char * (d.n_objects * rt_object_dtype.itemsize)).from_address(d.objects)
        return np.frombuffer(buf, dtype=rt_object_dtype)

    def children(self):
        d = self.desc.contents
        buf = (C.c_uint32 * d.n_children).from_address(d.children)
        return np.frombuffer(buf, dtype=np.uint32)

    def __del__(self):
        try:
            if self._h:
                host_lib().rth_scene_free(self._h)
                self._h = None
        except Exception:
            pass


def named_scene(name, seed=1, params=()):
    """book2_final | cornell_glass | cornell_shipped | book1_final [width, spp, depth];
    tri_soup | sphere_soup [n]."""
    arr = (C.c_double * max(1, len(params)))(*params)
    return HostScene(host_lib().rth_scene_named(name.encode(), seed, arr, len(params)))


class Builder:
    """Scene construction with the reference's constructor names (SURVEY.md §8b)."""

    def __init__(self, seed=1):
        self.L = host_lib()
        self.b = self.L.rth_builder_new(seed)

    def __del__(self):
        try:
            self.L.rth_builder_free(self.b)
        except Exception:
            pass

    # textures
    def solid(self, r, g, b): return self.L.rth_tex_solid(self.b, r, g, b)
    def checker(self, scale, even, odd): return self.L.rth_tex_checker(self.b, scale, even, odd)
    def noise(self, scale): return self.L.rth_tex_noise(self.b, scale)
    def image_missing(self): return self.L.rth_tex_image_missing(self.b)

    def image(self, rgba, raw=False, linear_format=False):
        a = np.ascontiguousarray(rgba, dtype=np.float32)
        h, w, c = a.shape
        assert c == 4
        return self.L.rth_tex_image(self.b, w, h, a.ctypes.data, int(raw), int(linear_format))

    def gradient(self, bottom, top): return self.L.rth_tex_gradient(self.b, _d3(bottom), _d3(top))
    # materials
    def empty(self): return self.L.rth_mat_empty(self.b)
    def lambertian(self, tex): return self.L.rth_mat_lambertian(self.b, tex)
    def metal(self, albedo, fuzz): return self.L.rth_mat_metal(self.b, _d3(albedo), fuzz)
    def dielectric(self, tex, ri): return self.L.rth_mat_dielectric(self.b, tex, ri)
    def diffuse_light(self, tex, inner=RT_NONE): return self.L.rth_mat_diffuse_light(self.b, tex, inner)
    def isotropic(self, tex): return self.L.rth_mat_isotropic(self.b, tex)
    def transparent(self): return self.L.rth_mat_transparent(self.b)
    def mix(self, m1, m2, ratio): return self.L.rth_mat_mix(self.b, m1, m2, ratio)
    def mix_image(self, m1, m2, tex): return self.L.rth_mat_mix_image(self.b, m1, m2, tex)
    def portal(self, att, offset, quat): return self.L.rth_mat_portal(self.b, _d3(att), _d3(offset), _d3(quat))

    DISNEY_ORDER = ["roughness", "anisotropic", "sheen", "sheen_tint", "clearcoat", "clearcoat_gloss", "specular_tint", "metallic",
                    "ior", "flatness", "spec_trans", "diff_trans", "thin"]
    DISNEY_DEFAULTS = dict(roughness=0.5, anisotropic=0.0, sheen=0.0, sheen_tint=0.0, clearcoat=0.0, clearcoat_gloss=0.0,
                           specular_tint=0.0, metallic=0.0, ior=1.45, flatness=0.0, spec_trans=0.0, diff_trans=0.0, thin=0.0)

    def disney(self, base_color=(0.8, 0.8, 0.8), tex=RT_NONE, **params):
        """Disney::builder()...build() (material/disney.rs:718-805); tex = base-colour texture as the OBJ loader uses."""
        p = dict(self.DISNEY_DEFAULTS)
        for k, v in params.items():
            assert k in p, k
            p[k] = float(v)
        return self.L.rth_mat_disney(self.b, _d3(base_color), tex, _d3([p[k] for k in self.DISNEY_ORDER]))

    def remapped(self, inner, pos, uv, nrm, normal_tex=RT_NONE):
        """RemappedMaterial for one OBJ face (shapes/obj.rs:143-183): pos, nrm 3x3; uv 3x2."""
        uv3 = [[float(a), float(b), 0.0] for a, b in uv]
        flat = lambda m: _d3([x for row in m for x in row])
        return self.L.rth_mat_remapped(self.b, inner, flat(pos), flat(uv3), flat(nrm), normal_tex)

    def obj_face(self, inner, pos, uv, nrm, normal_tex=RT_NONE):
        """One face as load_object emits it: Triangle::new(p1, p2-p1, p3-p1, RemappedMaterial{..}); RT_NONE if degenerate."""
        m = self.remapped(inner, pos, uv, nrm, normal_tex)
        p1, p2, p3 = [np.asarray(p, dtype=np.float64) for p in pos]
        return self.triangle(p1, p2 - p1, p3 - p1, m)

    # shapes and containers
    def sphere(self, c, r, mat): return self.L.rth_sphere(self.b, _d3(c), r, mat)
    def sphere_moving(self, c1, c2, r, mat): return self.L.rth_sphere_moving(self.b, _d3(c1), _d3(c2), r, mat)
    def quad(self, q, u, v, mat): return self.L.rth_quad(self.b, _d3(q), _d3(u), _d3(v), mat)
    def triangle(self, q, u, v, mat): return self.L.rth_triangle(self.b, _d3(q), _d3(u), _d3(v), mat)
    def box(self, a, b, mat): return self.L.rth_box(self.b, _d3(a), _d3(b), mat)

    def list(self, ids, use_new=False):
        arr = (C.c_uint32 * max(1, len(ids)))(*ids)
        return self.L.rth_list(self.b, arr, len(ids), int(use_new))

    def bvh(self, ids):
        arr = (C.c_uint32 * max(1, len(ids)))(*ids)
        r = self.L.rth_bvh(self.b, arr, len(ids))
        if r == RT_NONE:
            raise RtError(self.L.rth_last_error().decode())
        return r

    def transform(self, child, offset=None, quat=None, scale=None):
        return self.L.rth_transform(self.b, child, _d3(offset) if offset is not None else None,
                                    _d3(quat) if quat is not None else None,
                                    _d3(scale) if scale is not None else None)

    def quat_axis_angle(self, axis, degrees):
        out = (C.c_double * 4)()
        self.L.rth_quat_from_axis_angle(_d3(axis), degrees, out)
        return list(out)

    def medium(self, boundary, density, tex): return self.L.rth_medium(self.b, boundary, density, tex)

    def finish(self, world, lights=RT_NONE, *, width=64, aspect=1.0, spp=4, max_depth=8, vfov=40.0,
               look_from=(0, 0, 5), look_at=(0, 0, 0), vup=(0, 1, 0), defocus_angle=0.0, focus_dist=10.0,
               background=RT_NONE, toon_map=0):
        cp = rth_camera_params()
        cp.aspect_ratio, cp.image_width, cp.samples_per_pixel, cp.max_depth = aspect, width, spp, max_depth
        cp.background_tex, cp.vertical_fov_in_degrees = background, vfov
        cp.look_from[:], cp.look_at[:], cp.vec_up[:] = list(map(float, look_from)), list(map(float, look_at)), list(map(float, vup))
        cp.defocus_angle_in_degrees, cp.focus_distance, cp.toon_map = defocus_angle, focus_dist, toon_map
        return HostScene(self.L.rth_builder_finish(self.b, world, lights, C.byref(cp)))


def make_rays(origins, directions, times=None):
    n = len(origins)
    rays = np.zeros(n, dtype=rt_ray_dtype)
    rays["origin"] = origins
    rays["direction"] = directions
    if times is not None:
        rays["time"] = times
    return rays


def _check(rc, L):
    if rc != 0:
        raise RtError(f"rt2025 error {rc}: {L.rt_last_error().decode()}")


class Scene:
    """Device-resident compiled scene (rt_scene_create / rt_scene_destroy)."""

    def __init__(self, host_scene, flags=0, device=-1):
        self.L = product_lib()
        self.host = host_scene
        opts = rt_build_opts(C.sizeof(rt_build_opts), flags, device, 0)
        h = C.c_void_p()
        _check(self.L.rt_scene_create(host_scene.desc, C.byref(opts), C.byref(h)), self.L)
        self.h = h

    def close(self):
        if self.h:
            self.L.rt_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        i = rt_scene_info()
        _check(self.L.rt_scene_get_info(self.h, C.byref(i)), self.L)
        return i

    def ranks(self):
        n = self.host.desc.contents.n_objects
        out = np.empty(n, dtype=np.uint32)
        _check(self.L.rt_scene_get_ranks(self.h, out.ctypes.data, n), self.L)
        return out

    def closest_hit(self, rays, t_min=1e-8, t_max=float("inf"), flags=0):
        rays = np.ascontiguousarray(rays, dtype=rt_ray_dtype)
        out = np.empty(len(rays), dtype=rt_hit_dtype)
        st = rt_stats()
        _check(self.L.rt_closest_hit(self.h, rays.ctypes.data, len(rays), t_min, t_max, flags, out.ctypes.data,
                                     C.byref(st)), self.L)
        return out, st

    def closest_hit_device(self, d_rays_ptr, n, d_out_ptr, t_min=1e-8, t_max=float("inf"), flags=0, stream=None):
        st = rt_stats()
        _check(self.L.rt_closest_hit_device(self.h, d_rays_ptr, n, t_min, t_max, flags, d_out_ptr, stream,
                                            C.byref(st)), self.L)
        return st

    def occluded(self, rays, t_min=1e-8, t_max=float("inf"), flags=0):
        """rt_occluded: for each ray, is there a surface hit with t in [t_min, t_max]?  `t_max` is a scalar or one value per ray.
        Returns (bool array, stats)."""
        rays = np.ascontiguousarray(rays, dtype=rt_ray_dtype)
        out = np.empty(len(rays), dtype=np.uint8)
        per_ray = None
        if np.ndim(t_max) != 0:
            per_ray = np.ascontiguousarray(t_max, dtype=np.float64)
            if per_ray.shape != (len(rays),):
                raise ValueError(f"t_max has shape {per_ray.shape}; a scalar or {len(rays)} values expected")
            t_max = float("inf")
        st = rt_stats()
        _check(self.L.rt_occluded(self.h, rays.ctypes.data, None if per_ray is None else per_ray.ctypes.data, len(rays), t_min, t_max,
                                  flags, out.ctypes.data, C.byref(st)), self.L)
        return out.view(np.bool_), st

    def occluded_device(self, d_rays_ptr, n, d_out_ptr, d_t_max_ptr=None, t_min=1e-8, t_max=float("inf"), flags=0, stream=None):
        """rt_occluded_device: n bytes at d_out_ptr; d_t_max_ptr (n doubles) overrides the scalar t_max."""
        st = rt_stats()
        _check(self.L.rt_occluded_device(self.h, d_rays_ptr, d_t_max_ptr, n, t_min, t_max, flags, d_out_ptr, stream, C.byref(st)), self.L)
        return st

    def transmittance(self, rays, t_min=1e-8, t_max=float("inf"), flags=0):
        """rt_transmittance: for each ray, the probability that nothing in [t_min, t_max] stops it - 0 behind a surface, else the
        product of the media's exp(L / neg_inv_density).  `t_max` is a scalar or one value per ray.  Returns (float64 array, stats)."""
        rays = np.ascontiguousarray(rays, dtype=rt_ray_dtype)
        out = np.empty(len(rays), dtype=np.float64)
        per_ray = None
        if np.ndim(t_max) != 0:
            per_ray = np.ascontiguousarray(t_max, dtype=np.float64)
            if per_ray.shape != (len(rays),):
                raise ValueError(f"t_max has shape {per_ray.shape}; a scalar or {len(rays)} values expected")
            t_max = float("inf")
        st = rt_stats()
        _check(self.L.rt_transmittance(self.h, rays.ctypes.data, None if per_ray is None else per_ray.ctypes.data, len(rays), t_min, t_max,
                                       flags, out.ctypes.data, C.byref(st)), self.L)
        return out, st

    def transmittance_device(self, d_rays_ptr, n, d_out_ptr, d_t_max_ptr=None, t_min=1e-8, t_max=float("inf"), flags=0, stream=None):
        """rt_transmittance_device: n doubles at d_out_ptr; d_t_max_ptr (n doubles) overrides the scalar t_max."""
        st = rt_stats()
        _check(self.L.rt_transmittance_device(self.h, d_rays_ptr, d_t_max_ptr, n, t_min, t_max, flags, d_out_ptr, stream, C.byref(st)),
               self.L)
        return st

    def world_hit(self, rays, t_min=1e-8, t_max=float("inf"), seed=0, segment=0, flags=0):
        """rt_world_hit: for each ray the HitRecord world.hit(ray, [t_min, t_max]) returns, media sampled with the addressed draws
        of (seed, pixel = ray index, sample 0, segment).  `t_max` is a scalar or one value per ray.  Returns
        (rt_hit_record_dtype array, stats)."""
        rays = np.ascontiguousarray(rays, dtype=rt_ray_dtype)
        out = np.empty(len(rays), dtype=rt_hit_record_dtype)
        per_ray = None
        if np.ndim(t_max) != 0:
            per_ray = np.ascontiguousarray(t_max, dtype=np.float64)
            if per_ray.shape != (len(rays),):
                raise ValueError(f"t_max has shape {per_ray.shape}; a scalar or {len(rays)} values expected")
            t_max = float("inf")
        st = rt_stats()
        _check(self.L.rt_world_hit(self.h, rays.ctypes.data, None if per_ray is None else per_ray.ctypes.data, len(rays), t_min, t_max, seed,
                                   segment, flags, out.ctypes.data, C.byref(st)), self.L)
        return out, st

    def world_hit_device(self, d_rays_ptr, n, d_out_ptr, d_t_max_ptr=None, t_min=1e-8, t_max=float("inf"), seed=0, segment=0, flags=0,
                         stream=None):
        """rt_world_hit_device: n 96-byte rt_hit_record at d_out_ptr; d_t_max_ptr (n doubles) overrides the scalar t_max."""
        st = rt_stats()
        _check(self.L.rt_world_hit_device(self.h, d_rays_ptr, d_t_max_ptr, n, t_min, t_max, seed, segment, flags, d_out_ptr, stream,
                                          C.byref(st)), self.L)
        return st

    def shade(self, records, rays, beta, radiance, state, seed=0, segment=0, camera=None, flags=0):
        """rt_shade: the step of ray_color after world.hit for the rows with state & RT_PATH_ALIVE, from the records world_hit
        returned for `rays`, with the draws of (seed, pixel = row index, sample 0, segment).  Updates the caller's arrays in place:
        rays (rt_ray_dtype) and beta (n x 3 float64) of the paths that go on, radiance (n x 3 float64, the segment's contribution
        is added) and state (uint8 RT_PATH_* bits).  Returns the stats."""
        cam = camera if camera is not None else self.host.camera
        records = np.ascontiguousarray(records, dtype=rt_hit_record_dtype)
        n = len(records)
        for name, a, dt, shape in (("rays", rays, rt_ray_dtype, (n,)), ("beta", beta, np.float64, (n, 3)), ("radiance", radiance, np.float64, (n, 3)),
                                   ("state", state, np.uint8, (n,))):
            if not (isinstance(a, np.ndarray) and a.dtype == dt and a.shape == shape and a.flags.c_contiguous and a.flags.writeable):
                raise ValueError(f"{name}: a writeable C-contiguous {np.dtype(dt)} array of shape {shape} is updated in place")
        st = rt_stats()
        _check(self.L.rt_shade(self.h, C.byref(cam), records.ctypes.data, n, seed, segment, flags, rays.ctypes.data, beta.ctypes.data,
                               radiance.ctypes.data, state.ctypes.data, C.byref(st)), self.L)
        return st

    def shade_device(self, d_records_ptr, n, d_rays_ptr, d_beta_ptr, d_radiance_ptr, d_state_ptr, seed=0, segment=0, camera=None, flags=0,
                     stream=None):
        """rt_shade_device: the same on device buffers (n records, n rays, n x 3 beta and radiance doubles, n state bytes)."""
        cam = camera if camera is not None else self.host.camera
        st = rt_stats()
        _check(self.L.rt_shade_device(self.h, C.byref(cam), d_records_ptr, n, seed, segment, flags, d_rays_ptr, d_beta_ptr, d_radiance_ptr,
                                      d_state_ptr, stream, C.byref(st)), self.L)
        return st

    def world_hit_ids(self, rays, ids, t_min=1e-8, t_max=float("inf"), seed=0, flags=0):
        """rt_world_hit_ids: world_hit with the draws of ray i addressed by ids[i] (rt_path_id_dtype: pixel, sample, segment) instead
        of (i, 0, segment).  Returns (rt_hit_record_dtype array, stats)."""
        rays = np.ascontiguousarray(rays, dtype=rt_ray_dtype)
        ids = np.ascontiguousarray(ids, dtype=rt_path_id_dtype)
        if ids.shape != (len(rays),):
            raise ValueError(f"ids has shape {ids.shape}; {len(rays)} path ids expected")
        out = np.empty(len(rays), dtype=rt_hit_record_dtype)
        per_ray = None
        if np.ndim(t_max) != 0:
            per_ray = np.ascontiguousarray(t_max, dtype=np.float64)
            if per_ray.shape != (len(rays),):
                raise ValueError(f"t_max has shape {per_ray.shape}; a scalar or {len(rays)} values expected")
            t_max = float("inf")
        st = rt_stats()
        _check(self.L.rt_world_hit_ids(self.h, rays.ctypes.data, ids.ctypes.data, None if per_ray is None else per_ray.ctypes.data, len(rays),
                                       t_min, t_max, seed, flags, out.ctypes.data, C.byref(st)), self.L)
        return out, st

    def world_hit_ids_device(self, d_rays_ptr, d_ids_ptr, n, d_out_ptr, d_t_max_ptr=None, t_min=1e-8, t_max=float("inf"), seed=0, flags=0,
                             stream=None):
        """rt_world_hit_ids_device: the same on device buffers (n rays, n 16-byte path ids, n records out)."""
        st = rt_stats()
        _check(self.L.rt_world_hit_ids_device(self.h, d_rays_ptr, d_ids_ptr, d_t_max_ptr, n, t_min, t_max, seed, flags, d_out_ptr, stream,
                                              C.byref(st)), self.L)
        return st

    def shade_ids(self, records, ids, rays, beta, radiance, state, seed=0, camera=None, flags=0):
        """rt_shade_ids: shade with the draws and the segment of row i taken from ids[i] (rt_path_id_dtype).  Updates ids in place
        with rays, beta, radiance and state: the rows that go on get ids["segment"] + 1.  radiance is still per row.  Returns the
        stats."""
        cam = camera if camera is not None else self.host.camera
        records = np.ascontiguousarray(records, dtype=rt_hit_record_dtype)
        n = len(records)
        for name, a, dt, shape in (("ids", ids, rt_path_id_dtype, (n,)), ("rays", rays, rt_ray_dtype, (n,)), ("beta", beta, np.float64, (n, 3)),
                                   ("radiance", radiance, np.float64, (n, 3)), ("state", state, np.uint8, (n,))):
            if not (isinstance(a, np.ndarray) and a.dtype == dt and a.shape == shape and a.flags.c_contiguous and a.flags.writeable):
                raise ValueError(f"{name}: a writeable C-contiguous {np.dtype(dt)} array of shape {shape} is updated in place")
        st = rt_stats()
        _check(self.L.rt_shade_ids(self.h, C.byref(cam), records.ctypes.data, ids.ctypes.data, n, seed, flags, rays.ctypes.data,
                                   beta.ctypes.data, radiance.ctypes.data, state.ctypes.data, C.byref(st)), self.L)
        return st

    def shade_ids_device(self, d_records_ptr, d_ids_ptr, n, d_rays_ptr, d_beta_ptr, d_radiance_ptr, d_state_ptr, seed=0, camera=None, flags=0,
                         stream=None):
        """rt_shade_ids_device: the same on device buffers (n records, n path ids, n rays, n x 3 beta and radiance doubles, n state
        bytes)."""
        cam = camera if camera is not None else self.host.camera
        st = rt_stats()
        _check(self.L.rt_shade_ids_device(self.h, C.byref(cam), d_records_ptr, d_ids_ptr, n, seed, flags, d_rays_ptr, d_beta_ptr,
                                          d_radiance_ptr, d_state_ptr, stream, C.byref(st)), self.L)
        return st

    def render_opts(self, seed=1, accum_type=RT_ACCUM_F64, part_index=0, part_count=1, sample_begin=0, sample_end=0,
                    flags=0, max_paths_in_flight=0, no_binning=False, classic_media_order=False):
        o = rt_render_opts()
        o.struct_size = C.sizeof(rt_render_opts)
        o.flags, o.seed, o.accum_type = flags, seed, accum_type
        o.part_index, o.part_count = part_index, part_count
        o.sample_begin, o.sample_end, o.max_paths_in_flight = sample_begin, sample_end, max_paths_in_flight
        # A/B switches: bit 0 = one general shade kernel instead of one per class, bit 1 = sample the media after extend
        # (the order of the reference's loop) instead of before it
        o.reserved[0] = (1 if no_binning else 0) | (2 if classic_media_order else 0)
        return o

    def render(self, camera=None, **kw):
        """Camera::render up to the 8-bit encode: returns (H, W, 3) mean linear radiance + stats."""
        cam = camera if camera is not None else self.host.camera
        o = self.render_opts(**kw)
        dt = np.float64 if o.accum_type == RT_ACCUM_F64 else np.float32
        img = np.zeros((cam.image_height, cam.image_width, 3), dtype=dt)
        st = rt_stats()
        _check(self.L.rt_render(self.h, C.byref(cam), C.byref(o), img.ctypes.data, C.byref(st)), self.L)
        return img, st

    def render_rgb8(self, camera=None, **kw):
        """Camera::render: the RgbImage bytes (H, W, 3) straight from the device."""
        cam = camera if camera is not None else self.host.camera
        o = self.render_opts(**kw)
        img = np.zeros((cam.image_height, cam.image_width, 3), dtype=np.uint8)
        st = rt_stats()
        _check(self.L.rt_render_rgb8(self.h, C.byref(cam), C.byref(o), img.ctypes.data, C.byref(st)), self.L)
        return img, st

    def render_device(self, d_accum_ptr, camera=None, stream=None, **kw):
        cam = camera if camera is not None else self.host.camera
        o = self.render_opts(**kw)
        st = rt_stats()
        _check(self.L.rt_render_device(self.h, C.byref(cam), C.byref(o), d_accum_ptr, stream, C.byref(st)), self.L)
        return st


def render_multi_rgb8(scenes, camera=None, **kw):
    """rt_render_multi_rgb8: Camera::render on several GPUs of one process -> RgbImage bytes (H, W, 3)."""
    L = product_lib()
    cam = camera if camera is not None else scenes[0].host.camera
    o = scenes[0].render_opts(**kw)
    img = np.zeros((cam.image_height, cam.image_width, 3), dtype=np.uint8)
    handles = (C.c_void_p * len(scenes))(*[s.h for s in scenes])
    st = rt_stats()
    _check(L.rt_render_multi_rgb8(handles, len(scenes), C.byref(cam), C.byref(o), img.ctypes.data, C.byref(st)), L)
    return img, st


def render_multi(scenes, camera=None, **kw):
    """rt_render_multi: one process, scenes[i] on distinct GPUs; GPU 0 sums the partial frames through peer mappings."""
    L = product_lib()
    cam = camera if camera is not None else scenes[0].host.camera
    o = scenes[0].render_opts(**kw)
    dt = np.float64 if o.accum_type == RT_ACCUM_F64 else np.float32
    img = np.zeros((cam.image_height, cam.image_width, 3), dtype=dt)
    handles = (C.c_void_p * len(scenes))(*[s.h for s in scenes])
    st = rt_stats()
    _check(L.rt_render_multi(handles, len(scenes), C.byref(cam), C.byref(o), img.ctypes.data, C.byref(st)), L)
    return img, st


def camera_rays(camera, seed, sample=0):
    """rt_camera_rays: Camera::get_ray of stratum `sample` through every pixel, image_width * image_height rays in the render's
    pixel order (pixel = j * image_width + i)."""
    L = product_lib()
    out = np.empty(camera.image_width * camera.image_height, dtype=rt_ray_dtype)
    _check(L.rt_camera_rays(C.byref(camera), seed, sample, out.ctypes.data), L)
    return out


def camera_rays_device(camera, seed, sample, d_out_ptr, stream=None):
    """rt_camera_rays_device: the same into image_width * image_height rays at d_out_ptr on the current device."""
    L = product_lib()
    _check(L.rt_camera_rays_device(C.byref(camera), seed, sample, d_out_ptr, stream), L)


def camera_rays_ids(camera, seed, ids):
    """rt_camera_rays_ids: out[i] = Camera::get_ray of pixel ids[i]["pixel"] (j * image_width + i) and stratum ids[i]["sample"]."""
    L = product_lib()
    ids = np.ascontiguousarray(ids, dtype=rt_path_id_dtype)
    out = np.empty(len(ids), dtype=rt_ray_dtype)
    _check(L.rt_camera_rays_ids(C.byref(camera), seed, ids.ctypes.data, len(ids), out.ctypes.data), L)
    return out


def camera_rays_ids_device(camera, seed, d_ids_ptr, n, d_out_ptr, stream=None):
    """rt_camera_rays_ids_device: the same from n path ids at d_ids_ptr into n rays at d_out_ptr on the current device."""
    L = product_lib()
    _check(L.rt_camera_rays_ids_device(C.byref(camera), seed, d_ids_ptr, n, d_out_ptr, stream), L)


def tonemap_device(d_accum_ptr, n_pixels, d_rgb_ptr, toon_map=0, accum_type=RT_ACCUM_F32, stream=None):
    """rt_tonemap_device: Color::to_rgb on a framebuffer that already lives on the current device."""
    L = product_lib()
    _check(L.rt_tonemap_device(d_accum_ptr, accum_type, n_pixels, toon_map, d_rgb_ptr, stream), L)


def tonemap(accum, toon_map=0):
    """Color::to_rgb over an image of mean linear radiance -> uint8 (H, W, 3)."""
    L = product_lib()
    a = np.ascontiguousarray(accum)
    t = RT_ACCUM_F64 if a.dtype == np.float64 else RT_ACCUM_F32
    if t == RT_ACCUM_F32:
        a = a.astype(np.float32, copy=False)
    out = np.empty(a.shape, dtype=np.uint8)
    _check(L.rt_tonemap(a.ctypes.data, t, a.size // 3, toon_map, out.ctypes.data), L)
    return out
