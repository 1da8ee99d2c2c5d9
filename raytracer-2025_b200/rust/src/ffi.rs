//! `#[repr(C)]` mirrors of include/rt2025.h (ABI version 1).  Field order and types must match the
//! header exactly; tests/test_abi.py checks the C side of every size.
#![allow(non_camel_case_types, dead_code)]
use core::ffi::{c_char, c_void};

pub const RT_ABI_VERSION: u32 = 1;
pub const RT_NONE: u32 = 0xFFFF_FFFF;

pub const RT_OBJ_SPHERE: u32 = 1;
pub const RT_OBJ_QUAD: u32 = 2;
pub const RT_OBJ_TRIANGLE: u32 = 3;
pub const RT_OBJ_LIST: u32 = 4;
pub const RT_OBJ_BVH: u32 = 5;
pub const RT_OBJ_TRANSFORM: u32 = 6;
pub const RT_OBJ_MEDIUM: u32 = 7;

pub const RT_MAT_EMPTY: u32 = 0;
pub const RT_MAT_LAMBERTIAN: u32 = 1;
pub const RT_MAT_METAL: u32 = 2;
pub const RT_MAT_DIELECTRIC: u32 = 3;
pub const RT_MAT_DIFFUSE_LIGHT: u32 = 4;
pub const RT_MAT_ISOTROPIC: u32 = 5;
pub const RT_MAT_TRANSPARENT: u32 = 6;
pub const RT_MAT_MIX: u32 = 7;
pub const RT_MAT_PORTAL: u32 = 8;
pub const RT_MAT_DISNEY: u32 = 9;
pub const RT_MAT_REMAPPED: u32 = 10;

pub const RT_TEX_SOLID: u32 = 0;
pub const RT_TEX_CHECKER: u32 = 1;
pub const RT_TEX_IMAGE: u32 = 2;
pub const RT_TEX_NOISE: u32 = 3;
pub const RT_TEX_GRADIENT_Y: u32 = 4;

pub const RT_IMG_LINEAR: u32 = 1;
pub const RT_IMG_INTERP: u32 = 2;
pub const RT_ACCUM_F32: u32 = 0;
pub const RT_ACCUM_F64: u32 = 1;
// order of the DisneyParameters scalars in rt_material.v (rt2025.h)
pub const RT_DISNEY_ROUGHNESS: usize = 0;
pub const RT_DISNEY_ANISOTROPIC: usize = 1;
pub const RT_DISNEY_SHEEN: usize = 2;
pub const RT_DISNEY_SHEEN_TINT: usize = 3;
pub const RT_DISNEY_CLEARCOAT: usize = 4;
pub const RT_DISNEY_CLEARCOAT_GLOSS: usize = 5;
pub const RT_DISNEY_SPECULAR_TINT: usize = 6;
pub const RT_DISNEY_METALLIC: usize = 7;
pub const RT_DISNEY_IOR: usize = 8;
pub const RT_DISNEY_FLATNESS: usize = 9;
pub const RT_DISNEY_SPEC_TRANS: usize = 10;
pub const RT_DISNEY_DIFF_TRANS: usize = 11;
pub const RT_DISNEY_THIN: usize = 12;

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_object { pub kind: u32, pub material: u32, pub first_child: u32, pub child_count: u32, pub data: u32, pub reserved: u32, pub bbox: [f64; 6] }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_sphere { pub center: [f64; 3], pub center_vec: [f64; 3], pub radius: f64, pub reserved: f64 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_planar { pub anchor: [f64; 3], pub u: [f64; 3], pub v: [f64; 3], pub normal: [f64; 3], pub parm_d: f64, pub w: [f64; 3], pub area: f64, pub reserved: f64 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_transform { pub offset: [f64; 3], pub quat: [f64; 4], pub scale: [f64; 3] }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_medium { pub neg_inv_density: f64, pub reserved: f64 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_material { pub kind: u32, pub tex: u32, pub inner: u32, pub inner2: u32, pub color: [f64; 3], pub param: f64, pub v: [f64; 16] }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_remap { pub tex_ori: [f64; 3], pub tex_u: [f64; 3], pub tex_v: [f64; 3], pub u_vec: [f64; 3], pub v_vec: [f64; 3], pub normal: [[f64; 3]; 3], pub has_uv_vecs: u32, pub normal_tex: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_texture { pub kind: u32, pub a: u32, pub b: u32, pub reserved: u32, pub color: [f64; 3], pub color2: [f64; 3], pub scale: f64, pub reserved2: f64 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_image { pub width: u32, pub height: u32, pub flags: u32, pub reserved: u32, pub texel_offset: u64 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct rt_perlin { pub randvec: [[f64; 3]; 256], pub perm_x: [u32; 256], pub perm_y: [u32; 256], pub perm_z: [u32; 256] }

#[repr(C)]
pub struct rt_scene_desc {
    pub version: u32, pub struct_size: u32, pub world_root: u32, pub lights_root: u32,
    pub n_objects: u32, pub n_children: u32, pub n_spheres: u32, pub n_planars: u32,
    pub n_transforms: u32, pub n_media: u32, pub n_materials: u32, pub n_textures: u32,
    pub n_images: u32, pub n_perlins: u32, pub n_texels: u64, pub n_remaps: u32, pub reserved0: u32,
    pub objects: *const rt_object, pub children: *const u32, pub spheres: *const rt_sphere, pub planars: *const rt_planar,
    pub transforms: *const rt_transform, pub media: *const rt_medium, pub materials: *const rt_material,
    pub textures: *const rt_texture, pub images: *const rt_image, pub texels: *const f32, pub perlins: *const rt_perlin, pub remaps: *const rt_remap,
}

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_camera {
    pub image_width: u32, pub image_height: u32, pub sqrt_spp: u32, pub max_depth: u32, pub background_tex: u32, pub toon_map: u32,
    pub recip_sqrt_spp: f64, pub pixel_sample_scale: f64,
    pub center: [f64; 3], pub pixel00_loc: [f64; 3], pub pixel_delta_u: [f64; 3], pub pixel_delta_v: [f64; 3],
    pub defocus_angle_in_degrees: f64, pub defocus_disk_u: [f64; 3], pub defocus_disk_v: [f64; 3],
}
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_build_opts { pub struct_size: u32, pub flags: u32, pub device: i32, pub reserved: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_render_opts {
    pub struct_size: u32, pub flags: u32, pub seed: u64, pub accum_type: u32, pub part_index: u32, pub part_count: u32,
    pub sample_begin: u32, pub sample_end: u32, pub max_paths_in_flight: u32, pub reserved: [u32; 4],
}
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_stats {
    pub paths: u64, pub segments: u64, pub node_visits: u64, pub prim_tests: u64, pub errors: u64, pub kernel_launches: u64,
    pub ms_total: f64, pub ms_raygen: f64, pub ms_extend: f64, pub ms_shade: f64, pub ms_other: f64, pub iterations: u64, pub reserved: [u64; 4],
}
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_ray { pub origin: [f64; 3], pub direction: [f64; 3], pub time: f64 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_hit { pub t: f64, pub prim_id: u32, pub inst_id: u32, pub u: f32, pub v: f32 }
pub const RT_HIT_MISS: u32 = 0;
pub const RT_HIT_SURFACE: u32 = 1;
pub const RT_HIT_MEDIUM: u32 = 2;
pub const RT_PATH_ALIVE: u8 = 1;
pub const RT_PATH_ERROR: u8 = 2;
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct rt_hit_record {
    pub t: f64, pub p: [f64; 3], pub normal: [f64; 3], pub u: f64, pub v: f64,
    pub kind: u32, pub front_face: u32, pub prim_id: u32, pub inst_id: u32, pub material: u32, pub reserved: u32,
}
#[repr(C)] pub struct rt_scene { _private: [u8; 0] }

extern "C" {
    pub fn rt_scene_create(desc: *const rt_scene_desc, opts: *const rt_build_opts, out: *mut *mut rt_scene) -> i32;
    pub fn rt_scene_destroy(scene: *mut rt_scene) -> i32;
    pub fn rt_closest_hit(scene: *const rt_scene, rays: *const rt_ray, n: u64, t_min: f64, t_max: f64, flags: u32, out: *mut rt_hit, stats: *mut rt_stats) -> i32;
    pub fn rt_occluded(scene: *const rt_scene, rays: *const rt_ray, t_max_per_ray: *const f64, n: u64, t_min: f64, t_max: f64, flags: u32, out: *mut u8, stats: *mut rt_stats) -> i32;
    pub fn rt_occluded_device(scene: *const rt_scene, d_rays: *const rt_ray, d_t_max_per_ray: *const f64, n: u64, t_min: f64, t_max: f64, flags: u32, d_out: *mut u8, stream: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_transmittance(scene: *const rt_scene, rays: *const rt_ray, t_max_per_ray: *const f64, n: u64, t_min: f64, t_max: f64, flags: u32, out: *mut f64, stats: *mut rt_stats) -> i32;
    pub fn rt_transmittance_device(scene: *const rt_scene, d_rays: *const rt_ray, d_t_max_per_ray: *const f64, n: u64, t_min: f64, t_max: f64, flags: u32, d_out: *mut f64, stream: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_world_hit(scene: *const rt_scene, rays: *const rt_ray, t_max_per_ray: *const f64, n: u64, t_min: f64, t_max: f64, seed: u64, segment: u32, flags: u32, out: *mut rt_hit_record, stats: *mut rt_stats) -> i32;
    pub fn rt_world_hit_device(scene: *const rt_scene, d_rays: *const rt_ray, d_t_max_per_ray: *const f64, n: u64, t_min: f64, t_max: f64, seed: u64, segment: u32, flags: u32, d_out: *mut rt_hit_record, stream: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_shade(scene: *const rt_scene, cam: *const rt_camera, records: *const rt_hit_record, n: u64, seed: u64, segment: u32, flags: u32, rays: *mut rt_ray, beta: *mut f64, radiance: *mut f64, state: *mut u8, stats: *mut rt_stats) -> i32;
    pub fn rt_shade_device(scene: *const rt_scene, cam: *const rt_camera, d_records: *const rt_hit_record, n: u64, seed: u64, segment: u32, flags: u32, d_rays: *mut rt_ray, d_beta: *mut f64, d_radiance: *mut f64, d_state: *mut u8, stream: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_camera_rays(cam: *const rt_camera, seed: u64, sample: u32, out: *mut rt_ray) -> i32;
    pub fn rt_camera_rays_device(cam: *const rt_camera, seed: u64, sample: u32, d_out: *mut rt_ray, stream: *mut c_void) -> i32;
    pub fn rt_render(scene: *const rt_scene, cam: *const rt_camera, opts: *const rt_render_opts, accum: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_render_device(scene: *const rt_scene, cam: *const rt_camera, opts: *const rt_render_opts, d_accum: *mut c_void, stream: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_render_rgb8(scene: *const rt_scene, cam: *const rt_camera, opts: *const rt_render_opts, rgb: *mut u8, stats: *mut rt_stats) -> i32;
    pub fn rt_render_multi(scenes: *const *mut rt_scene, n_scenes: u32, cam: *const rt_camera, opts: *const rt_render_opts, accum: *mut c_void, stats: *mut rt_stats) -> i32;
    pub fn rt_render_multi_rgb8(scenes: *const *mut rt_scene, n_scenes: u32, cam: *const rt_camera, opts: *const rt_render_opts, rgb: *mut u8, stats: *mut rt_stats) -> i32;
    pub fn rt_tonemap(accum: *const c_void, accum_type: u32, n_pixels: u64, toon_map: u32, rgb: *mut u8) -> i32;
    pub fn rt_tonemap_device(d_accum: *const c_void, accum_type: u32, n_pixels: u64, toon_map: u32, d_rgb: *mut u8, stream: *mut c_void) -> i32;
    pub fn rt_last_error() -> *const c_char;
    pub fn rt_abi_version() -> u32;
    pub fn rt_device_count() -> i32;
}

pub fn check(rc: i32) {
    if rc != 0 {
        let msg = unsafe { std::ffi::CStr::from_ptr(rt_last_error()) }.to_string_lossy().into_owned();
        panic!("rt2025 error {rc}: {msg}"); // the reference's failure mode is a panic everywhere
    }
}
