//! `#[repr(C)]` mirrors of include/rt1w.h (ABI version 1), one to one.
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_void};

pub const RT1W_OK: i32 = 0;

// rt1w_node_type
pub const RT1W_NODE_SPHERE: i32 = 0;
pub const RT1W_NODE_MOVING_SPHERE: i32 = 1;
pub const RT1W_NODE_XY_RECT: i32 = 2;
pub const RT1W_NODE_XZ_RECT: i32 = 3;
pub const RT1W_NODE_YZ_RECT: i32 = 4;
pub const RT1W_NODE_AABOX: i32 = 5;
pub const RT1W_NODE_TRANSLATE: i32 = 6;
pub const RT1W_NODE_ROTATE_Y: i32 = 7;
pub const RT1W_NODE_FLIP_FACE: i32 = 8;
pub const RT1W_NODE_CONSTANT_MEDIUM: i32 = 9;
pub const RT1W_NODE_BVH: i32 = 10;
// rt1w_material_type
pub const RT1W_MAT_LAMBERTIAN: i32 = 0;
pub const RT1W_MAT_METAL: i32 = 1;
pub const RT1W_MAT_DIELECTRIC: i32 = 2;
pub const RT1W_MAT_DIFFUSE_LIGHT: i32 = 3;
pub const RT1W_MAT_ISOTROPIC: i32 = 4;
pub const RT1W_MAT_NONE: i32 = 5;
// rt1w_texture_type
pub const RT1W_TEX_SOLID: i32 = 0;
pub const RT1W_TEX_CHECKER: i32 = 1;
pub const RT1W_TEX_NOISE: i32 = 2;
pub const RT1W_TEX_IMAGE: i32 = 3;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_node {
    pub type_: i32,
    pub material: i32,
    pub child_begin: i32,
    pub child_count: i32,
    pub p: [f64; 10],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_material {
    pub type_: i32,
    pub texture: i32,
    pub albedo: [f64; 3],
    pub fuzz: f64,
    pub ir: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_texture {
    pub type_: i32,
    pub odd: i32,
    pub even: i32,
    pub table: i32,
    pub color: [f64; 3],
    pub scale: f64,
}
#[repr(C)]
#[derive(Clone)]
pub struct rt1w_perlin {
    pub ranvec: [[f64; 3]; 256],
    pub perm_x: [i32; 256],
    pub perm_y: [i32; 256],
    pub perm_z: [i32; 256],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_image {
    pub rgb8: *const u8,
    pub width: i32,
    pub height: i32,
}
#[repr(C)]
pub struct rt1w_scene_desc {
    pub nodes: *const rt1w_node,
    pub n_nodes: i32,
    pub children: *const i32,
    pub n_children: i32,
    pub materials: *const rt1w_material,
    pub n_materials: i32,
    pub textures: *const rt1w_texture,
    pub n_textures: i32,
    pub perlins: *const rt1w_perlin,
    pub n_perlins: i32,
    pub images: *const rt1w_image,
    pub n_images: i32,
    pub world: i32,
    pub has_lights: i32,
    pub lights: *const i32,
    pub n_lights: i32,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_camera {
    pub origin: [f64; 3],
    pub lower_left_corner: [f64; 3],
    pub horizontal: [f64; 3],
    pub vertical: [f64; 3],
    pub u: [f64; 3],
    pub v: [f64; 3],
    pub w: [f64; 3],
    pub lens_radius: f64,
    pub time0: f64,
    pub time1: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_render_params {
    pub width: i32,
    pub height: i32,
    pub sample_begin: i32,
    pub sample_end: i32,
    pub max_depth: i32,
    pub flags: u32,
    pub seed: u64,
    pub background: [f64; 3],
    pub stat_clamp: f64,
    pub pool_paths: i32,
    pub reserved: i32,
}
// the denoiser's parameters (include/rt1w.h: the filter's definition); a null pointer means the defaults (5, 0, 4, 128, 1)
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_denoise_params {
    pub iterations: i32,
    pub reserved: i32,
    pub sigma_luminance: f64,
    pub sigma_normal: f64,
    pub sigma_depth: f64,
}
// light groups: group_of_node[node] for the leaf nodes with a DiffuseLight material (the other entries are ignored), the
// background group for every other ending of a path; reserved = 0
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_light_groups {
    pub group_of_node: *const i32,
    pub n_nodes: i32,
    pub n_groups: i32,
    pub background_group: i32,
    pub reserved: i32,
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rt1w_render_stats {
    pub paths: u64,
    pub rays: u64,
    pub waves: u64,
    pub launches: u64,
    pub render_ms: f64,
    pub kernel_ms: [f64; 7],
    pub kernel_launches: [u64; 7],
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rt1w_scene_info {
    pub n_prims: i32,
    pub n_bvh_nodes: i32,
    pub n_frames: i32,
    pub n_lights: i32,
    pub bvh_depth: i32,
    pub material_mask: i32,
    pub build_ms: f64,
    pub upload_ms: f64,
    pub sah_cost: f64,
    pub n_wide_nodes: i32,
    pub wide_depth: i32,
    pub wide_default: i32,
    pub n_global_prims: i32,
    pub wide_children: f64,
    pub flat_plan: i32,
}
/// One lowered primitive in primitive-id order (the ids `rt1w_trace_closest` reports).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rt1w_flat_prim {
    pub kind: i32,
    pub node: i32,
    pub material: i32,
    pub frame: i32,
    pub flags: i32,
    pub boundary: i32,
    pub p: [f64; 10],
    pub bbox_min: [f64; 3],
    pub bbox_max: [f64; 3],
    pub time0: f64,
    pub time1: f64,
}
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rt1w_ray {
    pub origin: [f32; 3],
    pub direction: [f32; 3],
    pub time: f32,
}
pub const RT1W_COMM_ID_BYTES: usize = 128;
pub enum rt1w_context {}
pub enum rt1w_scene {}

extern "C" {
    pub fn rt1w_abi_version() -> i32;
    pub fn rt1w_last_error() -> *const c_char;
    pub fn rt1w_context_create(device_id: i32, out: *mut *mut rt1w_context) -> i32;
    pub fn rt1w_context_destroy(ctx: *mut rt1w_context);
    // Multi-GPU (include/rt1w.h "Multi-GPU"): sample ranges sharded inside the library, one ncclReduce per render call.
    // (a) this process drives n devices: every later call on the context / its scenes is unchanged
    pub fn rt1w_context_create_multi(device_ids: *const i32, n: i32, out: *mut *mut rt1w_context) -> i32;
    // (b) one process per device: rank 0 makes the id, the host side ships it, every rank joins
    pub fn rt1w_comm_unique_id(out_id: *mut u8, capacity: usize) -> i32; // capacity >= RT1W_COMM_ID_BYTES
    pub fn rt1w_context_comm_init(ctx: *mut rt1w_context, id: *const u8, n_ranks: i32, rank: i32) -> i32;
    pub fn rt1w_context_get_comm(ctx: *const rt1w_context, rank: *mut i32, n_ranks: *mut i32, n_local_devices: *mut i32) -> i32;
    pub fn rt1w_shard_sample_range(rank: i32, n_ranks: i32, sample_begin: i32, sample_end: i32, out_begin: *mut i32, out_end: *mut i32);
    pub fn rt1w_scene_create(ctx: *mut rt1w_context, desc: *const rt1w_scene_desc, out: *mut *mut rt1w_scene) -> i32;
    pub fn rt1w_scene_destroy(scene: *mut rt1w_scene);
    pub fn rt1w_render(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        out_rgb_sum: *mut f32,
        out_stat: *mut f32,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    pub fn rt1w_render_rgb8(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        out_rgb8: *mut u8,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    pub fn rt1w_render_device(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        d_rgb_sum: *mut f32,
        cuda_stream: *mut c_void,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    // adaptive sampling (one device): params.sample_begin = 0, params.sample_end = the per-pixel cap; every output may be null
    pub fn rt1w_render_adaptive(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        min_spp: i32,
        max_error: f64,
        out_rgb_sum: *mut f32,
        out_spp: *mut i32,
        out_rgb8: *mut u8,
        out_stat: *mut f32,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    // batch rendering: n_frames cameras of one scene in one wavefront; seeds may be null (every frame params.seed); outputs
    // frame-major, either may be null but not both
    pub fn rt1w_render_batch(
        scene: *mut rt1w_scene,
        cameras: *const rt1w_camera,
        n_frames: i32,
        seeds: *const u64,
        params: *const rt1w_render_params,
        out_rgb_sum: *mut f32,
        out_rgb8: *mut u8,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    // light groups: the sums split by the emitter that ends each path, n_groups images group-major (rank 0 must pass
    // out_group_sum); they add up to rt1w_render's rgb_sum
    pub fn rt1w_render_light_groups(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        groups: *const rt1w_light_groups,
        out_group_sum: *mut f32,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    // first-hit feature buffers (albedo, normal, distance, hits) for denoisers and compositing: sums over the sample range
    pub fn rt1w_render_aov(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        out_albedo_sum: *mut f32,
        out_normal_sum: *mut f32,
        out_distance_sum: *mut f32,
        out_hits: *mut f32,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    // edge-aware denoising guided by the feature buffers: the filter alone on host sums of n_samples >= 2 samples, and the
    // render + feature buffers + filter in one call (rank 0 must pass out_rgb or out_rgb8)
    pub fn rt1w_denoise(
        ctx: *mut rt1w_context,
        width: i32,
        height: i32,
        n_samples: i32,
        rgb_sum: *const f32,
        stat: *const f32,
        albedo_sum: *const f32,
        normal_sum: *const f32,
        distance_sum: *const f32,
        hits: *const f32,
        dparams: *const rt1w_denoise_params,
        out_rgb: *mut f32,
        out_rgb8: *mut u8,
    ) -> i32;
    pub fn rt1w_render_denoised(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        dparams: *const rt1w_denoise_params,
        out_rgb: *mut f32,
        out_rgb8: *mut u8,
        out_rgb_sum: *mut f32,
        out_stat: *mut f32,
        stats: *mut rt1w_render_stats,
    ) -> i32;
    pub fn rt1w_resolve_rgb8(rgb_sum: *const f32, width: i32, height: i32, samples_per_pixel: i32, out_rgb8: *mut u8);

    // ---- scene introspection and the parity hooks (include/rt1w.h: test-only entry points) - what a `#[cfg(test)]` module of
    // the reference would hold `Hittable::hit`, `pdf_value`, `Texture::value`, `Perlin::noise/turb`, `refract` / `reflectance`
    // and `Material::scatter` against, value by value.  All buffers are host buffers.
    pub fn rt1w_scene_get_info(scene: *const rt1w_scene, out: *mut rt1w_scene_info) -> i32;
    pub fn rt1w_scene_get_prims(scene: *const rt1w_scene, out: *mut rt1w_flat_prim, capacity: i32, n_out: *mut i32) -> i32;
    pub fn rt1w_scene_get_leaf_prims(scene: *const rt1w_scene, prim_id_of_leaf: *mut i32, capacity: i32, n_out: *mut i32) -> i32;
    pub fn rt1w_lower_prims(desc: *const rt1w_scene_desc, out: *mut rt1w_flat_prim, capacity: i32, n_out: *mut i32) -> i32;
    pub fn rt1w_lower_face_groups(
        desc: *const rt1w_scene_desc,
        group_of_prim: *mut i32,
        face_of_prim: *mut i32,
        capacity: i32,
        n_groups: *mut i32,
    ) -> i32;
    pub fn rt1w_build_bvh_host(
        bbox_min3: *const f64,
        bbox_max3: *const f64,
        n: i32,
        nodes32: *mut c_void,
        node_capacity: i32,
        n_nodes: *mut i32,
        prim_order: *mut u32,
        wide_nodes80: *mut c_void,
        wide_capacity: i32,
        n_wide: *mut i32,
        wide_leaf_remap: *mut u32,
        depth: *mut i32,
        wide_depth: *mut i32,
    ) -> i32;
    // Test-only: the same outputs from the device LBVH builder of scene commit (lbvh.cu) on the context's device.
    pub fn rt1w_build_bvh_device(
        ctx: *mut rt1w_context,
        bbox_min3: *const f64,
        bbox_max3: *const f64,
        n: i32,
        nodes32: *mut c_void,
        node_capacity: i32,
        n_nodes: *mut i32,
        prim_order: *mut u32,
        wide_nodes80: *mut c_void,
        wide_capacity: i32,
        n_wide: *mut i32,
        wide_leaf_remap: *mut u32,
        depth: *mut i32,
        wide_depth: *mut i32,
    ) -> i32;
    pub fn rt1w_trace_closest(
        scene: *mut rt1w_scene,
        rays: *const rt1w_ray,
        n: usize,
        seed: u64,
        prim_id: *mut i32,
        t: *mut f32,
        normal3: *mut f32,
        front_face: *mut u8,
        uv2: *mut f32,
    ) -> i32;
    pub fn rt1w_eval_camera_rays(
        scene: *mut rt1w_scene,
        camera: *const rt1w_camera,
        params: *const rt1w_render_params,
        pixel_seed: *const u32,
        sample: *const i32,
        n: usize,
        out: *mut rt1w_ray,
    ) -> i32;
    pub fn rt1w_eval_light_pdf(scene: *mut rt1w_scene, light: i32, origin3: *const f64, dir3: *const f32, n: usize, pdf: *mut f32) -> i32;
    pub fn rt1w_eval_texture(scene: *mut rt1w_scene, texture: i32, p3: *const f64, uv2: *const f32, n: usize, rgb3: *mut f32) -> i32;
    pub fn rt1w_eval_perlin(scene: *mut rt1w_scene, table: i32, turb_depth: i32, p3: *const f64, n: usize, out: *mut f32) -> i32;
    pub fn rt1w_eval_dielectric(
        ctx: *mut rt1w_context,
        unit_dir3: *const f32,
        normal3: *const f32,
        ratio: *const f32,
        n: usize,
        reflect3: *mut f32,
        refract3: *mut f32,
        reflectance: *mut f32,
    ) -> i32;
    pub fn rt1w_eval_scatter(
        scene: *mut rt1w_scene,
        rays: *const rt1w_ray,
        n: usize,
        seed: u64,
        prim_id: *mut i32,
        material_type: *mut i32,
        dir3: *mut f32,
        weight3: *mut f32,
        time: *mut f32,
    ) -> i32;
    pub fn rt1w_philox4x32(counter: *const u32, key: *const u32, out: *mut u32);
}

/// The reference has no `Result` anywhere: it panics (bvh.rs:61,65-67; hittable.rs:153). Keep that behaviour.
pub fn check(status: i32) {
    if status != RT1W_OK {
        let msg = unsafe { std::ffi::CStr::from_ptr(rt1w_last_error()) }.to_string_lossy().into_owned();
        panic!("rt1w status {}: {}", status, msg);
    }
}
