//! Raw FFI mirror of `include/vanrijn_cuda.h` (ABI version 1).
//! UNCOMPILED SOURCE: there is no Rust toolchain in the build image; field order and widths follow the header,
//! whose layout is checked against the C compiler in tests/test_host_cpu.py.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub const VRJ_ABI_VERSION: u32 = 2;
pub const VRJ_OK: i32 = 0;
pub const VRJ_MAT_LAMBERTIAN: u32 = 0;
pub const VRJ_MAT_PHONG: u32 = 1;
pub const VRJ_MAT_REFLECTIVE: u32 = 2;
pub const VRJ_MAT_DIELECTRIC: u32 = 3;
pub const VRJ_INTEGRATOR_SIMPLE_RANDOM: u32 = 0;
pub const VRJ_INTEGRATOR_WHITTED: u32 = 1;
pub const VRJ_ITEM_SPHERE: u32 = 0;
pub const VRJ_ITEM_PLANE: u32 = 1;
pub const VRJ_ITEM_TRIANGLE: u32 = 2;
pub const VRJ_ITEM_BVH: u32 = 3;
pub const VRJ_FILTER_F32: u32 = 0;
pub const VRJ_FILTER_F64: u32 = 1;
pub const VRJ_FILTER_F32X4: u32 = 2;
pub const VRJ_FILTER_Q16: u32 = 3;
pub const VRJ_PRECISION_F64: u32 = 0;
pub const VRJ_PRECISION_F32_FAST: u32 = 1;
pub const VRJ_MEM_HOST: u32 = 0;
pub const VRJ_MEM_DEVICE: u32 = 1;
pub const VRJ_TONEMAP_XYZ: u32 = 0;
pub const VRJ_TONEMAP_LINEAR_RGB: u32 = 1;

#[repr(C)] pub struct VrjScene { _private: [u8; 0] }
#[repr(C)] pub struct VrjComm { _private: [u8; 0] }
#[repr(C)] pub struct VrjMultiScene { _private: [u8; 0] }

#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjSpectrum { pub shortest_wavelength: f64, pub longest_wavelength: f64, pub first_sample: u32, pub n_samples: u32 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjMaterial { pub kind: u32, pub spectrum: u32, pub p0: f64, pub p1: f64, pub p2: f64 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjSphere { pub centre: [f64; 3], pub radius: f64, pub material: u32, pub pad: u32 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjPlane { pub normal: [f64; 3], pub tangent: [f64; 3], pub cotangent: [f64; 3], pub distance_from_origin: f64, pub material: u32, pub pad: u32 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjBvh { pub first_node: u64, pub n_nodes: u64, pub first_triangle: u64, pub n_triangles: u64, pub depth: u32, pub pad: u32 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjItem { pub kind: u32, pub index: u32, pub object_id: u32, pub prim_id: u32 }

#[repr(C)]
pub struct VrjSceneDesc {
    pub abi_version: u32, pub pad0: u32,
    pub camera_location: [f64; 3], pub pad1: f64,
    pub n_spectra: u32, pub n_spectrum_samples: u32,
    pub spectra: *const VrjSpectrum, pub spectrum_samples: *const f64,
    pub n_materials: u32, pub n_spheres: u32,
    pub materials: *const VrjMaterial, pub spheres: *const VrjSphere,
    pub n_planes: u32, pub n_bvhs: u32,
    pub planes: *const VrjPlane, pub bvhs: *const VrjBvh,
    pub n_triangles: u64,
    pub tri_v0: *const f64, pub tri_v1: *const f64, pub tri_v2: *const f64,
    pub tri_n0: *const f64, pub tri_n1: *const f64, pub tri_n2: *const f64,
    pub tri_material: *const u32, pub tri_prim_id: *const u32,
    pub n_nodes: u64,
    pub node_min: *const f64, pub node_max: *const f64, pub node_child: *const i32,
    pub n_items: u32, pub pad2: u32,
    pub items: *const VrjItem,
}

#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjTile { pub start_column: u64, pub end_column: u64, pub start_row: u64, pub end_row: u64 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjSpectrumData { pub shortest_wavelength: f64, pub longest_wavelength: f64, pub n_samples: u32, pub pad: u32, pub samples: *const f64 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct VrjLight { pub direction: [f64; 3], pub spectrum: VrjSpectrumData }

#[repr(C)]
pub struct VrjRenderParams {
    pub spp: u32, pub max_depth: u32,
    pub sample_offset: u64, pub seed: u64,
    pub integrator: u32, pub bvh_filter: u32,
    pub bias: f64,
    pub lights: *const VrjLight, pub ambient_light: *const VrjSpectrumData,
    pub n_lights: u32, pub sample_stride: u32, pub count_traversal: u32, pub precision: u32,
}

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct VrjStats {
    pub primary_rays: u64, pub bounce_rays: u64, pub shadow_rays: u64,
    pub paths_missed: u64, pub paths_escaped: u64, pub paths_depth_limited: u64,
    pub node_visits: u64, pub triangle_tests: u64, pub kernel_launches: u64,
    pub device_ms: f64, pub primary_ms: f64, pub bounce_ms: f64, pub resolve_ms: f64,
    pub primary_launches: u64, pub bounce_launches: u64, pub resolve_launches: u64,
    pub shade_ms: f64, pub shade_launches: u64, pub staged_rays: u64,
    pub tail_ms: f64, pub tail_launches: u64,
    pub coalesced_calls: u64,
}

#[repr(C)]
pub struct VrjAccumOut {
    pub memory: u32, pub accumulate: u32,
    pub colour: *mut f64, pub colour_sum: *mut f64, pub colour_bias: *mut f64,
    pub weight: *mut f64, pub weight_bias: *mut f64,
    pub photons: *mut f64,
    pub stats: *mut VrjStats,
    pub srgb8: *mut u8,
}

/// Timing / shape of a device BVH build (`vrj_bvh_build`).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct VrjBvhBuildStats {
    pub device_ms: f64,
    pub global_levels: u32,
    pub radix_passes: u32,
    pub small_subtrees: u32,
    pub pad: u32,
}

/// Sample counts and error target of `vrj_render_adaptive` (see the header for the passes and the stopping rule).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct VrjAdaptiveParams {
    pub min_samples: u32,
    pub max_samples: u32,
    pub pass_samples: u32,
    pub pad: u32,
    pub rel_error: f64,
    pub abs_floor: f64,
}

/// What `vrj_render_adaptive` did: passes, samples over all pixels, pixels stopped by the rule / at `max_samples`.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct VrjAdaptiveStats {
    pub passes: u64,
    pub samples: u64,
    pub pixels_converged: u64,
    pub pixels_unconverged: u64,
}

/// Sample counts, pass limit and error target of `vrj_render_progressive` (the header states the schedule).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct VrjProgressiveParams {
    pub min_samples: u32,
    pub max_samples: u32,
    pub pass_samples: u32,
    pub max_passes: u32,
    pub rel_error: f64,
    pub abs_floor: f64,
}

impl Default for VrjProgressiveParams {
    /// A preview loop's: one pass of 4 samples per call, at most 64 per pixel, 5 % relative error of the mean Y
    fn default() -> Self {
        VrjProgressiveParams { min_samples: 4, max_samples: 64, pass_samples: 4, max_passes: 1, rel_error: 0.05, abs_floor: 0.0 }
    }
}

/// What `vrj_render_counts` rendered: samples (the sum of the map), pixels with a count above 0, wavefront batches.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct VrjCountsStats {
    pub samples: u64,
    pub pixels: u64,
    pub batches: u64,
}

/// What `vrj_plan_counts` planned: samples (the sum of the map) and the pixels planned / converged / at `max_samples`.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct VrjPlanStats {
    pub samples: u64,
    pub pixels_planned: u64,
    pub pixels_converged: u64,
    pub pixels_at_max: u64,
}

/// What `vrj_render_progressive` did (passes, samples) and the state it left: pixels converged / at `max_samples` / active.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct VrjProgressiveStats {
    pub passes: u64,
    pub samples: u64,
    pub pixels_converged: u64,
    pub pixels_at_max: u64,
    pub pixels_active: u64,
}

/// Outputs of `vrj_render_aux`: per-pixel first-hit features (see the header for the sums); any pointer may be NULL.
#[repr(C)]
pub struct VrjAuxOut {
    pub memory: u32,
    pub pad: u32,
    pub normal: *mut f64,
    pub depth: *mut f64,
    pub object_id: *mut i32,
    pub material: *mut i32,
    pub stats: *mut VrjStats,
}

/// Parameters of `vrj_denoise` (the header states the filter operation by operation).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct VrjDenoiseParams {
    pub iterations: u32,
    pub pad: u32,
    pub sigma_luminance: f64,
    pub sigma_normal: f64,
    pub sigma_depth: f64,
}

impl Default for VrjDenoiseParams {
    /// `VRJ_DENOISE_DEFAULT_*` of the header
    fn default() -> Self {
        VrjDenoiseParams { iterations: 4, pad: 0, sigma_luminance: 32.0, sigma_normal: 128.0, sigma_depth: 0.5 }
    }
}

extern "C" {
    pub fn vrj_last_error() -> *const c_char;
    pub fn vrj_abi_version() -> i32;
    pub fn vrj_device_count() -> i32;
    pub fn vrj_scene_create(desc: *const VrjSceneDesc, device: i32, out: *mut *mut VrjScene) -> i32;
    pub fn vrj_scene_destroy(scene: *mut VrjScene);
    pub fn vrj_scene_device_bytes(scene: *const VrjScene) -> u64;
    pub fn vrj_scene_upload_bytes(scene: *const VrjScene) -> u64;
    pub fn vrj_release_scratch();
    pub fn vrj_alloc_host(bytes: u64) -> *mut c_void;
    pub fn vrj_free_host(p: *mut c_void);
    pub fn vrj_alloc_device(device: i32, bytes: u64) -> *mut c_void;
    pub fn vrj_free_device(p: *mut c_void);
    pub fn vrj_copy_to_host(device: i32, host_dst: *mut c_void, device_src: *const c_void, bytes: u64) -> i32;
    pub fn vrj_render_tile(scene: *const VrjScene, tile: *const VrjTile, height: u64, width: u64,
                           params: *const VrjRenderParams, out: *mut VrjAccumOut) -> i32;
    /// Per-pixel sample counts from an on-device noise estimate; a pixel with n samples holds what
    /// `vrj_render_tile` with spp = n gives it.  `params.spp` must be 0; `y_sq_sum` may be NULL.
    pub fn vrj_render_adaptive(scene: *const VrjScene, tile: *const VrjTile, height: u64, width: u64,
                               params: *const VrjRenderParams, ap: *const VrjAdaptiveParams, out: *mut VrjAccumOut,
                               y_sq_sum: *mut f64, astats: *mut VrjAdaptiveStats) -> i32;
    /// Continues the state in `out` (colour_sum, colour_bias, weight, weight_bias) and `y_sq_sum`, all required, with
    /// the adaptive schedule for at most `pp.max_passes` passes; `params.spp` must be 0.
    pub fn vrj_render_progressive(scene: *const VrjScene, tile: *const VrjTile, height: u64, width: u64,
                                  params: *const VrjRenderParams, pp: *const VrjProgressiveParams, out: *mut VrjAccumOut,
                                  y_sq_sum: *mut f64, pstats: *mut VrjProgressiveStats) -> i32;
    /// Gives pixel p `counts[p]` new samples (its samples n .. n + counts[p] - 1, n = weight[p]) rendered in full
    /// wavefronts, from a zero state or (`out.accumulate`) the state in `out`; `y_sq_sum` may be null; `params.spp` must be 0.
    pub fn vrj_render_counts(scene: *const VrjScene, tile: *const VrjTile, height: u64, width: u64,
                             params: *const VrjRenderParams, counts: *const u32, out: *mut VrjAccumOut,
                             y_sq_sum: *mut f64, cstats: *mut VrjCountsStats) -> i32;
    /// The count map the header's rule gives each of `npix` pixels of a state (weight, colour_sum, y_sq_sum).
    pub fn vrj_plan_counts(device: i32, memory: u32, npix: u64, weight: *const f64, colour_sum: *const f64,
                           y_sq_sum: *const f64, rule: *const VrjAdaptiveParams, counts: *mut u32,
                           pstats: *mut VrjPlanStats) -> i32;
    /// First-hit normal, depth, object id and material of the camera rays a render with the same
    /// spp / seed / sample_offset / sample_stride traces.
    pub fn vrj_render_aux(scene: *const VrjScene, tile: *const VrjTile, height: u64, width: u64,
                          params: *const VrjRenderParams, out: *mut VrjAuxOut) -> i32;
    /// Variance-guided a-trous filter over one tile of `vrj_render_adaptive` + `vrj_render_aux` outputs.
    pub fn vrj_denoise(device: i32, memory: u32, tile_width: u64, tile_height: u64, colour_sum: *const f64,
                       weight: *const f64, y_sq_sum: *const f64, normal: *const f64, depth: *const f64,
                       material: *const i32, dp: *const VrjDenoiseParams, colour: *mut f64, srgb8: *mut u8,
                       device_ms: *mut f64) -> i32;
    pub fn vrj_comm_create(n_devices: i32, devices: *const i32, out: *mut *mut VrjComm) -> i32;
    pub fn vrj_comm_destroy(comm: *mut VrjComm);
    pub fn vrj_comm_scene_create(comm: *mut VrjComm, desc: *const VrjSceneDesc, out: *mut *mut VrjMultiScene) -> i32;
    pub fn vrj_comm_scene_destroy(scene: *mut VrjMultiScene);
    pub fn vrj_render_sharded(scene: *mut VrjMultiScene, tile: *const VrjTile, height: u64, width: u64,
                              params: *const VrjRenderParams, out: *mut VrjAccumOut) -> i32;
    pub fn vrj_tone_map(device: i32, memory: u32, source: u32, colour: *const f64, n_pixels: u64, rgb8: *mut u8) -> i32;
    /// `BoundingVolumeHierarchy::build` (src/raycasting/bounding_volume_hierarchy.rs:38-75) on the device: the same tree.
    pub fn vrj_bvh_build(device: i32, n_triangles: u64, vertices: *const f64, order: *mut u32, node_min: *mut f64,
                         node_max: *mut f64, node_child: *mut i32, depth: *mut u32, stats: *mut VrjBvhBuildStats) -> i32;
    pub fn vrj_trace_rays(scene: *const VrjScene, n: u64, origins: *const f64, directions: *const f64, bvh_filter: u32,
                          object_id: *mut i32, prim_id: *mut i32, t: *mut f64, stats: *mut VrjStats) -> i32;
}
