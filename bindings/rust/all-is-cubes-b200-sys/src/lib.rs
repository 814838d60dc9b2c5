//! `include/aicb200.h`, item for item.  ABI version 2 (`aicb_abi_version()`).
//! Layouts are checked against the C header by `tests/test_abi.py` on the Python mirror; keep the three in step.
#![allow(non_camel_case_types)]
#![no_std]

use core::ffi::{c_char, c_int, c_void};

pub type aicb_status = c_int;
pub const AICB_OK: aicb_status = 0;
pub const AICB_ERR_INVALID: aicb_status = 1;
pub const AICB_ERR_OOM: aicb_status = 2;
pub const AICB_ERR_CUDA: aicb_status = 3;
pub const AICB_ERR_UNSUPPORTED: aicb_status = 4;
pub const AICB_ERR_BUSY: aicb_status = 5;
pub const AICB_ERR_RETRY: aicb_status = 6;

pub const AICB_TEXT_ENTERED_SPACE: i32 = -1;
pub const AICB_TEXT_EMPTY: i32 = -2;
pub const AICB_TEXT_INCOMPLETE: i32 = -3;

/// `GridAab` (all-is-cubes-base/src/math/grid_aab.rs)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_aab {
    pub lower: [i32; 3],
    pub size: [u32; 3],
}

/// colour part of `Evoxel` (block/eval/voxel_storage.rs:41-53)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_voxel {
    pub rgba: [f32; 4],
    pub emission: [f32; 3],
    pub _pad: f32,
}

/// one entry of `Space::block_data()` as `TracingBlock::from_block` sees it (sr.rs:569-587) plus the
/// `EvaluatedBlock` members light propagation reads (block/eval/evaluated.rs:189-267)
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct aicb_block_desc {
    pub resolution: u8,
    pub is_air: u8,
    pub light_opaque_faces: u8,
    pub light_visible: u8,
    pub voxel_bounds: aicb_aab,
    pub indices: *const u16,
    pub n_indices: usize,
    pub palette: *const aicb_voxel,
    pub n_palette: usize,
    pub light_face_colors: [[f32; 4]; 6],
    pub light_color: [f32; 4],
    pub light_emission: [f32; 3],
    pub _pad: f32,
}

/// `Sky` (space/sky.rs:16-21): kind 0 = Uniform(colors[0]), 1 = Octants
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_sky {
    pub kind: u32,
    pub colors: [[f32; 3]; 8],
}

/// what `SpaceRaytracer::new` snapshots (sr.rs:64-88)
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct aicb_scene_desc {
    pub bounds: aicb_aab,
    pub block_ids: *const u16,
    pub light: *const [u8; 4],
    pub blocks: *const aicb_block_desc,
    pub n_blocks: usize,
    pub sky: aicb_sky,
    pub light_max_distance: u8,
    pub _pad: [u8; 7],
}

/// what `Camera::project_ndc_into_world` needs (camera_struct.rs:238-257)
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct aicb_camera {
    pub inverse_projection_view: [f64; 16],
    pub fb_width: u32,
    pub fb_height: u32,
    pub exposure: f32,
    pub _pad: u32,
}

/// the `GraphicsOptions` fields that affect pixels (graphics_options.rs:28-150)
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct aicb_options {
    pub fog: u8,
    pub lighting_display: u8,
    pub transparency: u8,
    pub antialiasing_always: u8,
    pub tone_mapping: u8,
    pub debug_pixel_cost: u8,
    pub include_sky: u8,
    pub bounce_samples: u8,
    pub transparency_threshold: f32,
    pub maximum_intensity: f32,
    pub view_distance: f64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_shard {
    pub strip_rows: u32,
    pub index: u32,
    pub count: u32,
}

/// `ImageInfo` / `RaytraceInfo` (renderer.rs:609-646, sr.rs:520-522) plus device timing
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_render_info {
    pub cubes_traced: u64,
    pub rays: u64,
    pub algorithmic_bytes: u64,
    pub counters: [u64; 6],
    pub kernel_ms: f32,
    pub flaws: u16,
    pub _pad: u16,
    pub stage_ms: [f32; 4],
}

/// `Position` of the first hit (hit.rs:92-101)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_hit {
    pub cube: [i32; 3],
    pub voxel: [i32; 3],
    pub resolution: i32,
    pub face: i32,
}

/// `LightUpdatesInfo` (updater.rs:970-984) of one `aicb_light_step`, plus counters
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct aicb_light_updates {
    pub update_count: u64,
    pub queue_count: u64,
    pub chart_node_visits: u64,
    pub rounds: u32,
    pub max_update_difference: u8,
    pub max_queue_priority: u8,
    pub _pad: [u8; 2],
    pub device_ms: f32,
}

#[repr(C)]
pub struct aicb_ctx {
    _opaque: [u8; 0],
}
#[repr(C)]
pub struct aicb_scene {
    _opaque: [u8; 0],
}
#[repr(C)]
pub struct aicb_group {
    _opaque: [u8; 0],
}
#[repr(C)]
pub struct aicb_group_scene {
    _opaque: [u8; 0],
}

/// one layer of `RtScene::trace_ray_through_layers` (renderer.rs:454-478)
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct aicb_layer {
    pub scene: *mut aicb_scene,
    pub camera: *const aicb_camera,
    pub options: *const aicb_options,
}

unsafe extern "C" {
    pub fn aicb_abi_version() -> u32;
    pub fn aicb_ctx_create(device_id: c_int, out: *mut *mut aicb_ctx) -> aicb_status;
    pub fn aicb_ctx_destroy(ctx: *mut aicb_ctx);
    pub fn aicb_last_error() -> *const c_char;

    pub fn aicb_scene_create(ctx: *mut aicb_ctx, desc: *const aicb_scene_desc, out: *mut *mut aicb_scene) -> aicb_status;
    pub fn aicb_scene_update_cubes(s: *mut aicb_scene, cubes: *const [i32; 3], block_ids: *const u16, light: *const [u8; 4], n: usize) -> aicb_status;
    pub fn aicb_scene_update_blocks(s: *mut aicb_scene, indices: *const u16, descs: *const aicb_block_desc, n: usize) -> aicb_status;
    pub fn aicb_scene_upload_light(s: *mut aicb_scene, light: *const [u8; 4], n_texels: usize) -> aicb_status;
    pub fn aicb_scene_destroy(s: *mut aicb_scene);
    pub fn aicb_scene_device_bytes(s: *const aicb_scene) -> u64;

    pub fn aicb_shard_pixel_count(cam: *const aicb_camera, shard: *const aicb_shard) -> usize;
    pub fn aicb_render_srgb8(s: *mut aicb_scene, cam: *const aicb_camera, opt: *const aicb_options, shard: *const aicb_shard,
                             out: *mut [u8; 4], out_len: usize, info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_render_rgba16f(s: *mut aicb_scene, cam: *const aicb_camera, opt: *const aicb_options, shard: *const aicb_shard,
                               out: *mut [u16; 4], out_len: usize, info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_render_colorbuf(s: *mut aicb_scene, cam: *const aicb_camera, opt: *const aicb_options, shard: *const aicb_shard,
                                out_colorbuf: *mut [f32; 4], depth: *mut f64, hit: *mut aicb_hit, steps: *mut u32,
                                out_len: usize, info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_render_text(s: *mut aicb_scene, cam: *const aicb_camera, opt: *const aicb_options, out: *mut i32, out_len: usize,
                            info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_render_layers_srgb8(world: *const aicb_layer, ui: *const aicb_layer, backdrop_rgba: *const [f32; 4],
                                    no_world_rgba: *const [f32; 4], out: *mut [u8; 4], out_len: usize,
                                    info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_ortho_image_size(s: *const aicb_scene, resolution: u32, width: *mut u32, height: *mut u32) -> aicb_status;
    pub fn aicb_render_orthographic(s: *mut aicb_scene, resolution: u32, out: *mut [u8; 4], out_len: usize,
                                    info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_render_srgb8_device(s: *mut aicb_scene, cam: *const aicb_camera, opt: *const aicb_options, shard: *const aicb_shard,
                                    d_out: *mut c_void, out_len: usize, stream: *mut c_void) -> aicb_status;
    pub fn aicb_render_srgb8_device_frame(s: *mut aicb_scene, cam: *const aicb_camera, opt: *const aicb_options,
                                          shard: *const aicb_shard, d_frame: *mut c_void, frame_len: usize,
                                          stream: *mut c_void) -> aicb_status;
    pub fn aicb_render_finish(s: *mut aicb_scene, info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_frame_create(ctx: *mut aicb_ctx, n_pixels: usize, d_frame: *mut *mut c_void, handle_out: *mut [u8; 64]) -> aicb_status;
    pub fn aicb_frame_open(ctx: *mut aicb_ctx, handle: *const [u8; 64], d_frame: *mut *mut c_void) -> aicb_status;
    pub fn aicb_frame_close(ctx: *mut aicb_ctx, d_frame: *mut c_void, opened: c_int) -> aicb_status;
    pub fn aicb_frame_read(ctx: *mut aicb_ctx, d_frame: *const c_void, out: *mut [u8; 4], n_pixels: usize, stream: *mut c_void) -> aicb_status;
    // delivery without a collective: two monotonic counters behind the frame's pixels (include/aicb200.h)
    pub fn aicb_frame_signal(ctx: *mut aicb_ctx, d_frame: *mut c_void, n_pixels: usize, stream: *mut c_void) -> aicb_status;
    pub fn aicb_frame_wait_arrived(ctx: *mut aicb_ctx, d_frame: *mut c_void, n_pixels: usize, count: u32, stream: *mut c_void) -> aicb_status;
    pub fn aicb_frame_release(ctx: *mut aicb_ctx, d_frame: *mut c_void, n_pixels: usize, frame_id: u32, stream: *mut c_void) -> aicb_status;
    pub fn aicb_frame_wait_consumed(ctx: *mut aicb_ctx, d_frame: *mut c_void, n_pixels: usize, frame_id: u32, stream: *mut c_void) -> aicb_status;
    pub fn aicb_frame_timed_out(ctx: *mut aicb_ctx, d_frame: *mut c_void, n_pixels: usize, out: *mut u32) -> aicb_status;
    pub fn aicb_ctx_stage_timing(ctx: *mut aicb_ctx, enable: c_int) -> aicb_status;

    pub fn aicb_group_create(device_ids: *const c_int, n_devices: c_int, out: *mut *mut aicb_group) -> aicb_status;
    pub fn aicb_group_destroy(g: *mut aicb_group);
    pub fn aicb_group_size(g: *const aicb_group) -> c_int;
    pub fn aicb_group_scene_create(g: *mut aicb_group, desc: *const aicb_scene_desc, out: *mut *mut aicb_group_scene) -> aicb_status;
    pub fn aicb_group_scene_destroy(gs: *mut aicb_group_scene);
    pub fn aicb_group_scene_update_cubes(gs: *mut aicb_group_scene, cubes: *const [i32; 3], block_ids: *const u16,
                                         light: *const [u8; 4], n: usize) -> aicb_status;
    pub fn aicb_group_render_srgb8(gs: *mut aicb_group_scene, cam: *const aicb_camera, opt: *const aicb_options,
                                   out: *mut [u8; 4], out_len: usize, info: *mut aicb_render_info) -> aicb_status;
    pub fn aicb_group_scene_update_blocks(gs: *mut aicb_group_scene, indices: *const u16, descs: *const aicb_block_desc,
                                          n: usize) -> aicb_status;
    pub fn aicb_group_scene_upload_light(gs: *mut aicb_group_scene, light: *const [u8; 4], n_texels: usize) -> aicb_status;
    pub fn aicb_group_light_fast_evaluate(gs: *mut aicb_group_scene) -> aicb_status;
    pub fn aicb_group_light_evaluate(gs: *mut aicb_group_scene, epsilon: u8, updates_done: *mut u64, max_diff: *mut u8,
                                     chart_node_visits: *mut u64) -> aicb_status;
    pub fn aicb_group_light_edit_and_propagate(gs: *mut aicb_group_scene, cubes: *const [i32; 3], new_ids: *const u16,
                                               n_edits: usize, epsilon: u8, updates_done: *mut u64,
                                               max_diff: *mut u8) -> aicb_status;
    /// `member` is a position in the group (0..size-1), not a device id.
    pub fn aicb_group_light_download(gs: *mut aicb_group_scene, member: c_int, out: *mut [u8; 4], n_texels: usize) -> aicb_status;
    /// `member` -1: the group's totals; else that member's own counters.
    pub fn aicb_group_light_stats(gs: *const aicb_group_scene, member: c_int, out: *mut [u64; 4]) -> aicb_status;
    /// `max_updates` u64::MAX / `budget_us` < 0: no limit; `out` may be null.
    pub fn aicb_light_step(s: *mut aicb_scene, cubes: *const [i32; 3], new_ids: *const u16, n_edits: usize, epsilon: u8,
                           max_updates: u64, budget_us: f64, out: *mut aicb_light_updates) -> aicb_status;
    pub fn aicb_group_light_step(gs: *mut aicb_group_scene, cubes: *const [i32; 3], new_ids: *const u16, n_edits: usize,
                                 epsilon: u8, max_updates: u64, budget_us: f64, out: *mut aicb_light_updates) -> aicb_status;
    pub fn aicb_light_track_changes(s: *mut aicb_scene, enable: c_int) -> aicb_status;
    /// Writes and consumes nothing when `*n_changed` (always the count) exceeds `cap`.
    pub fn aicb_light_take_changes(s: *mut aicb_scene, cubes: *mut [i32; 3], texels: *mut [u8; 4], cap: usize,
                                   n_changed: *mut usize) -> aicb_status;
    pub fn aicb_group_light_track_changes(gs: *mut aicb_group_scene, enable: c_int) -> aicb_status;
    pub fn aicb_group_light_take_changes(gs: *mut aicb_group_scene, cubes: *mut [i32; 3], texels: *mut [u8; 4], cap: usize,
                                         n_changed: *mut usize) -> aicb_status;

    pub fn aicb_trace_rays(s: *mut aicb_scene, origin_dir: *const [f64; 6], n: usize, opt: *const aicb_options,
                           out_colorbuf: *mut [f32; 4], depth: *mut f64, hit: *mut aicb_hit, steps: *mut u32,
                           info: *mut aicb_render_info) -> aicb_status;

    pub fn aicb_camera_look_at(eye: *const [f64; 3], target: *const [f64; 3], fov_y_degrees: f64, view_distance: f64,
                               nominal_width: f64, nominal_height: f64, fb_width: u32, fb_height: u32, exposure: f32,
                               out: *mut aicb_camera) -> aicb_status;
    pub fn aicb_camera_from_view(rotation_ijkr: *const [f64; 4], translation: *const [f64; 3], fov_y_degrees: f64,
                                 view_distance: f64, nominal_width: f64, nominal_height: f64, fb_width: u32,
                                 fb_height: u32, exposure: f32, out: *mut aicb_camera) -> aicb_status;
    pub fn aicb_eye_for_look_at(bounds: *const aicb_aab, direction: *const [f64; 3], out_eye: *mut [f64; 3]);
    pub fn aicb_camera_project_ndc(cam: *const aicb_camera, ndc_x: f64, ndc_y: f64, out_origin_dir: *mut [f64; 6]);

    pub fn aicb_light_chart(weights: *mut f32, children: *mut u32) -> u32;
    pub fn aicb_light_chart_chains(preorder: *mut u32, chains: *mut [u32; 6], euler: *mut u16) -> u32;
    pub fn aicb_light_fast_evaluate(s: *mut aicb_scene) -> aicb_status;
    pub fn aicb_light_compute(s: *mut aicb_scene, cubes: *const [i32; 3], n: usize, out: *mut [u8; 4]) -> aicb_status;
    pub fn aicb_light_evaluate(s: *mut aicb_scene, epsilon: u8, updates_done: *mut u64, max_diff: *mut u8,
                               chart_node_visits: *mut u64) -> aicb_status;
    pub fn aicb_light_edit_and_propagate(s: *mut aicb_scene, cubes: *const [i32; 3], new_ids: *const u16, n_edits: usize,
                                         epsilon: u8, updates_done: *mut u64, max_diff: *mut u8) -> aicb_status;
    pub fn aicb_light_download(s: *mut aicb_scene, out: *mut [u8; 4], n_texels: usize) -> aicb_status;
    pub fn aicb_light_stats(s: *const aicb_scene, out: *mut [u64; 4]) -> aicb_status;
}
