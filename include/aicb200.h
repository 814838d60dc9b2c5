/*
 * aicb200.h — C ABI of libaicb200.so: the B200-native (sm_100a) replacement for the
 * per-pixel voxel raytracer of kpreid/all-is-cubes, behind the reference's own
 * HeadlessRenderer / Camera / SpaceRaytracer surface.
 *
 * Every entry point cites the reference interface it replaces (paths relative to the
 * reference checkout, commit 7ab02ee1).  All structs are plain data; all pointers in are
 * borrowed for the duration of the call only; all pointers out are caller-allocated with
 * explicit lengths.  Nothing throws or aborts across this boundary: errors are status codes
 * plus aicb_last_error().
 *
 * There is NO CPU fallback.  Every compute entry point fails with AICB_ERR_CUDA when no
 * sm_100-class device is available.
 */
#ifndef AICB200_H
#define AICB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AICB_ABI_VERSION 2

typedef enum aicb_status {
    AICB_OK = 0,
    AICB_ERR_INVALID = 1,     /* bad argument / length mismatch (the reference panics: renderer.rs:193-197) */
    AICB_ERR_OOM = 2,         /* cudaMalloc failed  -> Flaws::OUT_OF_MEMORY (flaws.rs) */
    AICB_ERR_CUDA = 3,        /* no device, launch failure, lost GPU (lib.rs:53 "TODO: lost GPU") */
    AICB_ERR_UNSUPPORTED = 4, /* an option value this build does not implement */
    AICB_ERR_BUSY = 5,        /* aicb_render_finish for a scene whose frame is not the context's last one */
    AICB_ERR_RETRY = 6        /* asynchronous render only: the frame's hit stream overflowed its device buffer; the
                                 buffer has been enlarged, issue the same render again (the synchronous entry points
                                 retry internally) */
} aicb_status;

/* ---------------------------------------------------------------------------------------------
 * Plain-data mirrors of reference types
 * ------------------------------------------------------------------------------------------- */

/* GridAab (all-is-cubes-base/src/math/grid_aab.rs): lower corner + size. */
typedef struct aicb_aab {
    int32_t lower[3];
    uint32_t size[3];
} aicb_aab;

/* Colour part of Evoxel (all-is-cubes/src/block/eval/voxel_storage.rs:41-53):
 * non-premultiplied linear RGBA reflectance + RGB emission. 32 bytes. */
typedef struct aicb_voxel {
    float rgba[4];
    float emission[3];
    float _pad;
} aicb_voxel;

/* Face7 (all-is-cubes-base/src/math/face.rs:105). */
enum { AICB_FACE_WITHIN = 0, AICB_FACE_NX = 1, AICB_FACE_NY = 2, AICB_FACE_NZ = 3,
       AICB_FACE_PX = 4, AICB_FACE_PY = 5, AICB_FACE_PZ = 6 };

/* One entry of Space::block_data() as the raytracer sees it: TracingBlock (sr.rs:569-587)
 * = Evoxels (voxel_storage.rs:190-209).  `indices == NULL` means Evoxels::One(palette[0]).
 * Otherwise `indices` holds one u16 palette index per voxel of `voxel_bounds`, Z-major
 * (vol.rs:1013-1018: ((x-lx)*size_y + (y-ly))*size_z + (z-lz)); voxel_bounds may be smaller
 * than resolution^3 (voxel_storage.rs:176-178) but must lie inside [0,resolution)^3.
 * `is_air` is TracingCubeData::always_invisible (sr.rs:547).
 * The `light_*` members are EvaluatedBlock derived data (block/eval/derived.rs:33-80) read
 * only by the light-propagation path (space/light/updater.rs:760-884). */
typedef struct aicb_block_desc {
    uint8_t resolution;            /* 1,2,4,...,128 (resolution.rs:18-27) */
    uint8_t is_air;
    uint8_t light_opaque_faces;    /* bit (face-1) set if EvaluatedBlock::opaque()[face], NX..PZ */
    uint8_t light_visible;         /* EvaluatedBlock::visible_or_animated() */
    aicb_aab voxel_bounds;
    const uint16_t *indices;       /* NULL => single voxel */
    size_t n_indices;
    const aicb_voxel *palette;
    size_t n_palette;
    float light_face_colors[6][4]; /* EvaluatedBlock::face7_color(face), NX..PZ */
    float light_color[4];          /* EvaluatedBlock::color() */
    float light_emission[3];       /* EvaluatedBlock::light_emission() */
    float _pad;
} aicb_block_desc;

/* Sky (all-is-cubes/src/space/sky.rs:16-21). kind 0 = Uniform(colors[0]), 1 = Octants.
 * Octant index = (x>=0)<<2 | (y>=0)<<1 | (z>=0)  (sky.rs:36-39). */
typedef struct aicb_sky {
    uint32_t kind;
    float colors[8][3];
} aicb_sky;

/* What SpaceRaytracer::new (sr.rs:64-88) snapshots from space::Read:
 * bounds, per-cube block index (Space::contents, Z-major), per-cube PackedLight texels
 * (light/data.rs:162 as_texel: r,g,b,status; NULL => LightPhysics::None => PackedLight::ONE,
 * space.rs:1241-1246), the block table and the sky. */
typedef struct aicb_scene_desc {
    aicb_aab bounds;
    const uint16_t *block_ids;     /* volume entries */
    const uint8_t (*light)[4];     /* volume texels or NULL */
    const aicb_block_desc *blocks;
    size_t n_blocks;
    aicb_sky sky;
    uint8_t light_max_distance;    /* LightPhysics::Rays{maximum_distance} (space/physics.rs:94-104); 0 = None */
    uint8_t _pad[7];
} aicb_scene_desc;

/* Camera as the raytracer consumes it: Camera::project_ndc_into_world (camera_struct.rs:238-257)
 * needs only inverse_projection_view (euclid Transform3D, row-vector convention, m11..m44 in
 * row-major order), the framebuffer size (viewport.rs:104-113) and exposure
 * (camera_struct.rs:376-382).  aicb_camera_look_at()/aicb_camera_from_view() below build it
 * exactly as Camera::compute_matrices (camera_struct.rs:387-416) does. */
typedef struct aicb_camera {
    double inverse_projection_view[16];
    uint32_t fb_width, fb_height;
    float exposure;
    uint32_t _pad;
} aicb_camera;

enum { AICB_FOG_NONE = 0, AICB_FOG_ABRUPT = 1, AICB_FOG_COMPROMISE = 2, AICB_FOG_PHYSICAL = 3 };
enum { AICB_LIGHT_NONE = 0, AICB_LIGHT_FLAT = 1, AICB_LIGHT_COARSE = 2, AICB_LIGHT_LINEAR = 3,
       AICB_LIGHT_SMOOTHSTEP = 4, AICB_LIGHT_BOUNCE = 5 /* secondary Lambertian rays (surface.rs:113-166); needs aicb_options::bounce_samples */ };
enum { AICB_TRANSPARENCY_SURFACE = 0, AICB_TRANSPARENCY_VOLUMETRIC = 1, AICB_TRANSPARENCY_THRESHOLD = 2 };
enum { AICB_TONE_CLAMP = 0, AICB_TONE_REINHARD = 1 };

/* The GraphicsOptions fields that affect pixels (graphics_options.rs:28-150). */
typedef struct aicb_options {
    uint8_t fog;
    uint8_t lighting_display;
    uint8_t transparency;
    uint8_t antialiasing_always;   /* AntialiasingOption::Always => 4 fixed sub-samples (renderer.rs:426-444) */
    uint8_t tone_mapping;
    uint8_t debug_pixel_cost;
    uint8_t include_sky;           /* trace_ray's include_sky argument (sr.rs:113-120); renders use 1 */
    uint8_t bounce_samples;        /* LightingOption::Bounce { samples } (graphics_options.rs:464-467); >= 1 with Bounce */
    float transparency_threshold;  /* TransparencyOption::Threshold(t) */
    float maximum_intensity;       /* +inf disables tone mapping (graphics_options.rs:352-357) */
    double view_distance;          /* repaired to [1, 10000] by the caller (graphics_options.rs:194-198) */
} aicb_options;

/* Row-strip sharding of one frame across ranks (SURVEY §8(e)): rows are cut into strips of
 * `strip_rows`; strip s belongs to shard (s % count).  count = 1 renders everything. */
typedef struct aicb_shard {
    uint32_t strip_rows;
    uint32_t index;
    uint32_t count;
} aicb_shard;

/* ImageInfo / RaytraceInfo (renderer.rs:609-646, sr.rs:520-522) plus device timing. */
typedef struct aicb_render_info {
    uint64_t cubes_traced;         /* RaytraceInfo::cubes_traced, summed over all rays */
    uint64_t rays;                 /* primary rays traced (pixels * samples) */
    uint64_t algorithmic_bytes;    /* SURVEY §8(d) formula, from device counters */
    uint64_t counters[6];          /* outer steps, inner steps, surface hits, light texels, blocks entered, pixels */
    float kernel_ms;               /* CUDA-event duration of the whole frame (all kernels) on its stream */
    uint16_t flaws;                /* Flaws bits (flaws.rs:20-91) */
    uint16_t _pad;
    float stage_ms[4];             /* the frame's kernels (first chunk): ray generation, marching, shading, encode */
} aicb_render_info;

/* CharacterBuf states (raytracer/text.rs:52-123) of aicb_render_text: a value >= 0 is the block index (Space palette
 * index) of the first block hit; the caller maps it to that block's string like TracingBlock's D::from_block does. */
#define AICB_TEXT_ENTERED_SPACE (-1) /* the ray entered the Space's bounds but hit nothing: " " */
#define AICB_TEXT_EMPTY (-2)         /* the ray never entered the Space: "." */
#define AICB_TEXT_INCOMPLETE (-3)    /* Exception::Incomplete (step cap) before any hit: "X" */

/* Per-pixel hit record: Position of the first non-exception Hit (hit.rs:92-101):
 * cube xyz, voxel xyz, resolution, face; all -1 when the ray hit nothing. */
typedef struct aicb_hit {
    int32_t cube[3];
    int32_t voxel[3];
    int32_t resolution;
    int32_t face;
} aicb_hit;

typedef struct aicb_ctx aicb_ctx;     /* one CUDA device + stream */
typedef struct aicb_scene aicb_scene; /* device-resident flattened Space */

/* ---------------------------------------------------------------------------------------------
 * Context
 * ------------------------------------------------------------------------------------------- */
uint32_t aicb_abi_version(void);
/* device_id < 0 selects the current device. Fails with AICB_ERR_CUDA if there is no GPU. */
aicb_status aicb_ctx_create(int device_id, aicb_ctx **out);
void aicb_ctx_destroy(aicb_ctx *);
/* aicb_render_info::stage_ms needs five event records per frame; on by default, off for callers that only want frames. */
aicb_status aicb_ctx_stage_timing(aicb_ctx *, int enable);
/* Thread-local message for the last failing call on this thread. Never NULL. */
const char *aicb_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * update(): replaces SpaceRaytracer::new / UpdatingSpaceRaytracer::update
 * (sr.rs:64-88, updating.rs:107-172). The library copies everything before returning.
 * ------------------------------------------------------------------------------------------- */
aicb_status aicb_scene_create(aicb_ctx *, const aicb_scene_desc *, aicb_scene **out);
/* SpaceChange::CubeBlock / CubeLight (space.rs:1062-1100): light may be NULL to leave light alone. */
aicb_status aicb_scene_update_cubes(aicb_scene *, const int32_t (*cubes)[3], const uint16_t *block_ids,
                                    const uint8_t (*light)[4], size_t n);
/* SpaceChange::BlockEvaluation / BlockIndex (space.rs:1062-1100; updating.rs:128-150): new definitions for EXISTING
 * block indices (an index beyond the table needs a new scene).  Voxel data is appended to the device pools; cubes
 * holding a block whose classification (invisible / single voxel / voxel brick) changed are re-encoded.  Light is not
 * re-propagated (call aicb_light_evaluate).  GPU test: tests/test_gpu_parity.py::test_block_definition_update_equals_fresh_snapshot. */
aicb_status aicb_scene_update_blocks(aicb_scene *, const uint16_t *indices, const aicb_block_desc *descs, size_t n);
/* Whole light volume replaced (after light propagation on the host or on another rank). */
aicb_status aicb_scene_upload_light(aicb_scene *, const uint8_t (*light)[4], size_t n_texels);
void aicb_scene_destroy(aicb_scene *);
uint64_t aicb_scene_device_bytes(const aicb_scene *);

/* ---------------------------------------------------------------------------------------------
 * draw(): replaces RtRenderer::draw_rgba / RtRenderer::draw::<ColorBuf> and the Rayon pixel
 * dispatch trace_scene_to_image_impl (renderer.rs:183-220, 282-308, 516-556).
 * Host-buffer variants copy device->host inside the call (blocking, like draw_rgba).
 * `out_len` must equal aicb_shard_pixel_count(camera, shard) or AICB_ERR_INVALID is returned.
 * Pixels of the shard's rows are packed in increasing row order, row-major, top-left origin.
 * ------------------------------------------------------------------------------------------- */
size_t aicb_shard_pixel_count(const aicb_camera *, const aicb_shard *shard_or_null);

/* == draw_rgba: sRGB8 RGBA, post_process_color + to_srgb8 applied (renderer.rs:287-291). */
aicb_status aicb_render_srgb8(aicb_scene *, const aicb_camera *, const aicb_options *,
                              const aicb_shard *shard_or_null,
                              uint8_t (*out)[4], size_t out_len, aicb_render_info *info_or_null);

/* == the per-pixel colour of raytrace_to_texture (all-is-cubes-gpu/src/raytrace_to_texture.rs:645-661):
 * ColorBuf::into_premultiplied_rgba (all-is-cubes/src/raytracer_components.rs:70-77) with the camera's exposure
 * applied to r, g, b, rounded to IEEE binary16 like half::f16::from_f32; not tone-mapped (the caller's GPU
 * postprocessing does that).  out[i] = {r, g, b, a} as raw f16 bits. */
aicb_status aicb_render_rgba16f(aicb_scene *, const aicb_camera *, const aicb_options *,
                                const aicb_shard *shard_or_null,
                                uint16_t (*out)[4], size_t out_len, aicb_render_info *info_or_null);

/* == draw::<ColorBuf> (+ DepthBuf, + Position): raw accumulators for parity and other callers.
 * out_colorbuf: light.xyz, transmittance (raytracer_components.rs:20-39).
 * depth_or_null: DepthBuf::depth (accum.rs:254-311) of the first Hit carrying a t_distance.
 * hit_or_null: Position of the first surface hit. */
aicb_status aicb_render_colorbuf(aicb_scene *, const aicb_camera *, const aicb_options *,
                                 const aicb_shard *shard_or_null,
                                 float (*out_colorbuf)[4], double *depth_or_null, aicb_hit *hit_or_null,
                                 uint32_t *steps_or_null, size_t out_len, aicb_render_info *info_or_null);

/* == print_space's image (raytracer/text.rs:139-180): per pixel the CharacterBuf state (text.rs:52-123) — the block
 * index of the first block the ray hit, or one of AICB_TEXT_*.  The caller prints each value with the string its block
 * data gives that block (D::from_block). */
aicb_status aicb_render_text(aicb_scene *, const aicb_camera *, const aicb_options *, int32_t *out, size_t out_len,
                             aicb_render_info *info_or_null);

/* == RtScene::trace_ray_through_layers + draw_rgba (renderer.rs:454-478, 282-308): the UI layer (its own Space and
 * camera, traced without sky), the backdrop colour (StandardCameras' UiViewState::backdrop; NULL or transparent = none),
 * then the world layer continuing in the same accumulator; a pixel that is still not opaque (no world layer) is
 * painted `no_world_rgba` (palette::NO_WORLD_TO_SHOW, linear RGBA; NULL = leave).  Either layer may be NULL.  Both
 * scenes must belong to one context and both cameras to one framebuffer size; the world layer's options choose the
 * antialiasing sample points and the post-processing.  The info text of draw(info_text) is drawn by the caller over
 * the returned image (renderer.rs:659-683 needs the font of the universe). */
typedef struct aicb_layer {
    aicb_scene *scene;
    const aicb_camera *camera;
    const aicb_options *options;
} aicb_layer;
aicb_status aicb_render_layers_srgb8(const aicb_layer *world_or_null, const aicb_layer *ui_or_null,
                                     const float backdrop_rgba[4], const float no_world_rgba[4],
                                     uint8_t (*out)[4], size_t out_len, aicb_render_info *info_or_null);

/* == render_orthographic (raytracer/ortho.rs:30-84): the five axis-aligned views of MultiOrthoCamera (:143-199) in one
 * image at `resolution` pixels per cube (the reference uses 32), UNALTERED_COLORS, sRGB8 without post-processing,
 * transparent between the views.  aicb_ortho_image_size gives the image size for a scene. */
aicb_status aicb_ortho_image_size(const aicb_scene *, uint32_t resolution, uint32_t *width, uint32_t *height);
aicb_status aicb_render_orthographic(aicb_scene *, uint32_t resolution, uint8_t (*out)[4], size_t out_len,
                                     aicb_render_info *info_or_null);

/* Device-resident output (for multi-GPU gather and kernel-only timing): `d_out` is a device
 * pointer on the ctx's device with room for out_len pixels; `stream` is a cudaStream_t (0 =
 * the ctx stream). Does not synchronise; info (if given) is filled by
 * aicb_render_finish(). */
aicb_status aicb_render_srgb8_device(aicb_scene *, const aicb_camera *, const aicb_options *,
                                     const aicb_shard *shard_or_null,
                                     void *d_out, size_t out_len, void *stream);
/* As above, but `d_frame` is a FULL framebuffer (fb_width*fb_height pixels) and the shard's pixels
 * are stored at their framebuffer positions.  `d_frame` may be peer memory of another GPU mapped
 * into this process (cudaIpcOpenMemHandle / P2P): the trace kernel's epilogue then delivers its
 * row strips straight into the root GPU's frame over NVLink, replacing the gather collective. */
aicb_status aicb_render_srgb8_device_frame(aicb_scene *, const aicb_camera *, const aicb_options *,
                                           const aicb_shard *shard_or_null,
                                           void *d_frame, size_t frame_len, void *stream);
aicb_status aicb_render_finish(aicb_scene *, aicb_render_info *info_or_null);

/* Full-frame buffers shared between the ranks of one node (one process per GPU): the root creates
 * the frame on its GPU and publishes a 64-byte CUDA IPC handle; the other ranks open it on THEIR
 * device (peer access over NVLink is enabled lazily) and pass the mapped pointer to
 * aicb_render_srgb8_device_frame().  aicb_frame_read() is the root's device->host copy. */
aicb_status aicb_frame_create(aicb_ctx *, size_t n_pixels, void **d_frame, uint8_t handle_out[64]);
aicb_status aicb_frame_open(aicb_ctx *, const uint8_t handle[64], void **d_frame);
aicb_status aicb_frame_close(aicb_ctx *, void *d_frame, int opened);
aicb_status aicb_frame_read(aicb_ctx *, const void *d_frame, uint8_t (*out)[4], size_t n_pixels, void *stream);
/* Delivery without a collective.  A shared frame carries two monotonic counters behind its pixels:
 *   aicb_frame_signal          (every rank, after aicb_render_srgb8_device_frame on the same stream): "my strips of this
 *                              frame are stored" — arrived += 1, system-scope fence first so the pixels are visible;
 *   aicb_frame_wait_arrived    (owner): stream-ordered wait until arrived >= count (= ranks x frames so far);
 *   aicb_frame_release         (owner): consumed := frame_id once it is through with the frame (copied, displayed);
 *   aicb_frame_wait_consumed   (every rank, before storing into the frame again): wait until consumed >= frame_id.
 * All four are stream operations (one-thread kernels), none touches the host.  A wait gives up after ~2 s;
 * aicb_frame_timed_out reports it.  `n_pixels` is the frame's pixel count as given to aicb_frame_create. */
aicb_status aicb_frame_signal(aicb_ctx *, void *d_frame, size_t n_pixels, void *stream);
aicb_status aicb_frame_wait_arrived(aicb_ctx *, void *d_frame, size_t n_pixels, uint32_t count, void *stream);
aicb_status aicb_frame_release(aicb_ctx *, void *d_frame, size_t n_pixels, uint32_t frame_id, void *stream);
aicb_status aicb_frame_wait_consumed(aicb_ctx *, void *d_frame, size_t n_pixels, uint32_t frame_id, void *stream);
aicb_status aicb_frame_timed_out(aicb_ctx *, void *d_frame, size_t n_pixels, uint32_t *out);

/* ---------------------------------------------------------------------------------------------
 * Several GPUs from ONE process (csrc/group.cu): replaces the Rayon rows x pixels dispatch of
 * trace_scene_to_image_impl (renderer.rs:516-556) across devices for hosts that own their process (the Rust
 * `impl HeadlessRenderer`, INTEGRATION.md).  The scene is replicated on every device of the group; a frame is cut into
 * interleaved 16-row strips (strip s -> device s mod n); every device's encode kernel stores its pixels straight into
 * device 0's frame over NVLink (peer access) and device 0 copies the frame to the caller once the other devices'
 * completion events have fired: no collective, no host thread per GPU.  The same device may be named more than once
 * (tests).  aicb_render_info: counters summed over the devices, times = the slowest device's.
 * ------------------------------------------------------------------------------------------- */
typedef struct aicb_group aicb_group;
typedef struct aicb_group_scene aicb_group_scene;
aicb_status aicb_group_create(const int *device_ids, int n_devices, aicb_group **out);
void aicb_group_destroy(aicb_group *);
int aicb_group_size(const aicb_group *);
aicb_status aicb_group_scene_create(aicb_group *, const aicb_scene_desc *, aicb_group_scene **out);
void aicb_group_scene_destroy(aicb_group_scene *);
aicb_status aicb_group_scene_update_cubes(aicb_group_scene *, const int32_t (*cubes)[3], const uint16_t *block_ids,
                                          const uint8_t (*light)[4], size_t n);
/* == draw_rgba on the whole group: out_len must be fb_width * fb_height. */
aicb_status aicb_group_render_srgb8(aicb_group_scene *, const aicb_camera *, const aicb_options *,
                                    uint8_t (*out)[4], size_t out_len, aicb_render_info *info_or_null);
/* aicb_scene_update_blocks / aicb_scene_upload_light on every replica. */
aicb_status aicb_group_scene_update_blocks(aicb_group_scene *, const uint16_t *indices, const aicb_block_desc *descs, size_t n);
aicb_status aicb_group_scene_upload_light(aicb_group_scene *, const uint8_t (*light)[4], size_t n_texels);
/* Light propagation on the group: the aicb_light_* calls of the same names, same semantics and errors.  The relaxation
 * is sharded by slabs: member i owns an even share of whole queue tiles (1024 cubes, a slab along x) and only the owner
 * computes and applies its cubes; every applied texel is stored into every replica, so on return every member holds
 * the same light and aicb_group_render_srgb8 renders it.  Needs peer access with native atomics between every pair of
 * distinct member devices (AICB_ERR_UNSUPPORTED otherwise; enabled on the first call) and at most 16 members.  Edits
 * are validated in full before any replica changes.  A group of one member runs the single-scene propagation. */
aicb_status aicb_group_light_fast_evaluate(aicb_group_scene *);
aicb_status aicb_group_light_evaluate(aicb_group_scene *, uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff,
                                      uint64_t *chart_node_visits_or_null);
aicb_status aicb_group_light_edit_and_propagate(aicb_group_scene *, const int32_t (*cubes)[3], const uint16_t *new_ids,
                                                size_t n_edits, uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff);
/* member = position in the group (0..size-1), not a device id: the same device may be named twice */
aicb_status aicb_group_light_download(aicb_group_scene *, int member, uint8_t (*out)[4], size_t n_texels);
/* As aicb_light_stats for the last group propagation.  member -1: cube updates and chart node visits summed over the
 * members, rounds, device time of the slowest member; else that member's own counters. */
aicb_status aicb_group_light_stats(const aicb_group_scene *, int member, uint64_t out[4]);

/* == SpaceRaytracer::trace_ray (sr.rs:113-120) for a batch of explicit rays:
 * origin_dir[i] = {ox,oy,oz,dx,dy,dz}. Output as aicb_render_colorbuf. */
aicb_status aicb_trace_rays(aicb_scene *, const double (*origin_dir)[6], size_t n, const aicb_options *,
                            float (*out_colorbuf)[4], double *depth_or_null, aicb_hit *hit_or_null,
                            uint32_t *steps_or_null, aicb_render_info *info_or_null);

/* ---------------------------------------------------------------------------------------------
 * Camera construction (host only, no GPU): Camera::new + look_at_y_up + compute_matrices
 * (camera_struct.rs:86-110, 387-416, 459-471); eye_for_look_at (all-is-cubes/src/camera.rs:34-40).
 * ------------------------------------------------------------------------------------------- */
/* fov_y_degrees and view_distance are repaired like GraphicsOptions::repair. nominal_* is the
 * Viewport nominal size (aspect ratio); fb_* the framebuffer size. */
aicb_status aicb_camera_look_at(const double eye[3], const double target[3], double fov_y_degrees,
                                double view_distance, double nominal_width, double nominal_height,
                                uint32_t fb_width, uint32_t fb_height, float exposure, aicb_camera *out);
/* General form: rotation quaternion (i,j,k,r) + translation of the eye-to-world ViewTransform. */
aicb_status aicb_camera_from_view(const double rotation_ijkr[4], const double translation[3],
                                  double fov_y_degrees, double view_distance, double nominal_width,
                                  double nominal_height, uint32_t fb_width, uint32_t fb_height,
                                  float exposure, aicb_camera *out);
void aicb_eye_for_look_at(const aicb_aab *bounds, const double direction[3], double out_eye[3]);
/* Camera::project_ndc_into_world for one NDC point (host, for tests): out = origin xyz, dir xyz. */
void aicb_camera_project_ndc(const aicb_camera *, double ndc_x, double ndc_y, double out_origin_dir[6]);

/* ---------------------------------------------------------------------------------------------
 * Light propagation (secondary path): replaces Mutation::set x n + evaluate_light(epsilon)
 * (space.rs:1346-1352, 1496-1527; space/light/updater.rs:181-363).
 * ------------------------------------------------------------------------------------------- */
/* The static light-ray chart (space/light/chart/generator.rs:49-215) as the flat prefix tree the kernels
 * walk: 6 f32 weights + 6 child indices (0 = none) per node, root = 0.  Returns the node count
 * (114 779); either pointer may be NULL.  Host only. */
uint32_t aicb_light_chart(float *weights_or_null, uint32_t *children_or_null);
/* The same chart the way the kernels walk it: in depth-first preorder (children in Face6 order, the order walk_ray_tree
 * recurses in, updater.rs:500) and cut into chains — maximal paths of single-child nodes, which carry bit-identical
 * weights; a chain's nodes are consecutive in preorder and chains are numbered breadth first.  Host only; any pointer
 * may be NULL.  preorder[i] = index in aicb_light_chart's numbering of the i-th node in preorder (node count entries);
 * chains[c] = {first node (preorder), nodes, child chains, first child chain, parent's branch slot or 0xffff, own
 * branch slot or 0xffff}; euler = the Euler tour of the chain tree, chain | 0x8000 for the chain's exit (n_euler
 * entries = 2 * n_chains): the order in which the terms of a walk are added.  Returns the number of chains (1043). */
uint32_t aicb_light_chart_chains(uint32_t *preorder_or_null, uint32_t (*chains_or_null)[6], uint16_t *euler_or_null);
/* LightStorage::fast_evaluate_light (updater.rs:537-582): column-sweep initial guess + queue seeding. */
aicb_status aicb_light_fast_evaluate(aicb_scene *);
/* LightStorage::compute_light (updater.rs:368-418) for explicit cubes against the current field; does not
 * store anything (parity tests). out[i] = PackedLight::as_texel. */
aicb_status aicb_light_compute(aicb_scene *, const int32_t (*cubes)[3], size_t n, uint8_t (*out)[4]);
/* Mutation::evaluate_light(epsilon) (space.rs:1496-1527): relax until the highest queued priority is
 * <= Priority::from_difference(epsilon). */
aicb_status aicb_light_evaluate(aicb_scene *, uint8_t epsilon, uint64_t *updates_done, uint8_t *max_diff,
                                uint64_t *chart_node_visits_or_null);
aicb_status aicb_light_edit_and_propagate(aicb_scene *, const int32_t (*cubes)[3], const uint16_t *new_ids,
                                          size_t n_edits, uint8_t epsilon, uint64_t *updates_done,
                                          uint8_t *max_diff);
aicb_status aicb_light_download(aicb_scene *, uint8_t (*out)[4], size_t n_texels);
/* Counters of the last propagation (aicb_light_evaluate / aicb_light_edit_and_propagate) on this scene:
 * out[0] cube updates (compute_light calls, updater.rs:368), out[1] chart nodes visited by them, out[2] relaxation
 * rounds queued, out[3] device time of the propagation in microseconds (CUDA events on the context's stream).
 * After aicb_light_compute: out[0] cubes computed, out[1] chart nodes visited, out[2] cubes whose walk needed more
 * term slots than the chain walk holds and took the overflow walk instead, out[3] 0. */
aicb_status aicb_light_stats(const aicb_scene *, uint64_t out[4]);

/* ---------------------------------------------------------------------------------------------
 * Light propagation in budgeted steps, for a host that drives light once per tick (update_light_system,
 * space/step.rs:340-368): each step relaxes until nothing above epsilon is queued or its budget is used up, and
 * reports what is left in the queue.  The cubes whose light changed (SpaceChange::CubeLight) are listed on request.
 * ------------------------------------------------------------------------------------------- */
/* LightUpdatesInfo (space/light/updater.rs:970-984) of one step, plus counters.  40 bytes. */
typedef struct aicb_light_updates {
    uint64_t update_count;          /* compute_light calls applied by this step */
    uint64_t queue_count;           /* cubes queued on return (queue byte > 0, any priority) */
    uint64_t chart_node_visits;
    uint32_t rounds;                /* relaxation rounds queued by this step (as aicb_light_stats out[2]) */
    uint8_t  max_update_difference;
    uint8_t  max_queue_priority;    /* highest queued Priority on return, 0 = empty (queue.rs:28-50 values) */
    uint8_t  _pad[2];
    float    device_ms;             /* CUDA-event time of the step (group: the slowest member's) */
} aicb_light_updates;

/* Mutation::set x n_edits (exactly as aicb_light_edit_and_propagate), then update_light_from_queue(budget)
 * (updater.rs:181-291) down to epsilon, stopping when max_updates cube updates are done or the time budget is
 * used up.  max_updates: UINT64_MAX = no limit, 0 = no relaxation (edits and the report only).
 * budget_us < 0 = no time limit, 0 = no relaxation; a positive budget becomes an update cap (at least 1) through the
 * scene's running estimate of device microseconds per cube update, which every step that updated a cube refines.
 * With neither limit the step relaxes exactly as aicb_light_edit_and_propagate does.  A step stops between rounds:
 * the cubes a round takes are the first ones of its priority band in index order.  out may be NULL; after a step
 * aicb_light_stats reports its counters.  LightPhysics::None, NULL arrays with n_edits > 0, an invalid edit or a NaN
 * budget is AICB_ERR_INVALID, and then nothing changed. */
aicb_status aicb_light_step(aicb_scene *, const int32_t (*cubes)[3], const uint16_t *new_ids, size_t n_edits,
                            uint8_t epsilon, uint64_t max_updates, double budget_us, aicb_light_updates *out);
aicb_status aicb_group_light_step(aicb_group_scene *, const int32_t (*cubes)[3], const uint16_t *new_ids,
                                  size_t n_edits, uint8_t epsilon, uint64_t max_updates, double budget_us,
                                  aicb_light_updates *out);

/* SpaceChange::CubeLight for a host that mirrors the light.  Enabling records the current light as the baseline
 * (4 bytes per cube of device memory, freed when disabled).  take_changes lists every cube whose texel differs
 * from the baseline, in increasing linear (Z-major) index, as world coordinates plus the current texel.  If the
 * count is <= cap, it writes the list and moves the baseline of those cubes to the current value.  Otherwise it
 * writes and consumes nothing.  *n_changed is always the count.  cubes / texels may be NULL only with cap == 0.
 * Taking changes without tracking enabled is AICB_ERR_INVALID.  A group tracks member 0's replica; all replicas
 * are identical on return from every light call. */
aicb_status aicb_light_track_changes(aicb_scene *, int enable);
aicb_status aicb_light_take_changes(aicb_scene *, int32_t (*cubes)[3], uint8_t (*texels)[4], size_t cap,
                                    size_t *n_changed);
aicb_status aicb_group_light_track_changes(aicb_group_scene *, int enable);
aicb_status aicb_group_light_take_changes(aicb_group_scene *, int32_t (*cubes)[3], uint8_t (*texels)[4],
                                          size_t cap, size_t *n_changed);

#ifdef __cplusplus
}
#endif
#endif /* AICB200_H */
