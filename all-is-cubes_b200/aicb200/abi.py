"""ctypes mirror of include/aicb200.h (plain data only; no compute)."""
import ctypes as C

ABI_VERSION = 2

OK, ERR_INVALID, ERR_OOM, ERR_CUDA, ERR_UNSUPPORTED, ERR_BUSY, ERR_RETRY = range(7)
STATUS_NAMES = {0: "OK", 1: "ERR_INVALID", 2: "ERR_OOM", 3: "ERR_CUDA", 4: "ERR_UNSUPPORTED", 5: "ERR_BUSY", 6: "ERR_RETRY"}

FACE_WITHIN, FACE_NX, FACE_NY, FACE_NZ, FACE_PX, FACE_PY, FACE_PZ = range(7)
FOG_NONE, FOG_ABRUPT, FOG_COMPROMISE, FOG_PHYSICAL = range(4)
LIGHT_NONE, LIGHT_FLAT, LIGHT_COARSE, LIGHT_LINEAR, LIGHT_SMOOTHSTEP, LIGHT_BOUNCE = range(6)
TRANSPARENCY_SURFACE, TRANSPARENCY_VOLUMETRIC, TRANSPARENCY_THRESHOLD = range(3)
TONE_CLAMP, TONE_REINHARD = range(2)


class Aab(C.Structure):
    _fields_ = [("lower", C.c_int32 * 3), ("size", C.c_uint32 * 3)]


class Voxel(C.Structure):
    _fields_ = [("rgba", C.c_float * 4), ("emission", C.c_float * 3), ("_pad", C.c_float)]


class BlockDesc(C.Structure):
    _fields_ = [
        ("resolution", C.c_uint8),
        ("is_air", C.c_uint8),
        ("light_opaque_faces", C.c_uint8),
        ("light_visible", C.c_uint8),
        ("voxel_bounds", Aab),
        ("indices", C.c_void_p),
        ("n_indices", C.c_size_t),
        ("palette", C.c_void_p),
        ("n_palette", C.c_size_t),
        ("light_face_colors", (C.c_float * 4) * 6),
        ("light_color", C.c_float * 4),
        ("light_emission", C.c_float * 3),
        ("_pad", C.c_float),
    ]


class Sky(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("colors", (C.c_float * 3) * 8)]


class SceneDesc(C.Structure):
    _fields_ = [
        ("bounds", Aab),
        ("block_ids", C.c_void_p),
        ("light", C.c_void_p),
        ("blocks", C.POINTER(BlockDesc)),
        ("n_blocks", C.c_size_t),
        ("sky", Sky),
        ("light_max_distance", C.c_uint8),
        ("_pad", C.c_uint8 * 7),
    ]


class CameraData(C.Structure):
    _fields_ = [
        ("inverse_projection_view", C.c_double * 16),
        ("fb_width", C.c_uint32),
        ("fb_height", C.c_uint32),
        ("exposure", C.c_float),
        ("_pad", C.c_uint32),
    ]


class Options(C.Structure):
    _fields_ = [
        ("fog", C.c_uint8),
        ("lighting_display", C.c_uint8),
        ("transparency", C.c_uint8),
        ("antialiasing_always", C.c_uint8),
        ("tone_mapping", C.c_uint8),
        ("debug_pixel_cost", C.c_uint8),
        ("include_sky", C.c_uint8),
        ("bounce_samples", C.c_uint8),
        ("transparency_threshold", C.c_float),
        ("maximum_intensity", C.c_float),
        ("view_distance", C.c_double),
    ]


class Shard(C.Structure):
    _fields_ = [("strip_rows", C.c_uint32), ("index", C.c_uint32), ("count", C.c_uint32)]


class RenderInfo(C.Structure):
    _fields_ = [
        ("cubes_traced", C.c_uint64),
        ("rays", C.c_uint64),
        ("algorithmic_bytes", C.c_uint64),
        ("counters", C.c_uint64 * 6),
        ("kernel_ms", C.c_float),
        ("flaws", C.c_uint16),
        ("_pad", C.c_uint16),
        ("stage_ms", C.c_float * 4),
    ]


class Hit(C.Structure):
    _fields_ = [("cube", C.c_int32 * 3), ("voxel", C.c_int32 * 3), ("resolution", C.c_int32), ("face", C.c_int32)]


# Every symbol include/aicb200.h declares (tests check the built library exports all of them).
class Layer(C.Structure):
    _fields_ = [("scene", C.c_void_p), ("camera", C.POINTER(CameraData)), ("options", C.POINTER(Options))]


class LightUpdates(C.Structure):
    """aicb_light_updates: LightUpdatesInfo (updater.rs:970-984) of one aicb_light_step, plus counters."""
    _fields_ = [
        ("update_count", C.c_uint64),
        ("queue_count", C.c_uint64),
        ("chart_node_visits", C.c_uint64),
        ("rounds", C.c_uint32),
        ("max_update_difference", C.c_uint8),
        ("max_queue_priority", C.c_uint8),
        ("_pad", C.c_uint8 * 2),
        ("device_ms", C.c_float),
    ]


TEXT_ENTERED_SPACE, TEXT_EMPTY, TEXT_INCOMPLETE = -1, -2, -3

EXPORTED_SYMBOLS = [
    "aicb_abi_version",
    "aicb_ctx_create",
    "aicb_ctx_destroy",
    "aicb_ctx_stage_timing",
    "aicb_last_error",
    "aicb_scene_create",
    "aicb_scene_update_cubes",
    "aicb_scene_update_blocks",
    "aicb_scene_upload_light",
    "aicb_scene_destroy",
    "aicb_scene_device_bytes",
    "aicb_shard_pixel_count",
    "aicb_render_srgb8",
    "aicb_render_rgba16f",
    "aicb_render_colorbuf",
    "aicb_render_text",
    "aicb_render_layers_srgb8",
    "aicb_ortho_image_size",
    "aicb_render_orthographic",
    "aicb_render_srgb8_device",
    "aicb_render_srgb8_device_frame",
    "aicb_render_finish",
    "aicb_frame_create",
    "aicb_frame_open",
    "aicb_frame_close",
    "aicb_frame_read",
    "aicb_frame_signal",
    "aicb_frame_wait_arrived",
    "aicb_frame_release",
    "aicb_frame_wait_consumed",
    "aicb_frame_timed_out",
    "aicb_trace_rays",
    "aicb_camera_look_at",
    "aicb_camera_from_view",
    "aicb_eye_for_look_at",
    "aicb_camera_project_ndc",
    "aicb_light_chart",
    "aicb_light_chart_chains",
    "aicb_light_fast_evaluate",
    "aicb_light_compute",
    "aicb_light_evaluate",
    "aicb_light_edit_and_propagate",
    "aicb_light_download",
    "aicb_light_stats",
    "aicb_group_create",
    "aicb_group_destroy",
    "aicb_group_size",
    "aicb_group_scene_create",
    "aicb_group_scene_destroy",
    "aicb_group_scene_update_cubes",
    "aicb_group_render_srgb8",
    "aicb_group_scene_update_blocks",
    "aicb_group_scene_upload_light",
    "aicb_group_light_fast_evaluate",
    "aicb_group_light_evaluate",
    "aicb_group_light_edit_and_propagate",
    "aicb_group_light_download",
    "aicb_group_light_stats",
    "aicb_light_step",
    "aicb_group_light_step",
    "aicb_light_track_changes",
    "aicb_light_take_changes",
    "aicb_group_light_track_changes",
    "aicb_group_light_take_changes",
]
