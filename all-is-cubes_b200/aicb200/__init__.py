"""aicb200 — Python binding over the C ABI of libaicb200.so.

Mirrors the reference's raytracer surface (names and argument meaning):
`GraphicsOptions` (all-is-cubes-render/src/camera/graphics_options.rs:28), `Viewport`
(camera/viewport.rs:24), `Camera` (camera/camera_struct.rs:43), `SpaceRaytracer`
(raytracer/sr.rs:51), `RtRenderer` / `HeadlessRenderer` (raytracer/renderer.rs:35,
headless.rs:17), `Rendering` (headless.rs:52).  `Space`/`Block` here are only the flattened
snapshot the raytracer reads (SpaceRaytracer::new, sr.rs:64-88) — not the reference's world model.

This module contains no compute: every pixel comes from the CUDA kernels behind the C ABI.
If the library is missing or there is no GPU the calls fail loudly (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math
import os
from typing import Optional, Sequence

import numpy as np

from . import abi
from .abi import (FOG_ABRUPT, FOG_COMPROMISE, FOG_NONE, FOG_PHYSICAL, LIGHT_BOUNCE, LIGHT_COARSE, LIGHT_FLAT, LIGHT_LINEAR,
                  LIGHT_NONE, LIGHT_SMOOTHSTEP, TONE_CLAMP, TONE_REINHARD, TRANSPARENCY_SURFACE,
                  TRANSPARENCY_THRESHOLD, TRANSPARENCY_VOLUMETRIC)

PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("AICB200_LIB") or os.path.join(PKG_DIR, "libaicb200.so")  # override: kernel experiments only


class AicbError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{abi.STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


_lib = None


def load_library() -> C.CDLL:
    """Load libaicb200.so (built in-tree by __graft_entry__.build()). Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.aicb_abi_version.restype = C.c_uint32
    lib.aicb_last_error.restype = C.c_char_p
    lib.aicb_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.aicb_ctx_destroy.argtypes = [C.c_void_p]
    lib.aicb_ctx_stage_timing.argtypes = [C.c_void_p, C.c_int]
    lib.aicb_scene_create.argtypes = [C.c_void_p, C.POINTER(abi.SceneDesc), C.POINTER(C.c_void_p)]
    lib.aicb_scene_destroy.argtypes = [C.c_void_p]
    lib.aicb_scene_device_bytes.argtypes = [C.c_void_p]
    lib.aicb_scene_device_bytes.restype = C.c_uint64
    lib.aicb_scene_update_cubes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_scene_update_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_scene_upload_light.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_shard_pixel_count.argtypes = [C.POINTER(abi.CameraData), C.POINTER(abi.Shard)]
    lib.aicb_shard_pixel_count.restype = C.c_size_t
    lib.aicb_render_srgb8.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options),
                                      C.POINTER(abi.Shard), C.c_void_p, C.c_size_t, C.POINTER(abi.RenderInfo)]
    lib.aicb_render_colorbuf.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options),
                                         C.POINTER(abi.Shard), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.POINTER(abi.RenderInfo)]
    lib.aicb_render_rgba16f.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options),
                                        C.POINTER(abi.Shard), C.c_void_p, C.c_size_t, C.POINTER(abi.RenderInfo)]
    lib.aicb_render_srgb8_device.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options),
                                             C.POINTER(abi.Shard), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.aicb_render_srgb8_device_frame.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options),
                                                   C.POINTER(abi.Shard), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.aicb_frame_create.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]
    lib.aicb_frame_open.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.aicb_frame_close.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.aicb_frame_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.aicb_frame_signal.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.aicb_frame_wait_arrived.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]
    lib.aicb_frame_release.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]
    lib.aicb_frame_wait_consumed.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]
    lib.aicb_frame_timed_out.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32)]
    lib.aicb_render_finish.argtypes = [C.c_void_p, C.POINTER(abi.RenderInfo)]
    lib.aicb_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(abi.Options), C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(abi.RenderInfo)]
    lib.aicb_camera_look_at.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double, C.c_double,
                                        C.c_double, C.c_double, C.c_uint32, C.c_uint32, C.c_float,
                                        C.POINTER(abi.CameraData)]
    lib.aicb_camera_from_view.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double, C.c_double,
                                          C.c_double, C.c_double, C.c_uint32, C.c_uint32, C.c_float,
                                          C.POINTER(abi.CameraData)]
    lib.aicb_eye_for_look_at.argtypes = [C.POINTER(abi.Aab), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.aicb_eye_for_look_at.restype = None
    lib.aicb_camera_project_ndc.argtypes = [C.POINTER(abi.CameraData), C.c_double, C.c_double,
                                            C.POINTER(C.c_double)]
    lib.aicb_camera_project_ndc.restype = None
    lib.aicb_light_edit_and_propagate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint8,
                                                  C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)]
    lib.aicb_light_download.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_light_stats.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.aicb_render_text.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options), C.c_void_p, C.c_size_t,
                                     C.POINTER(abi.RenderInfo)]
    lib.aicb_render_layers_srgb8.argtypes = [C.POINTER(abi.Layer), C.POINTER(abi.Layer), C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_size_t, C.POINTER(abi.RenderInfo)]
    lib.aicb_ortho_image_size.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.aicb_render_orthographic.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.POINTER(abi.RenderInfo)]
    lib.aicb_group_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
    lib.aicb_group_destroy.argtypes = [C.c_void_p]
    lib.aicb_group_destroy.restype = None
    lib.aicb_group_size.argtypes = [C.c_void_p]
    lib.aicb_group_scene_create.argtypes = [C.c_void_p, C.POINTER(abi.SceneDesc), C.POINTER(C.c_void_p)]
    lib.aicb_group_scene_destroy.argtypes = [C.c_void_p]
    lib.aicb_group_scene_destroy.restype = None
    lib.aicb_group_scene_update_cubes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_group_render_srgb8.argtypes = [C.c_void_p, C.POINTER(abi.CameraData), C.POINTER(abi.Options), C.c_void_p,
                                            C.c_size_t, C.POINTER(abi.RenderInfo)]
    lib.aicb_group_scene_update_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_group_scene_upload_light.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.aicb_group_light_fast_evaluate.argtypes = [C.c_void_p]
    lib.aicb_group_light_evaluate.argtypes = [C.c_void_p, C.c_uint8, C.POINTER(C.c_uint64), C.POINTER(C.c_uint8),
                                              C.POINTER(C.c_uint64)]
    lib.aicb_group_light_edit_and_propagate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint8,
                                                        C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)]
    lib.aicb_group_light_download.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    lib.aicb_group_light_stats.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]
    lib.aicb_light_chart.argtypes = [C.c_void_p, C.c_void_p]
    lib.aicb_light_chart.restype = C.c_uint32
    lib.aicb_light_fast_evaluate.argtypes = [C.c_void_p]
    lib.aicb_light_compute.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.aicb_light_evaluate.argtypes = [C.c_void_p, C.c_uint8, C.POINTER(C.c_uint64), C.POINTER(C.c_uint8),
                                        C.POINTER(C.c_uint64)]
    for prefix in ("aicb_", "aicb_group_"):   # the scene and the group versions take the same arguments
        getattr(lib, prefix + "light_step").argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint8,
                                                        C.c_uint64, C.c_double, C.POINTER(abi.LightUpdates)]
        getattr(lib, prefix + "light_track_changes").argtypes = [C.c_void_p, C.c_int]
        getattr(lib, prefix + "light_take_changes").argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                                                C.POINTER(C.c_size_t)]
    if lib.aicb_abi_version() != abi.ABI_VERSION:
        raise RuntimeError("libaicb200.so ABI version mismatch")
    _lib = lib
    return lib


# The camera matrices (host-only code, all-is-cubes_b200/host/camera.cpp) are reached through the C ABI of
# libaicb200.so by default.  bench.py's reference arm must not load the product library at all, so the same host
# source is also compiled into the oracle library under orc_* names; use_camera_library() points Camera at it.
_camera_lib = None
_camera_prefix = "aicb_"


def use_camera_library(lib, prefix: str):
    """Route Camera / eye_for_look_at through another shared library exporting <prefix>camera_look_at,
    <prefix>camera_from_view, <prefix>eye_for_look_at, <prefix>camera_project_ndc (same signatures)."""
    global _camera_lib, _camera_prefix
    for name in ("camera_look_at", "camera_from_view"):
        fn = getattr(lib, prefix + name)
        fn.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double, C.c_double, C.c_double, C.c_double,
                       C.c_uint32, C.c_uint32, C.c_float, C.POINTER(abi.CameraData)]
        fn.restype = C.c_int
    fn = getattr(lib, prefix + "eye_for_look_at")
    fn.argtypes = [C.POINTER(abi.Aab), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    fn.restype = None
    fn = getattr(lib, prefix + "camera_project_ndc")
    fn.argtypes = [C.POINTER(abi.CameraData), C.c_double, C.c_double, C.POINTER(C.c_double)]
    fn.restype = None
    _camera_lib, _camera_prefix = lib, prefix


def _cam(name: str):
    lib = _camera_lib if _camera_lib is not None else load_library()
    return getattr(lib, _camera_prefix + name)


def _check_cam(status: int):
    if status != abi.OK:
        if _camera_lib is not None:
            raise AicbError(status, "camera construction failed")
        _check(status)


def _check(status: int):
    if status != abi.OK:
        raise AicbError(status, load_library().aicb_last_error().decode("utf-8", "replace"))


# ------------------------------------------------------------------------------------------------
# GraphicsOptions / Viewport / Camera
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class GraphicsOptions:
    """The pixel-affecting subset of GraphicsOptions (graphics_options.rs:28-150).
    Defaults are GraphicsOptions::default() (graphics_options.rs:251-281)."""
    fog: int = FOG_ABRUPT
    fov_y: float = 90.0
    tone_mapping: int = TONE_CLAMP
    maximum_intensity: float = math.inf
    exposure: float = 1.0  # ExposureOption::Fixed(1)
    view_distance: float = 200.0
    lighting_display: int = LIGHT_LINEAR
    transparency: int = TRANSPARENCY_VOLUMETRIC
    transparency_threshold: float = 0.5
    antialiasing_always: bool = False
    debug_pixel_cost: bool = False
    bounce_samples: int = 1  # LightingOption::Bounce { samples } (graphics_options.rs:464-467)

    @staticmethod
    def unaltered_colors() -> "GraphicsOptions":
        """GraphicsOptions::UNALTERED_COLORS (graphics_options.rs:168-190)."""
        return GraphicsOptions(fog=FOG_NONE, lighting_display=LIGHT_NONE)

    def repair(self) -> "GraphicsOptions":
        """graphics_options.rs:194-198"""
        return dataclasses.replace(self, fov_y=min(max(self.fov_y, 1.0), 189.0),
                                   view_distance=min(max(self.view_distance, 1.0), 10000.0))

    def to_abi(self, include_sky: bool = True) -> abi.Options:
        o = abi.Options()
        o.fog = self.fog
        o.lighting_display = self.lighting_display
        o.transparency = self.transparency
        o.antialiasing_always = 1 if self.antialiasing_always else 0
        o.tone_mapping = self.tone_mapping
        o.debug_pixel_cost = 1 if self.debug_pixel_cost else 0
        o.include_sky = 1 if include_sky else 0
        o.bounce_samples = self.bounce_samples if self.lighting_display == LIGHT_BOUNCE else 0
        o.transparency_threshold = self.transparency_threshold
        o.maximum_intensity = self.maximum_intensity
        o.view_distance = min(max(self.view_distance, 1.0), 10000.0)
        return o


@dataclasses.dataclass
class Viewport:
    """camera/viewport.rs:24-37"""
    nominal_size: tuple
    framebuffer_size: tuple

    @staticmethod
    def with_scale(scale: float, framebuffer_size) -> "Viewport":
        w, h = framebuffer_size
        return Viewport((w / scale if scale else math.inf, h / scale if scale else math.inf), (int(w), int(h)))


class Camera:
    """Camera (camera_struct.rs:43): options + viewport + view transform -> matrices.
    Matrix construction happens in the C ABI (host code, aicb_camera_*)."""

    def __init__(self, options: GraphicsOptions, viewport: Viewport):
        self.options = options.repair()
        self.viewport = viewport
        self._rotation = (0.0, 0.0, 0.0, 1.0)
        self._translation = (0.0, 0.0, 0.0)
        self.data = abi.CameraData()
        self._compute()

    def _compute(self):
        q = (C.c_double * 4)(*self._rotation)
        t = (C.c_double * 3)(*self._translation)
        _check_cam(_cam("camera_from_view")(q, t, self.options.fov_y, self.options.view_distance,
                                         float(self.viewport.nominal_size[0]), float(self.viewport.nominal_size[1]),
                                         self.viewport.framebuffer_size[0], self.viewport.framebuffer_size[1],
                                         self.options.exposure, C.byref(self.data)))

    def set_view_transform(self, rotation_ijkr: Sequence[float], translation: Sequence[float]):
        self._rotation = tuple(float(v) for v in rotation_ijkr)
        self._translation = tuple(float(v) for v in translation)
        self._compute()

    def look_at_y_up(self, eye: Sequence[float], target: Sequence[float]):
        """camera_struct.rs:459-471"""
        e = (C.c_double * 3)(*[float(v) for v in eye])
        t = (C.c_double * 3)(*[float(v) for v in target])
        _check_cam(_cam("camera_look_at")(e, t, self.options.fov_y, self.options.view_distance,
                                       float(self.viewport.nominal_size[0]), float(self.viewport.nominal_size[1]),
                                       self.viewport.framebuffer_size[0], self.viewport.framebuffer_size[1],
                                       self.options.exposure, C.byref(self.data)))

    def project_ndc_into_world(self, x: float, y: float) -> np.ndarray:
        """camera_struct.rs:238-257 -> [ox,oy,oz,dx,dy,dz]"""
        out = (C.c_double * 6)()
        _cam("camera_project_ndc")(C.byref(self.data), x, y, out)
        return np.array(out[:], dtype=np.float64)

    @property
    def inverse_projection_view(self) -> np.ndarray:
        return np.array(self.data.inverse_projection_view[:], dtype=np.float64).reshape(4, 4)


def eye_for_look_at(bounds_lower, bounds_size, direction) -> np.ndarray:
    """all-is-cubes/src/camera.rs:34-40"""
    b = abi.Aab()
    b.lower[:] = [int(v) for v in bounds_lower]
    b.size[:] = [int(v) for v in bounds_size]
    d = (C.c_double * 3)(*[float(v) for v in direction])
    out = (C.c_double * 3)()
    _cam("eye_for_look_at")(C.byref(b), d, out)
    return np.array(out[:], dtype=np.float64)


# ------------------------------------------------------------------------------------------------
# Flattened Space snapshot
# ------------------------------------------------------------------------------------------------
class Block:
    """One Space palette entry as the raytracer sees it (TracingBlock, sr.rs:569-587)."""

    def __init__(self, *, color=None, emission=(0.0, 0.0, 0.0), is_air=False, resolution=1, voxel_lower=None,
                 indices: Optional[np.ndarray] = None, palette: Optional[np.ndarray] = None):
        self.is_air = bool(is_air)
        self.resolution = int(resolution)
        if indices is None:
            c = (0.0, 0.0, 0.0, 0.0) if color is None else tuple(color)
            self.palette = np.zeros((1, 8), dtype=np.float32)
            self.palette[0, :4] = c
            self.palette[0, 4:7] = emission
            self.indices = None
            self.voxel_lower = (0, 0, 0)
            self.voxel_size = (1, 1, 1)
            self.resolution = 1
        else:
            assert indices.ndim == 3 and indices.dtype == np.uint16
            self.indices = np.ascontiguousarray(indices)
            self.palette = np.ascontiguousarray(palette, dtype=np.float32)
            assert self.palette.ndim == 2 and self.palette.shape[1] == 8
            self.voxel_lower = tuple(int(v) for v in (voxel_lower or (0, 0, 0)))
            self.voxel_size = tuple(int(v) for v in indices.shape)
        self._derive_for_light()

    def _derive_for_light(self):
        """EvaluatedBlock derived data read by light propagation (block/eval/derived.rs:80-104 for single voxels,
        :105-235 for recursive blocks: a restatement for the synthetic blocks of the tests and benches — block
        evaluation itself is out of scope, SURVEY §2 #11; the oracle and the GPU consume whatever is supplied here)."""
        if self.is_air:
            self.light_opaque_faces = 0
            self.light_visible = False
            self.light_color = (0.0, 0.0, 0.0, 0.0)
            self.light_face_colors = [(0.0, 0.0, 0.0, 0.0)] * 6
            self.light_emission = (0.0, 0.0, 0.0)
            return
        if self.indices is None:
            c = tuple(float(v) for v in self.palette[0, :4])
            e = tuple(float(v) for v in self.palette[0, 4:7])
            self.light_color = c
            self.light_face_colors = [c] * 6
            self.light_emission = e
            self.light_opaque_faces = 0x3F if c[3] == 1.0 else 0
            self.light_visible = (c[3] != 0.0) or any(v != 0.0 for v in e)
            return
        # compute_derived (block/eval/derived.rs:80-235): every face is "rendered" by axis-aligned rays through the voxel
        # data (trace_for_eval, raytracer_components.rs:174-200), starting at the first layer of the DATA bounds seen
        # from that face; a face colour is the alpha-weighted mean of its pixels with alpha = coverage of the full
        # face.  The sums run in numpy's order, not iproduct!'s: last-bit differences only.
        f32 = np.float32
        r = self.resolution
        lo, sz = self.voxel_lower, self.voxel_size
        vox = self.palette[self.indices]            # [sx, sy, sz, 8]: rgba, emission
        thickness = f32(1.0) / f32(r)

        # apply_transmittance (raytracer_components.rs:215-258) of every voxel for thickness 1/resolution
        alpha_v = vox[..., 3]
        unit_t = (f32(1.0) - alpha_v).astype(np.float32)
        with np.errstate(invalid="ignore", divide="ignore"):
            depth_t = np.power(unit_t, thickness, dtype=np.float32)
            adj = np.clip(f32(1.0) - depth_t, f32(0.0), f32(1.0)).astype(np.float32)
            coeff = np.where(unit_t == 1.0, thickness, np.maximum((depth_t - f32(1.0)) / (unit_t - f32(1.0)), f32(0.0))).astype(np.float32)
        adj = np.where(alpha_v >= 1.0, f32(1.0), np.where(alpha_v <= 0.0, f32(0.0), adj)).astype(np.float32)
        coeff = np.where(alpha_v >= 1.0, f32(1.0), coeff).astype(np.float32)

        self.light_opaque_faces = 0
        cols = []
        all_color = np.zeros(3, dtype=np.float32)
        all_alpha = f32(0.0)
        all_em = np.zeros(3, dtype=np.float32)
        count = 0
        area = f32(r * r)
        for f in range(6):                          # NX NY NZ PX PY PZ
            axis, positive = f % 3, f >= 3
            # trace_for_eval for all pixels of the face at once: layers of the data from the face inwards
            order = range(sz[axis] - 1, -1, -1) if positive else range(sz[axis])
            shape = tuple(sz[a] for a in range(3) if a != axis)
            light = np.zeros(shape + (3,), dtype=np.float32)
            T = np.ones(shape, dtype=np.float32)
            em = np.zeros(shape + (3,), dtype=np.float32)
            live = np.ones(shape, dtype=bool)
            for k in order:
                v = np.take(vox, k, axis=axis)
                a = np.take(adj, k, axis=axis)
                c = np.take(coeff, k, axis=axis)
                em = np.where(live[..., None], em + (v[..., 4:7] * c[..., None]) * T[..., None], em).astype(np.float32)
                light = np.where(live[..., None], light + (v[..., :3] * a[..., None]) * T[..., None], light).astype(np.float32)
                T = np.where(live, T * (f32(1.0) - a), T).astype(np.float32)
                live &= ~(T < f32(1.0 / 256.0))
                if not live.any():
                    break
            pa = np.where(T >= 1.0, f32(0.0), f32(1.0) - T).astype(np.float32)              # Rgba::from(ColorBuf)
            with np.errstate(invalid="ignore", divide="ignore"):
                prgb = np.where(pa[..., None] > 0, light / pa[..., None], f32(0.0)).astype(np.float32)
            csum = (prgb * pa[..., None]).reshape(-1, 3).sum(axis=0, dtype=np.float32)
            asum = f32(pa.sum(dtype=np.float32))
            all_em = (all_em + em.reshape(-1, 3).sum(axis=0, dtype=np.float32)).astype(np.float32)
            count += pa.size
            all_color = (all_color + csum).astype(np.float32)
            all_alpha = f32(all_alpha + asum)
            if asum > 0:
                cm = csum / asum
                cols.append((float(cm[0]), float(cm[1]), float(cm[2]), float(min(max(asum / area, f32(0.0)), f32(1.0)))))
            else:
                cols.append((0.0, 0.0, 0.0, 0.0))
            # opaque[face] (derived.rs:196-209): the block's own surface layer lies inside the data and is fully opaque
            others = [a_ for a_ in range(3) if a_ != axis]
            covers = all((lo[a_] == 0 and sz[a_] == r) for a_ in others) and \
                ((lo[axis] + sz[axis] == r) if positive else (lo[axis] == 0))
            if covers and np.all(np.take(alpha_v, sz[axis] - 1 if positive else 0, axis=axis) == 1.0):
                self.light_opaque_faces |= 1 << f
        self.light_face_colors = cols
        surface = f32(6 * r * r)
        if all_alpha > 0:
            c = all_color / all_alpha
            self.light_color = (float(c[0]), float(c[1]), float(c[2]), float(min(max(all_alpha / surface, f32(0.0)), f32(1.0))))
        else:
            self.light_color = (0.0, 0.0, 0.0, 0.0)
        self.light_emission = tuple(float(v) for v in (all_em / surface)) if count else (0.0, 0.0, 0.0)
        self.light_visible = bool((vox[..., 3] != 0).any() or (vox[..., 4:7] != 0).any())

    @staticmethod
    def air() -> "Block":
        return Block(is_air=True)


class Space:
    """What SpaceRaytracer::new reads from space::Read (sr.rs:64-88): bounds, per-cube block
    index (shape [X,Y,Z], C order == Vol Z-major, vol.rs:1013-1018), optional PackedLight texels
    (shape [X,Y,Z,4]), block table, sky."""

    def __init__(self, lower, block_ids: np.ndarray, blocks: Sequence[Block], light: Optional[np.ndarray] = None,
                 sky_colors=None, light_max_distance: int = 0):
        assert block_ids.ndim == 3
        self.lower = tuple(int(v) for v in lower)
        self.block_ids = np.ascontiguousarray(block_ids, dtype=np.uint16)
        self.size = tuple(int(v) for v in self.block_ids.shape)
        self.blocks = list(blocks)
        self.light = None if light is None else np.ascontiguousarray(light, dtype=np.uint8)
        if self.light is not None:
            assert self.light.shape == self.size + (4,)
        if sky_colors is None:
            # Sky::DEFAULT = Uniform(DAY_SKY_COLOR = srgb[243 243 255]) (sky.rs:24, palette.rs:63)
            sky_colors = [srgb8_to_linear((243, 243, 255))]
        self.sky_colors = np.asarray(sky_colors, dtype=np.float32).reshape(-1, 3)
        assert self.sky_colors.shape[0] in (1, 8)
        self.light_max_distance = int(light_max_distance)

    def to_desc(self):
        """Returns (abi.SceneDesc, keepalive list)."""
        keep = []
        d = abi.SceneDesc()
        d.bounds.lower[:] = self.lower
        d.bounds.size[:] = self.size
        d.block_ids = self.block_ids.ctypes.data
        d.light = self.light.ctypes.data if self.light is not None else None
        arr = (abi.BlockDesc * len(self.blocks))()
        for i, b in enumerate(self.blocks):
            fill_block_desc(arr[i], b)
            keep.append(b)
        d.blocks = arr
        d.n_blocks = len(self.blocks)
        d.sky.kind = 0 if self.sky_colors.shape[0] == 1 else 1
        for k in range(self.sky_colors.shape[0]):
            d.sky.colors[k][:] = [float(v) for v in self.sky_colors[k]]
        d.light_max_distance = self.light_max_distance
        keep.append(arr)
        keep.append(self)
        return d, keep


def fill_block_desc(bd, b):
    """Block -> aicb_block_desc (the arrays stay owned by `b`)."""
    bd.resolution = b.resolution
    bd.is_air = 1 if b.is_air else 0
    bd.voxel_bounds.lower[:] = b.voxel_lower
    bd.voxel_bounds.size[:] = b.voxel_size
    if b.indices is not None:
        bd.indices = b.indices.ctypes.data
        bd.n_indices = b.indices.size
    else:
        bd.indices = None
        bd.n_indices = 0
    bd.palette = b.palette.ctypes.data
    bd.n_palette = b.palette.shape[0]
    bd.light_opaque_faces = b.light_opaque_faces
    bd.light_visible = 1 if b.light_visible else 0
    for f in range(6):
        bd.light_face_colors[f][:] = b.light_face_colors[f]
    bd.light_color[:] = b.light_color
    bd.light_emission[:] = b.light_emission


def light_chart():
    """The static light-ray chart (space/light/chart/generator.rs) as (weights [n,6] f32, children [n,6] u32)."""
    lib = load_library()
    n = lib.aicb_light_chart(None, None)
    w = np.zeros((n, 6), dtype=np.float32)
    ch = np.zeros((n, 6), dtype=np.uint32)
    lib.aicb_light_chart(w.ctypes.data, ch.ctypes.data)
    return w, ch


def light_chart_chains():
    """The chart as the chain walk sees it: (preorder [n] -> node of light_chart(), chains [c,6] u32 = first node in
    preorder, nodes, child chains, first child chain, parent's branch slot, own branch slot; euler [2c] u16)."""
    lib = load_library()
    lib.aicb_light_chart_chains.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.aicb_light_chart_chains.restype = C.c_uint32
    n_nodes = lib.aicb_light_chart(None, None)
    n_chains = lib.aicb_light_chart_chains(None, None, None)
    pre = np.zeros(n_nodes, dtype=np.uint32)
    chains = np.zeros((n_chains, 6), dtype=np.uint32)
    euler = np.zeros(2 * n_chains, dtype=np.uint16)
    lib.aicb_light_chart_chains(pre.ctypes.data, chains.ctypes.data, euler.ctypes.data)
    return pre, chains, euler


def srgb8_to_linear(rgb) -> tuple:
    """component_from_srgb8 (color.rs): f32 sRGB decode, used only for named palette constants."""
    out = []
    for c in rgb:
        f = np.float32(c) / np.float32(255.0)
        if f <= np.float32(0.04045):
            out.append(float(np.float32(f * np.float32(25.0 / 323.0))))
        else:
            x = np.float32(np.float32(200.0) * f + np.float32(11.0)) / np.float32(211.0)
            out.append(float(np.float32(float(x) ** float(np.float32(12.0 / 5.0)))))
    return tuple(out)


# ------------------------------------------------------------------------------------------------
# SpaceRaytracer / RtRenderer
# ------------------------------------------------------------------------------------------------
class Context:
    _default = None

    def __init__(self, device_id: int = -1):
        lib = load_library()
        self.handle = C.c_void_p()
        _check(lib.aicb_ctx_create(device_id, C.byref(self.handle)))

    @classmethod
    def default(cls) -> "Context":
        if cls._default is None:
            cls._default = Context(-1)
        return cls._default

    def close(self):
        if self.handle:
            load_library().aicb_ctx_destroy(self.handle)
            self.handle = C.c_void_p()


@dataclasses.dataclass
class RenderInfo:
    cubes_traced: int
    rays: int
    algorithmic_bytes: int
    counters: tuple
    kernel_ms: float
    flaws: int
    stage_ms: tuple = (0.0, 0.0, 0.0, 0.0)   # ray generation, marching, shading, encode (first chunk)

    @staticmethod
    def from_abi(i: abi.RenderInfo) -> "RenderInfo":
        return RenderInfo(int(i.cubes_traced), int(i.rays), int(i.algorithmic_bytes), tuple(int(c) for c in i.counters),
                          float(i.kernel_ms), int(i.flaws), tuple(float(v) for v in i.stage_ms))


@dataclasses.dataclass
class Rendering:
    """headless.rs:52-67"""
    size: tuple
    data: np.ndarray  # [H, W, 4] uint8 sRGB RGBA
    flaws: int
    info: RenderInfo


class SpaceRaytracer:
    """SpaceRaytracer<()> (sr.rs:51): device-resident snapshot of a Space + graphics options."""

    def __init__(self, space: Space, graphics_options: GraphicsOptions, ctx: Optional[Context] = None):
        self.ctx = ctx or Context.default()
        self.graphics_options = graphics_options.repair()
        self.space = space
        desc, keep = space.to_desc()
        self.handle = C.c_void_p()
        _check(load_library().aicb_scene_create(self.ctx.handle, C.byref(desc), C.byref(self.handle)))
        del keep

    def close(self):
        if self.handle:
            load_library().aicb_scene_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_bytes(self) -> int:
        return int(load_library().aicb_scene_device_bytes(self.handle))

    def trace_rays(self, origin_dir: np.ndarray, include_sky: bool = True, want_depth=False, want_hit=False,
                   want_steps=False):
        """SpaceRaytracer::trace_ray (sr.rs:113-120) over a batch: returns dict of arrays."""
        od = np.ascontiguousarray(origin_dir, dtype=np.float64).reshape(-1, 6)
        n = od.shape[0]
        cb = np.empty((n, 4), dtype=np.float32)
        depth = np.empty(n, dtype=np.float64) if want_depth else None
        hit = np.empty((n, 8), dtype=np.int32) if want_hit else None
        steps = np.empty(n, dtype=np.uint32) if want_steps else None
        info = abi.RenderInfo()
        opt = self.graphics_options.to_abi(include_sky)
        _check(load_library().aicb_trace_rays(self.handle, od.ctypes.data, n, C.byref(opt), cb.ctypes.data,
                                              depth.ctypes.data if want_depth else None,
                                              hit.ctypes.data if want_hit else None,
                                              steps.ctypes.data if want_steps else None, C.byref(info)))
        return {"colorbuf": cb, "depth": depth, "hit": hit, "steps": steps, "info": RenderInfo.from_abi(info)}

    def update_cubes(self, cubes: np.ndarray, block_ids: np.ndarray, light: Optional[np.ndarray] = None):
        c = np.ascontiguousarray(cubes, dtype=np.int32).reshape(-1, 3)
        ids = np.ascontiguousarray(block_ids, dtype=np.uint16)
        lt = None if light is None else np.ascontiguousarray(light, dtype=np.uint8).reshape(-1, 4)
        _check(load_library().aicb_scene_update_cubes(self.handle, c.ctypes.data, ids.ctypes.data,
                                                      lt.ctypes.data if lt is not None else None, c.shape[0]))

    def update_blocks(self, indices, blocks):
        """SpaceChange::BlockEvaluation / BlockIndex: new definitions for existing block indices."""
        idx = np.ascontiguousarray(indices, dtype=np.uint16)
        arr = (abi.BlockDesc * len(blocks))()
        for i, b in enumerate(blocks):
            fill_block_desc(arr[i], b)
        _check(load_library().aicb_scene_update_blocks(self.handle, idx.ctypes.data, arr, len(blocks)))

    # ---- light propagation (space::light; SURVEY 8(a) L1-L4) ----
    def light_fast_evaluate(self):
        """LightStorage::fast_evaluate_light (updater.rs:537-582)"""
        _check(load_library().aicb_light_fast_evaluate(self.handle))

    def light_compute(self, cubes: np.ndarray) -> np.ndarray:
        """LightStorage::compute_light (updater.rs:368-418) for explicit cubes; returns texels [n,4]."""
        c = np.ascontiguousarray(cubes, dtype=np.int32).reshape(-1, 3)
        out = np.zeros((c.shape[0], 4), dtype=np.uint8)
        _check(load_library().aicb_light_compute(self.handle, c.ctypes.data, c.shape[0], out.ctypes.data))
        return out

    def light_evaluate(self, epsilon: int = 0):
        """Mutation::evaluate_light (space.rs:1496-1527) -> (updates, max_difference, chart_node_visits)"""
        n, md, nv = C.c_uint64(0), C.c_uint8(0), C.c_uint64(0)
        _check(load_library().aicb_light_evaluate(self.handle, epsilon, C.byref(n), C.byref(md), C.byref(nv)))
        return int(n.value), int(md.value), int(nv.value)

    def light_edit_and_propagate(self, cubes: np.ndarray, block_ids: np.ndarray, epsilon: int = 0):
        """Mutation::set x n + evaluate_light(epsilon) -> (updates, max_difference)"""
        c = np.ascontiguousarray(cubes, dtype=np.int32).reshape(-1, 3)
        ids = np.ascontiguousarray(block_ids, dtype=np.uint16)
        n, md = C.c_uint64(0), C.c_uint8(0)
        _check(load_library().aicb_light_edit_and_propagate(self.handle, c.ctypes.data, ids.ctypes.data, c.shape[0], epsilon,
                                                            C.byref(n), C.byref(md)))
        return int(n.value), int(md.value)

    def light_stats(self) -> dict:
        """Counters of the last propagation: cube updates, chart node visits, rounds, device seconds."""
        out = (C.c_uint64 * 4)()
        _check(load_library().aicb_light_stats(self.handle, out))
        return {"cube_updates": int(out[0]), "chart_node_visits": int(out[1]), "rounds": int(out[2]),
                "device_seconds": int(out[3]) * 1e-6}

    def light_download(self) -> np.ndarray:
        out = np.zeros(self.space.size + (4,), dtype=np.uint8)
        _check(load_library().aicb_light_download(self.handle, out.ctypes.data, out.size // 4))
        return out

    def upload_light(self, light: np.ndarray):
        lt = np.ascontiguousarray(light, dtype=np.uint8).reshape(-1, 4)
        _check(load_library().aicb_scene_upload_light(self.handle, lt.ctypes.data, lt.shape[0]))

    def light_step(self, cubes=None, block_ids=None, epsilon: int = 0, max_updates: Optional[int] = None,
                   budget_us: Optional[float] = None) -> dict:
        """Mutation::set x n, then update_light_from_queue(budget) (updater.rs:181-291): relax until nothing above
        epsilon is queued, `max_updates` cube updates are done or `budget_us` device microseconds are used up (None:
        no limit).  -> update_count, queue_count, chart_node_visits, rounds, max_update_difference,
        max_queue_priority, device_ms."""
        return _light_step(load_library().aicb_light_step, self.handle, cubes, block_ids, epsilon, max_updates, budget_us)

    def light_track_changes(self, enable: bool = True):
        """Record the current light as the baseline of light_take_changes (or stop tracking)."""
        _check(load_library().aicb_light_track_changes(self.handle, 1 if enable else 0))

    def light_take_changes(self):
        """SpaceChange::CubeLight since the last take: (cubes [n,3] int32, texels [n,4] uint8) in index order."""
        return _light_take_changes(load_library().aicb_light_take_changes, self.handle)


NO_LIMIT = (1 << 64) - 1   # aicb_light_step's max_updates without a limit (UINT64_MAX)


def _light_step(fn, handle, cubes, block_ids, epsilon, max_updates, budget_us) -> dict:
    """aicb_light_step / aicb_group_light_step -> LightUpdatesInfo as a dict."""
    if cubes is None:
        c, ids = np.zeros((0, 3), dtype=np.int32), np.zeros(0, dtype=np.uint16)
    else:
        c = np.ascontiguousarray(cubes, dtype=np.int32).reshape(-1, 3)
        ids = np.ascontiguousarray(block_ids, dtype=np.uint16)
        if ids.shape != (c.shape[0],):
            raise ValueError("one block id per cube")
    info = abi.LightUpdates()
    _check(fn(handle, c.ctypes.data if c.shape[0] else None, ids.ctypes.data if c.shape[0] else None, c.shape[0], epsilon,
              NO_LIMIT if max_updates is None else int(max_updates), -1.0 if budget_us is None else float(budget_us),
              C.byref(info)))
    return {"update_count": int(info.update_count), "queue_count": int(info.queue_count),
            "chart_node_visits": int(info.chart_node_visits), "rounds": int(info.rounds),
            "max_update_difference": int(info.max_update_difference),
            "max_queue_priority": int(info.max_queue_priority), "device_ms": float(info.device_ms)}


def _light_take_changes(fn, handle):
    """The count query, then the take: (cubes [n,3] int32 world coordinates, texels [n,4] uint8)."""
    n = C.c_size_t(0)
    while True:
        _check(fn(handle, None, None, 0, C.byref(n)))
        cubes = np.zeros((n.value, 3), dtype=np.int32)
        texels = np.zeros((n.value, 4), dtype=np.uint8)
        if n.value == 0:
            return cubes, texels
        want = n.value
        _check(fn(handle, cubes.ctypes.data, texels.ctypes.data, want, C.byref(n)))
        if n.value <= want:    # (a light call between the two may have changed more cubes: ask again)
            return cubes[:n.value], texels[:n.value]


NO_WORLD_TO_SHOW_SRGB8 = (0xBC, 0xBC, 0xBC, 0xFF)   # content/palette.rs:76


def render_layers(world=None, ui=None, backdrop=None, no_world=None) -> "Rendering":
    """RtRenderer::draw_rgba through every layer (renderer.rs:282-308, 454-478).
    world / ui = (SpaceRaytracer, Camera, GraphicsOptions) or None; backdrop / no_world = linear RGBA or None."""
    lead = world if world else ui
    cam = lead[1]
    w, h = cam.data.fb_width, cam.data.fb_height
    keep = []

    def layer(l):
        if not l:
            return None
        o = l[2].to_abi(True)
        keep.append(o)
        s = abi.Layer(l[0].handle, C.pointer(l[1].data), C.pointer(o))
        keep.append(s)
        return C.byref(s)

    out = np.zeros((h, w, 4), dtype=np.uint8)
    info = abi.RenderInfo()
    b = np.array(backdrop, dtype=np.float32) if backdrop is not None else None
    nw = np.array(no_world, dtype=np.float32) if no_world is not None else None
    _check(load_library().aicb_render_layers_srgb8(layer(world), layer(ui), b.ctypes.data if b is not None else None,
                                                   nw.ctypes.data if nw is not None else None, out.ctypes.data, w * h,
                                                   C.byref(info)))
    return Rendering((w, h), out, int(info.flaws), RenderInfo.from_abi(info))


def render_orthographic(rt: "SpaceRaytracer", resolution: int = 32) -> "Rendering":
    """raytracer::ortho::render_orthographic (ortho.rs:30-84): the five-view pixel-perfect image of the whole Space."""
    w, h = C.c_uint32(0), C.c_uint32(0)
    _check(load_library().aicb_ortho_image_size(rt.handle, resolution, C.byref(w), C.byref(h)))
    out = np.zeros((h.value, w.value, 4), dtype=np.uint8)
    info = abi.RenderInfo()
    _check(load_library().aicb_render_orthographic(rt.handle, resolution, out.ctypes.data, w.value * h.value, C.byref(info)))
    return Rendering((w.value, h.value), out, int(info.flaws), RenderInfo.from_abi(info))


def print_space(space: "Space", direction, block_chars: dict, rt: "SpaceRaytracer" = None) -> list:
    """raytracer::print_space (text.rs:139-180): the 80 x 40 character image of a Space seen from `direction`, one
    string per row.  `block_chars` maps a block index to its character (what D::from_block gives each block)."""
    opts = GraphicsOptions()
    cam = Camera(opts, Viewport((40.0, 40.0), (80, 40)))
    center = [space.lower[a] + space.size[a] / 2.0 for a in range(3)]
    cam.look_at_y_up(eye_for_look_at(space.lower, space.size, direction), center)
    rt = rt or SpaceRaytracer(space, opts)
    o = opts.to_abi(True)
    out = np.zeros(80 * 40, dtype=np.int32)
    _check(load_library().aicb_render_text(rt.handle, C.byref(cam.data), C.byref(o), out.ctypes.data, out.size, None))
    special = {abi.TEXT_ENTERED_SPACE: " ", abi.TEXT_EMPTY: ".", abi.TEXT_INCOMPLETE: "X"}
    return ["".join(special[v] if v < 0 else block_chars[int(v)] for v in out[r * 80:(r + 1) * 80]) for r in range(40)]


class DeviceGroup:
    """Several GPUs driven from this one process through the C ABI (csrc/group.cu): scene replicated, frame cut into
    interleaved row strips, pixels stored straight into device 0's frame over NVLink.  Light propagation runs on the
    whole group, each member relaxing its own slab of the volume (csrc/light.cu); the light methods are
    SpaceRaytracer's."""

    def __init__(self, device_ids):
        ids = (C.c_int * len(device_ids))(*[int(d) for d in device_ids])
        h = C.c_void_p()
        _check(load_library().aicb_group_create(ids, len(device_ids), C.byref(h)))
        self.handle = h
        self.size = len(device_ids)
        self.scene = None
        self.space = None

    def update(self, space: "Space"):
        if self.scene:
            load_library().aicb_group_scene_destroy(self.scene)
            self.scene = None
        desc, keep = space.to_desc()
        h = C.c_void_p()
        _check(load_library().aicb_group_scene_create(self.handle, C.byref(desc), C.byref(h)))
        del keep
        self.scene = h
        self.space = space

    def update_cubes(self, cubes: np.ndarray, block_ids: np.ndarray, light: Optional[np.ndarray] = None):
        c = np.ascontiguousarray(cubes, dtype=np.int32).reshape(-1, 3)
        ids = np.ascontiguousarray(block_ids, dtype=np.uint16)
        lt = None if light is None else np.ascontiguousarray(light, dtype=np.uint8).reshape(-1, 4)
        _check(load_library().aicb_group_scene_update_cubes(self.scene, c.ctypes.data, ids.ctypes.data,
                                                            lt.ctypes.data if lt is not None else None, c.shape[0]))

    def update_blocks(self, indices, blocks):
        idx = np.ascontiguousarray(indices, dtype=np.uint16)
        arr = (abi.BlockDesc * len(blocks))()
        for i, b in enumerate(blocks):
            fill_block_desc(arr[i], b)
        _check(load_library().aicb_group_scene_update_blocks(self.scene, idx.ctypes.data, arr, len(blocks)))

    def upload_light(self, light: np.ndarray):
        lt = np.ascontiguousarray(light, dtype=np.uint8).reshape(-1, 4)
        _check(load_library().aicb_group_scene_upload_light(self.scene, lt.ctypes.data, lt.shape[0]))

    def light_fast_evaluate(self):
        _check(load_library().aicb_group_light_fast_evaluate(self.scene))

    def light_evaluate(self, epsilon: int = 0):
        """-> (updates, max_difference, chart_node_visits), summed over the members"""
        n, md, nv = C.c_uint64(0), C.c_uint8(0), C.c_uint64(0)
        _check(load_library().aicb_group_light_evaluate(self.scene, epsilon, C.byref(n), C.byref(md), C.byref(nv)))
        return int(n.value), int(md.value), int(nv.value)

    def light_edit_and_propagate(self, cubes: np.ndarray, block_ids: np.ndarray, epsilon: int = 0):
        """-> (updates, max_difference)"""
        c = np.ascontiguousarray(cubes, dtype=np.int32).reshape(-1, 3)
        ids = np.ascontiguousarray(block_ids, dtype=np.uint16)
        n, md = C.c_uint64(0), C.c_uint8(0)
        _check(load_library().aicb_group_light_edit_and_propagate(self.scene, c.ctypes.data, ids.ctypes.data, c.shape[0],
                                                                  epsilon, C.byref(n), C.byref(md)))
        return int(n.value), int(md.value)

    def light_download(self, member: int = 0) -> np.ndarray:
        """The light replica of one member (a position in the group, not a device id)."""
        out = np.zeros(self.space.size + (4,), dtype=np.uint8)
        _check(load_library().aicb_group_light_download(self.scene, member, out.ctypes.data, out.size // 4))
        return out

    def light_stats(self, member: Optional[int] = None) -> dict:
        """Counters of the last propagation: the group's (updates and visits summed, the slowest member's time) or
        one member's own."""
        out = (C.c_uint64 * 4)()
        _check(load_library().aicb_group_light_stats(self.scene, -1 if member is None else member, out))
        return {"cube_updates": int(out[0]), "chart_node_visits": int(out[1]), "rounds": int(out[2]),
                "device_seconds": int(out[3]) * 1e-6}

    def light_step(self, cubes=None, block_ids=None, epsilon: int = 0, max_updates: Optional[int] = None,
                   budget_us: Optional[float] = None) -> dict:
        """SpaceRaytracer.light_step on the group: counts summed over the members, the slowest member's time."""
        return _light_step(load_library().aicb_group_light_step, self.scene, cubes, block_ids, epsilon, max_updates,
                           budget_us)

    def light_track_changes(self, enable: bool = True):
        _check(load_library().aicb_group_light_track_changes(self.scene, 1 if enable else 0))

    def light_take_changes(self):
        """The changes of member 0's replica (every replica holds the same light)."""
        return _light_take_changes(load_library().aicb_group_light_take_changes, self.scene)

    def draw(self, camera: "Camera", options: "GraphicsOptions") -> "Rendering":
        w, h = camera.data.fb_width, camera.data.fb_height
        out = np.zeros((h, w, 4), dtype=np.uint8)
        info = abi.RenderInfo()
        o = options.to_abi(True)
        _check(load_library().aicb_group_render_srgb8(self.scene, C.byref(camera.data), C.byref(o), out.ctypes.data, w * h,
                                                     C.byref(info)))
        return Rendering((w, h), out, int(info.flaws), RenderInfo.from_abi(info))

    def close(self):
        if self.scene:
            load_library().aicb_group_scene_destroy(self.scene)
            self.scene = None
        if self.handle:
            load_library().aicb_group_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _shard_abi(shard):
    if shard is None:
        return None
    s = abi.Shard()
    s.strip_rows, s.index, s.count = shard
    return s


class RtRenderer:
    """RtRenderer<()> + impl HeadlessRenderer (renderer.rs:35, 338-355; headless.rs:17-44).

    update(): snapshot the Space onto the GPU (== SpaceRaytracer::new / UpdatingSpaceRaytracer).
    draw(): trace every pixel on the GPU and return a Rendering (== draw_rgba)."""

    def __init__(self, camera: Camera, ctx: Optional[Context] = None):
        self.camera = camera
        self.ctx = ctx or Context.default()
        self.rt: Optional[SpaceRaytracer] = None

    def update(self, space: Space):
        if self.rt is not None:
            self.rt.close()
        self.rt = SpaceRaytracer(space, self.camera.options, self.ctx)

    def _require(self) -> SpaceRaytracer:
        if self.rt is None:
            raise AicbError(abi.ERR_INVALID, "draw() before update()")
        return self.rt

    def pixel_count(self, shard=None) -> int:
        s = _shard_abi(shard)
        return int(load_library().aicb_shard_pixel_count(C.byref(self.camera.data), C.byref(s) if s else None))

    def draw(self, info_text: str = "", shard=None) -> Rendering:
        rt = self._require()
        n = self.pixel_count(shard)
        w = self.camera.data.fb_width
        out = np.empty((n, 4), dtype=np.uint8)
        info = abi.RenderInfo()
        opt = rt.graphics_options.to_abi(True)
        s = _shard_abi(shard)
        _check(load_library().aicb_render_srgb8(rt.handle, C.byref(self.camera.data), C.byref(opt),
                                                C.byref(s) if s else None, out.ctypes.data, n, C.byref(info)))
        h = n // w if w else 0
        return Rendering((w, h), out.reshape(h, w, 4) if w else out.reshape(0, 0, 4), int(info.flaws),
                         RenderInfo.from_abi(info))

    draw_rgba = draw

    def draw_rgba16f(self, shard=None):
        """The per-pixel colour raytrace_to_texture uploads (raytrace_to_texture.rs:645-661): premultiplied RGBA,
        exposure applied, as float16 [h, w, 4]."""
        rt = self._require()
        n = self.pixel_count(shard)
        w = self.camera.data.fb_width
        out = np.empty((n, 4), dtype=np.float16)
        info = abi.RenderInfo()
        opt = rt.graphics_options.to_abi(True)
        s = _shard_abi(shard)
        _check(load_library().aicb_render_rgba16f(rt.handle, C.byref(self.camera.data), C.byref(opt),
                                                  C.byref(s) if s else None, out.ctypes.data, n, C.byref(info)))
        h = n // w if w else 0
        return out.reshape(h, w, 4) if w else out.reshape(0, 0, 4)

    def draw_colorbuf(self, shard=None, want_depth=True, want_hit=True, want_steps=True):
        """RtRenderer::draw::<ColorBuf> (+DepthBuf, +Position) (renderer.rs:183-220)."""
        rt = self._require()
        n = self.pixel_count(shard)
        cb = np.empty((n, 4), dtype=np.float32)
        depth = np.empty(n, dtype=np.float64) if want_depth else None
        hit = np.empty((n, 8), dtype=np.int32) if want_hit else None
        steps = np.empty(n, dtype=np.uint32) if want_steps else None
        info = abi.RenderInfo()
        opt = rt.graphics_options.to_abi(True)
        s = _shard_abi(shard)
        _check(load_library().aicb_render_colorbuf(rt.handle, C.byref(self.camera.data), C.byref(opt),
                                                   C.byref(s) if s else None, cb.ctypes.data,
                                                   depth.ctypes.data if want_depth else None,
                                                   hit.ctypes.data if want_hit else None,
                                                   steps.ctypes.data if want_steps else None, n, C.byref(info)))
        return {"colorbuf": cb, "depth": depth, "hit": hit, "steps": steps, "info": RenderInfo.from_abi(info)}


HeadlessRenderer = RtRenderer
