"""Host-side mirror of `GaussianSplattingRasterizer` (util/gaussian_splatting_rasterizer.gd) on top of libgsr.

Same public surface as the GDScript class -- `_init(point_cloud, output_texture_size, render_texture,
camera)`, `init_gpu()`, `rasterize()`, `texture_size` setter, `update_camera_matrices() -> bool`,
`get_splat_position(Vector2i) -> Vector3`, `cleanup_gpu()`, the knobs `should_enable_heatmap`,
`render_scale`, `model_scale`, `basis_override`, `is_loaded`, `num_splats_loaded` -- so the parity tests read
like the reference's own call sites (main.gd:121-152).  Everything GPU-side goes through the C-ABI.

`render_texture` here is a `RenderTexture` holder: after `rasterize()` it exposes the device pointer of the
RGBA32F frame (the Texture2DRD's RID in the reference) and `read()` copies it to a numpy array.
"""
from __future__ import annotations

import ctypes as C
import math
import time as _time

import numpy as np

from . import _lib
from .camera import Camera3D, pack_camera_push_constants, transform_to_projection
from .ply_file import PlyFile, load_gaussian_splats

TILE_SIZE = 16            # rasterizer.gd:4
WORKGROUP_SIZE = 512      # rasterizer.gd:5
RADIX = 256               # rasterizer.gd:6
PARTITION_DIVISION = 8    # rasterizer.gd:7
PARTITION_SIZE = PARTITION_DIVISION * WORKGROUP_SIZE

VECTOR3_INF = np.array([np.inf, np.inf, np.inf], dtype=np.float32)


class RenderTexture:
    """Stand-in for Texture2DRD: holds the device pointer of the frame."""

    def __init__(self):
        self.device_ptr = 0
        self.size = (0, 0)
        self._owner = None

    def read(self) -> np.ndarray:
        if self._owner is None:
            raise RuntimeError("render texture is not bound to a rasterizer")
        return self._owner.read_framebuffer()


class GaussianSplattingRasterizer:
    def __init__(self, point_cloud: PlyFile, output_texture_size, render_texture: RenderTexture | None, camera: Camera3D,
                 device: int = 0, flags: int = 0, dup_capacity_factor: int = 10, clock=None):
        self.should_enable_heatmap = [False]
        self.render_scale = [1.0]
        self.model_scale = [1.0]
        self.should_terminate_thread = [False]
        self.num_splats_loaded = [0]
        self.basis_override = np.eye(3, dtype=np.float32)  # rows = basis columns x, y, z
        self.is_loaded = False
        self.loaded_callbacks = []  # signal `loaded`
        self._ctx = C.c_void_p(None)
        self._device, self._flags, self._factor = device, flags, dup_capacity_factor
        self._clock = clock or (lambda: _time.monotonic())
        self._t0 = self._clock()
        self.tile_dims = (0, 0)
        self._texture_size = (1, 1)
        self.point_cloud = point_cloud
        self.texture_size = output_texture_size
        self.render_texture = render_texture or RenderTexture()
        self.camera = camera
        self.camera_projection = None
        self.camera_transform = None
        self.camera_push_constants = None
        self._pinned = None
        self._num_views = 1

    # ---- texture_size setter (rasterizer.gd:26-48) ----
    @property
    def texture_size(self):
        return self._texture_size

    @texture_size.setter
    def texture_size(self, value):
        s = self.render_scale[0]
        w, h = max(1, int(value[0] * s)), max(1, int(value[1] * s))
        self._texture_size = (w, h)
        self.tile_dims = ((w + TILE_SIZE - 1) // TILE_SIZE, (h + TILE_SIZE - 1) // TILE_SIZE)
        if self._ctx:
            _lib.check(_lib.lib().gsr_resize(self._ctx, w, h), "gsr_resize")
            self._bind_texture()

    def _bind_texture(self):
        self.render_texture.device_ptr = int(_lib.lib().gsr_framebuffer_device_ptr(self._ctx) or 0)
        self.render_texture.size = self._texture_size
        self.render_texture._owner = self

    def ticks(self) -> float:
        """Time.get_ticks_msec()*1e-3 (rasterizer.gd:126, ply_file.gd:40)."""
        return self._clock() - self._t0

    # ---- init_gpu (rasterizer.gd:65-114) ----
    def init_gpu(self, load: bool = True, device_ingest: bool = False) -> None:
        """load=False creates the context only; the caller then streams splats in with `upload_splats` / `upload_ply_raw`.
        device_ingest=True runs the per-splat preprocessing of ply_file.gd:44-69 on the GPU instead of in numpy."""
        assert self.render_texture is not None, "An output Texture2DRD must be set!"
        L = _lib.lib()
        cfg = _lib.GsrConfig(self._device, self._flags, max(1, self.point_cloud.size), self._factor, 0)
        _lib.check(L.gsr_create(C.byref(cfg), C.byref(self._ctx)), "gsr_create")
        w, h = self._texture_size
        _lib.check(L.gsr_resize(self._ctx, w, h), "gsr_resize")
        self._bind_texture()
        self.should_terminate_thread[0] = False
        self.num_splats_loaded[0] = 0
        if not load:
            return
        # the reference starts a loader thread (:114); here the load runs inline, chunk by chunk
        stride = max(1, self.point_cloud.size // 1000)
        if device_ingest:
            table, n, i = self.point_cloud.table, self.point_cloud.size, 0
            while i * stride < n and not self.should_terminate_thread[0]:
                lo, hi = i * stride, min(n, (i + 1) * stride)
                self.upload_ply_raw(table[lo:hi], lo, self.ticks())
                i += 1
            self._emit_loaded()
            return
        load_gaussian_splats(self.point_cloud, stride, self._upload, self.should_terminate_thread, self.num_splats_loaded,
                             self._emit_loaded, clock=self.ticks)

    def _upload(self, first: int, block60: np.ndarray) -> None:
        block60 = np.ascontiguousarray(block60, dtype=np.float32)
        _lib.check(_lib.lib().gsr_upload_splats_aos(self._ctx, block60.ctypes.data_as(C.POINTER(C.c_float)), first,
                                                    block60.shape[0]), "gsr_upload_splats_aos")

    def upload_splats(self, splat60: np.ndarray, first: int = 0) -> None:
        """Direct upload of pre-swizzled 60-float structs (used by the bench for large scenes)."""
        if not self._ctx:
            raise RuntimeError("init_gpu() first")
        self._upload(first, splat60)
        self.num_splats_loaded[0] = max(self.num_splats_loaded[0], first + splat60.shape[0])

    def upload_ply_raw(self, table: np.ndarray, first: int = 0, creation_time: float = 0.0) -> None:
        """Device-side ingest (scope row f1): raw (m, nprops) PLY vertices -> SoA planes, preprocessing on the GPU."""
        if not self._ctx:
            raise RuntimeError("init_gpu() first")
        t = np.ascontiguousarray(table, dtype=np.float32)
        _lib.check(_lib.lib().gsr_upload_ply_raw(self._ctx, t.ctypes.data_as(C.POINTER(C.c_float)), t.shape[1], first, t.shape[0],
                                                 float(creation_time)), "gsr_upload_ply_raw")
        self.num_splats_loaded[0] = max(self.num_splats_loaded[0], first + t.shape[0])

    def _emit_loaded(self):
        self.is_loaded = True
        for cb in self.loaded_callbacks:
            cb()

    def set_framebuffer_external(self, device_ptr: int) -> None:
        _lib.check(_lib.lib().gsr_set_framebuffer_external(self._ctx, C.c_void_p(device_ptr)), "gsr_set_framebuffer_external")
        self._bind_texture()

    def render_raw(self, vp32: np.ndarray, uniforms32: bytes, heatmap: float = 0.0, host_ptr: int | None = None,
                   asynchronous: bool = True, rgb_only: bool = False, out_format: int | None = None) -> None:
        """rasterize() with pre-packed push constants / uniform block (bench hot loop).  out_format: GSR_OUT_* of the host frame
        (| GSR_OUT_SRGB_TO_LINEAR); rgb_only is shorthand for GSR_OUT_RGB32F (alpha is constant 1.0 and stays on the device)."""
        L = _lib.lib()
        fmt = _lib.GSR_OUT_RGB32F if (rgb_only and out_format is None) else (out_format or _lib.GSR_OUT_RGBA32F)
        vpp = vp32.ctypes.data_as(C.POINTER(C.c_float))
        hp = None if host_ptr is None else C.c_void_p(host_ptr)
        if not asynchronous:
            assert fmt == _lib.GSR_OUT_RGBA32F, "gsr_render returns the RGBA32F frame"
            _lib.check(L.gsr_render(self._ctx, vpp, uniforms32, float(heatmap), hp), "gsr_render")
        else:
            _lib.check(L.gsr_render_async_fmt(self._ctx, vpp, uniforms32, float(heatmap), hp, int(fmt)), "gsr_render_async_fmt")

    def debug_pipeline(self, overlap: int) -> None:
        """gsr_debug_pipeline: 1 / 0 = front/back overlap of consecutive frames on / off, -1 = automatic (include/gsr.h)."""
        _lib.check(_lib.lib().gsr_debug_pipeline(self._ctx, int(overlap)), "gsr_debug_pipeline")

    def set_stream(self, cuda_stream: int) -> None:
        _lib.check(_lib.lib().gsr_set_stream(self._ctx, C.c_void_p(cuda_stream)), "gsr_set_stream")

    def set_band(self, row_begin: int, row_end: int) -> None:
        _lib.check(_lib.lib().gsr_set_band(self._ctx, row_begin, row_end), "gsr_set_band")

    def set_row_interleave(self, rem: int, mod: int) -> None:
        """Own the tile rows with row % mod == rem (balanced multi-GPU sharding, fast mode; see include/gsr.h)."""
        _lib.check(_lib.lib().gsr_set_row_interleave(self._ctx, rem, mod), "gsr_set_row_interleave")

    def band_sync_word_ptr(self) -> int:
        return int(_lib.lib().gsr_band_sync_word(self._ctx) or 0)

    def band_fixup(self) -> None:
        _lib.check(_lib.lib().gsr_band_fixup(self._ctx), "gsr_band_fixup")

    def cleanup_gpu(self) -> None:  # rasterizer.gd:116-120
        self.should_terminate_thread[0] = True
        if self._ctx:
            _lib.lib().gsr_destroy(self._ctx)
            self._ctx = C.c_void_p(None)
        if self.render_texture:
            self.render_texture.device_ptr = 0

    # ---- rasterize (rasterizer.gd:122-160) ----
    def uniforms_bytes(self, time: float | None = None) -> bytes:
        cam_pos = self.basis_override.T @ np.asarray(self.camera.global_position, dtype=np.float32)
        w, h = self._texture_size
        t = self.ticks() if time is None else time
        buf = np.zeros(8, dtype=np.float32)
        buf[0], buf[1], buf[2], buf[3] = -cam_pos[0], -cam_pos[1], cam_pos[2], self.model_scale[0]
        buf[6] = t
        raw = bytearray(buf.tobytes())
        raw[16:24] = np.array([w, h], dtype=np.int32).tobytes()
        return bytes(raw)

    def rasterize(self, time: float | None = None, out_host: np.ndarray | None = None, asynchronous: bool = False) -> None:
        if not self._ctx:
            self.init_gpu()
        if self.camera_push_constants is None:
            self.update_camera_matrices()
        u = self.uniforms_bytes(time)
        vp = self.camera_push_constants
        fn = _lib.lib().gsr_render_async if asynchronous else _lib.lib().gsr_render
        outp = None if out_host is None else C.c_void_p(out_host.ctypes.data)
        _lib.check(fn(self._ctx, vp.ctypes.data_as(C.POINTER(C.c_float)), u, float(self.should_enable_heatmap[0]), outp),
                   "gsr_render")

    # ---- multiview (stereo / XR): K cameras of the same splats in one frame, K layers (include/gsr.h gsr_set_views) ----
    @property
    def num_views(self) -> int:
        return self._num_views

    def set_views(self, k: int) -> None:
        if not self._ctx:
            self.init_gpu(load=False)
        _lib.check(_lib.lib().gsr_set_views(self._ctx, int(k)), "gsr_set_views")
        self._num_views = int(k)
        self._bind_texture()

    def view_push_constants(self, camera: Camera3D, projection: np.ndarray | None = None) -> np.ndarray:
        """The 128-byte push constant of one view (update_camera_matrices with basis_override applied); `projection` overrides the
        camera's own perspective, e.g. with an off-axis camera.frustum for an XR eye."""
        cam = np.asarray(camera.get_camera_transform(), dtype=np.float32).reshape(4, 4)
        bo = self.basis_override
        if np.array_equal(bo, np.eye(3, dtype=np.float32)):
            view = cam.reshape(16)
        else:
            B = bo.T.astype(np.float32)
            view = transform_to_projection((B @ cam[:3, :3].T).T.astype(np.float32), (B @ cam[3, :3]).astype(np.float32))
        proj = camera.get_camera_projection() if projection is None else projection
        return pack_camera_push_constants(view, np.asarray(proj, dtype=np.float32))

    def rasterize_views(self, cameras, time: float | None = None, out_host: np.ndarray | None = None, asynchronous: bool = False,
                        projections=None) -> None:
        """rasterize() for K = num_views cameras at once: layer v of the frame is camera v's image, bit-identical to a single-view
        rasterize() of that camera.  out_host: None, or (K, H, W, 4) float32 (synchronous: filled on return; asynchronous: page-locked,
        filled once the copy stream is done, see sync())."""
        cameras = list(cameras)
        if len(cameras) != self._num_views:
            raise ValueError(f"{len(cameras)} cameras for a context with {self._num_views} views (set_views)")
        projections = list(projections) if projections is not None else [None] * len(cameras)
        vp = np.ascontiguousarray(np.concatenate([self.view_push_constants(c, p) for c, p in zip(cameras, projections)]), dtype=np.float32)
        t = self.ticks() if time is None else time
        saved = self.camera
        try:
            ub = b""
            for c in cameras:
                self.camera = c
                ub += self.uniforms_bytes(t)
        finally:
            self.camera = saved
        L = _lib.lib()
        outp = None if out_host is None else C.c_void_p(out_host.ctypes.data)
        heat = float(self.should_enable_heatmap[0])
        if asynchronous:
            _lib.check(L.gsr_render_views_async(self._ctx, vp.ctypes.data_as(C.POINTER(C.c_float)), ub, heat, outp, _lib.GSR_OUT_RGBA32F),
                       "gsr_render_views_async")
        else:
            _lib.check(L.gsr_render_views(self._ctx, vp.ctypes.data_as(C.POINTER(C.c_float)), ub, heat, outp), "gsr_render_views")

    def sync(self) -> None:
        _lib.check(_lib.lib().gsr_sync(self._ctx), "gsr_sync")

    def readback_async(self, host_ptr: int, rgb_only: bool = False, out_format: int | None = None) -> None:
        fmt = _lib.GSR_OUT_RGB32F if (rgb_only and out_format is None) else (out_format or _lib.GSR_OUT_RGBA32F)
        _lib.check(_lib.lib().gsr_readback_async(self._ctx, C.c_void_p(host_ptr), int(fmt)), "gsr_readback_async")

    def present_device(self, device_ptr: int, out_format: int = 0) -> None:
        """Converted copy of the last frame into caller-owned device memory (imported external image / torch tensor)."""
        _lib.check(_lib.lib().gsr_present_device(self._ctx, C.c_void_p(device_ptr), int(out_format)), "gsr_present_device")

    def peer_export(self) -> bytes:
        """Presenting rank: CUDA-IPC handles (128 bytes) of its two frames."""
        buf = (C.c_ubyte * 128)()
        _lib.check(_lib.lib().gsr_peer_export_framebuffers(self._ctx, buf), "gsr_peer_export_framebuffers")
        return bytes(buf)

    def peer_import(self, handles: bytes) -> None:
        buf = (C.c_ubyte * 128).from_buffer_copy(handles)
        _lib.check(_lib.lib().gsr_peer_import_framebuffers(self._ctx, buf), "gsr_peer_import_framebuffers")

    # ---- multi-GPU shard group (include/gsr.h gsr_group_*): NCCL-free frame path over NVLink peer memory ----
    def group_export(self) -> bytes:
        buf = (C.c_ubyte * _lib.GSR_GROUP_BLOB_BYTES)()
        _lib.check(_lib.lib().gsr_group_export(self._ctx, buf), "gsr_group_export")
        return bytes(buf)

    def group_attach(self, rank: int, world: int, blobs: bytes) -> None:
        assert len(blobs) == world * _lib.GSR_GROUP_BLOB_BYTES
        buf = (C.c_ubyte * len(blobs)).from_buffer_copy(blobs)
        _lib.check(_lib.lib().gsr_group_attach(self._ctx, int(rank), int(world), buf), "gsr_group_attach")

    def group_set_present(self, rows_local: bool) -> None:
        _lib.check(_lib.lib().gsr_group_set_present(self._ctx, int(bool(rows_local))), "gsr_group_set_present")

    def readback_rows_async(self, host_frame_ptr: int) -> None:
        _lib.check(_lib.lib().gsr_readback_rows_async(self._ctx, C.c_void_p(host_frame_ptr)), "gsr_readback_rows_async")

    def group_detach(self) -> None:
        _lib.check(_lib.lib().gsr_group_detach(self._ctx), "gsr_group_detach")

    def stream_join(self) -> None:
        """Make the render stream wait for the pipelined read-back copies enqueued so far."""
        _lib.check(_lib.lib().gsr_stream_join(self._ctx), "gsr_stream_join")

    # ---- get_splat_position (rasterizer.gd:162-171) ----
    def get_splat_position(self, screen_position) -> np.ndarray:
        s = self.render_scale[0]
        tile = (int(screen_position[0] * s) // TILE_SIZE, int(screen_position[1] * s) // TILE_SIZE)
        tile_id = tile[1] * self.tile_dims[0] + tile[0]
        out = (C.c_float * 4)()
        rc = _lib.lib().gsr_pick(self._ctx, tile_id & 0xFFFFFFFF, float(self.should_enable_heatmap[0]), out)
        if rc == _lib.GSR_ERR_STATE:   # no frame rasterized yet: the reference reads its zero-initialised buffer -> Vector3.INF
            return VECTOR3_INF.copy()
        _lib.check(rc, "gsr_pick")
        if out[3] == 0:
            return VECTOR3_INF.copy()
        v = np.array([-out[0], -out[1], out[2]], dtype=np.float32)
        return np.linalg.inv(self.basis_override.T.astype(np.float64)).astype(np.float32) @ v

    # ---- update_camera_matrices (rasterizer.gd:175-195) ----
    def update_camera_matrices(self) -> bool:
        cam = np.asarray(self.camera.get_camera_transform(), dtype=np.float32).reshape(4, 4)
        bo = self.basis_override  # rows are columns x,y,z
        if np.array_equal(bo, np.eye(3, dtype=np.float32)):
            view = cam.reshape(16)
        else:
            B = bo.T.astype(np.float32)  # matrix form
            basis = (B @ cam[:3, :3].T).T.astype(np.float32)
            origin = (B @ cam[3, :3]).astype(np.float32)
            view = transform_to_projection(basis, origin)
        proj = np.asarray(self.camera.get_camera_projection(), dtype=np.float32)
        if (self.camera_transform is None or not np.array_equal(view, self.camera_transform)
                or not np.array_equal(proj, self.camera_projection)):
            self.camera_transform, self.camera_projection = view, proj
            self.camera_push_constants = pack_camera_push_constants(view, proj)
            return True
        return False

    # ---- debug / stats (main.gd:93-119) ----
    def stats(self) -> _lib.GsrStats:
        st = _lib.GsrStats()
        _lib.check(_lib.lib().gsr_get_stats(self._ctx, C.byref(st)), "gsr_get_stats")
        return st

    def frame_history(self, max_frames: int = _lib.GSR_HISTORY_FRAMES) -> list:
        """Per-frame GPU timestamps + counters of the most recent frames (main.gd:106-119)."""
        n = min(max_frames, _lib.GSR_HISTORY_FRAMES)
        buf = (_lib.GsrFrameRecord * n)()
        got = C.c_uint32(0)
        _lib.check(_lib.lib().gsr_get_frame_history(self._ctx, n, buf, C.byref(got)), "gsr_get_frame_history")
        return [buf[i] for i in range(got.value)]

    def read_framebuffer(self) -> np.ndarray:
        """(H, W, 4) float32; (K, H, W, 4) in a context with K > 1 views."""
        w, h = self._texture_size
        out = np.empty((h, w, 4) if self._num_views == 1 else (self._num_views, h, w, 4), dtype=np.float32)
        _lib.check(_lib.lib().gsr_debug_copy(self._ctx, _lib.GSR_BUF_FRAMEBUFFER, C.c_void_p(out.ctypes.data), out.nbytes),
                   "gsr_debug_copy")
        return out

    def debug_copy(self, which: int, count: int, dtype) -> np.ndarray:
        out = np.empty(count, dtype=dtype)
        _lib.check(_lib.lib().gsr_debug_copy(self._ctx, which, C.c_void_p(out.ctypes.data), out.nbytes), "gsr_debug_copy")
        return out

    def keep_unsorted(self, enable: bool = True) -> None:
        _lib.check(_lib.lib().gsr_debug_keep_unsorted(self._ctx, int(enable)), "gsr_debug_keep_unsorted")


def sort_pairs(keys: np.ndarray, values: np.ndarray | None = None, device: int = 0):
    """Host convenience around gsr_sort_pairs_host (stable LSD radix sort on the GPU)."""
    k = np.array(keys, dtype=np.uint32, copy=True)
    v = None if values is None else np.array(values, dtype=np.uint32, copy=True)
    u32p = C.POINTER(C.c_uint32)
    _lib.check(_lib.lib().gsr_sort_pairs_host(device, k.ctypes.data_as(u32p), None if v is None else v.ctypes.data_as(u32p),
                                              k.size), "gsr_sort_pairs_host")
    return (k, v) if v is not None else k
