"""ctypes binding of the in-tree `libgsr.so` (include/gsr.h).

There is NO fallback: if the shared library is missing or does not load, importing a symbol raises, and
every entry point fails with GSR_ERR_CUDA when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GSR_LIB_PATH") or os.path.join(HERE, "libgsr.so")  # env override: kernel-variant experiments only

GSR_OK, GSR_ERR_INVALID, GSR_ERR_CUDA, GSR_ERR_OOM, GSR_ERR_STATE, GSR_ERR_OVERFLOW = range(6)
GSR_FLAG_REFERENCE_QUIRKS, GSR_FLAG_FIXED_RANGES, GSR_FLAG_FAST_REJECT, GSR_FLAG_STATIC_CAPACITY, GSR_FLAG_UNCONTRACTED_BLEND = 0x1, 0x2, 0x4, 0x8, 0x10
(GSR_BUF_RECORDS, GSR_BUF_KEYS, GSR_BUF_VALUES, GSR_BUF_BOUNDS, GSR_BUF_KEYS_UNSORTED, GSR_BUF_VALUES_UNSORTED,
 GSR_BUF_FRAMEBUFFER, GSR_BUF_COMPOSITOR_TRACE, GSR_BUF_COMPOSITOR_TRACE_COUNT) = range(9)

# every symbol include/gsr.h declares (tests/test_abi.py checks the header against this list and the .so)
EXPORTS = [
    "gsr_create", "gsr_destroy", "gsr_set_stream", "gsr_upload_splats_aos", "gsr_upload_ply_raw", "gsr_resize", "gsr_set_band", "gsr_set_row_interleave", "gsr_band_sync_word", "gsr_band_fixup", "gsr_render",
    "gsr_set_views", "gsr_render_views", "gsr_render_views_async",
    "gsr_render_async", "gsr_render_async_rgb", "gsr_render_async_fmt", "gsr_output_bytes", "gsr_present_device", "gsr_readback_async", "gsr_peer_export_framebuffers", "gsr_peer_import_framebuffers",
    "gsr_stream_join", "gsr_group_export", "gsr_group_attach", "gsr_group_detach", "gsr_group_set_present", "gsr_readback_rows_async", "gsr_sync", "gsr_framebuffer_device_ptr", "gsr_set_framebuffer_external", "gsr_pick",
    "gsr_get_stats", "gsr_get_frame_history", "gsr_debug_copy", "gsr_debug_enable_trace", "gsr_debug_compositor_config", "gsr_debug_pipeline", "gsr_debug_keep_unsorted", "gsr_sorter_create", "gsr_sorter_destroy",
    "gsr_sorter_sort_device", "gsr_sort_pairs_host", "gsr_sorter_last_ms", "gsr_error_string", "gsr_last_error",
    "gsr_device_count", "gsr_version",
]


class GsrConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_uint32), ("max_splats", C.c_uint64),
                ("dup_capacity_factor", C.c_uint32), ("reserved", C.c_uint32)]


class GsrStats(C.Structure):
    _fields_ = [("num_splats", C.c_uint64), ("duplicates", C.c_uint64), ("visible", C.c_uint64), ("capacity", C.c_uint64),
                ("last_tile", C.c_int64), ("overflow", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32),
                ("tiles_x", C.c_uint32), ("tiles_y", C.c_uint32), ("band_y0", C.c_uint32), ("band_y1", C.c_uint32),
                ("kernel_launches", C.c_uint32), ("stage_ms", C.c_float * 5), ("staged", C.c_uint64)]


GSR_HISTORY_FRAMES = 512
GSR_OUT_RGBA32F, GSR_OUT_RGB32F, GSR_OUT_RGBA16F, GSR_OUT_RGBA8 = range(4)
GSR_OUT_SRGB_TO_LINEAR = 0x100
GSR_GROUP_BLOB_BYTES = 320
GSR_MAX_VIEWS = 4


class GsrFrameRecord(C.Structure):
    _fields_ = [("frame_index", C.c_uint64), ("duplicates", C.c_uint64), ("visible", C.c_uint64), ("staged", C.c_uint64),
                ("overflow", C.c_uint32), ("reserved", C.c_uint32), ("stage_ms", C.c_float * 5), ("front_ms", C.c_float)]


class GsrError(RuntimeError):
    def __init__(self, code: int, where: str):
        L = lib()
        super().__init__(f"{where}: {L.gsr_error_string(code).decode()} [{code}] -- {L.gsr_last_error().decode()}")
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m godotgaussiansplatting_b200.build` "
                              "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        vp, fp, u32 = C.c_void_p, C.POINTER(C.c_float), C.c_uint32
        L.gsr_create.argtypes = [C.POINTER(GsrConfig), C.POINTER(vp)]
        L.gsr_destroy.argtypes = [vp]
        L.gsr_set_stream.argtypes = [vp, vp]
        L.gsr_upload_splats_aos.argtypes = [vp, fp, C.c_uint64, C.c_uint64]
        L.gsr_upload_ply_raw.argtypes = [vp, fp, u32, C.c_uint64, C.c_uint64, C.c_float]
        L.gsr_resize.argtypes = [vp, C.c_int32, C.c_int32]
        L.gsr_set_band.argtypes = [vp, C.c_int32, C.c_int32]
        L.gsr_set_row_interleave.argtypes = [vp, C.c_int32, C.c_int32]
        L.gsr_band_sync_word.argtypes = [vp]
        L.gsr_band_sync_word.restype = vp
        L.gsr_band_fixup.argtypes = [vp]
        L.gsr_render.argtypes = [vp, fp, vp, C.c_float, vp]
        L.gsr_render_async.argtypes = [vp, fp, vp, C.c_float, vp]
        L.gsr_set_views.argtypes = [vp, C.c_int32]
        L.gsr_render_views.argtypes = [vp, fp, vp, C.c_float, vp]
        L.gsr_render_views_async.argtypes = [vp, fp, vp, C.c_float, vp, C.c_int32]
        L.gsr_render_async_rgb.argtypes = [vp, fp, vp, C.c_float, vp]
        L.gsr_render_async_fmt.argtypes = [vp, fp, vp, C.c_float, vp, C.c_int32]
        L.gsr_output_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
        L.gsr_output_bytes.restype = C.c_size_t
        L.gsr_present_device.argtypes = [vp, vp, C.c_int32]
        L.gsr_sync.argtypes = [vp]
        L.gsr_stream_join.argtypes = [vp]
        L.gsr_group_export.argtypes = [vp, vp]
        L.gsr_group_attach.argtypes = [vp, C.c_int32, C.c_int32, vp]
        L.gsr_group_detach.argtypes = [vp]
        L.gsr_group_set_present.argtypes = [vp, C.c_int32]
        L.gsr_readback_rows_async.argtypes = [vp, vp]
        L.gsr_readback_async.argtypes = [vp, vp, C.c_int]
        L.gsr_peer_export_framebuffers.argtypes = [vp, vp]
        L.gsr_peer_import_framebuffers.argtypes = [vp, vp]
        L.gsr_framebuffer_device_ptr.argtypes = [vp]
        L.gsr_framebuffer_device_ptr.restype = vp
        L.gsr_set_framebuffer_external.argtypes = [vp, vp]
        L.gsr_pick.argtypes = [vp, u32, C.c_float, fp]
        L.gsr_get_stats.argtypes = [vp, C.POINTER(GsrStats)]
        L.gsr_get_frame_history.argtypes = [vp, u32, C.POINTER(GsrFrameRecord), C.POINTER(u32)]
        L.gsr_debug_copy.argtypes = [vp, C.c_int, vp, C.c_size_t]
        L.gsr_debug_keep_unsorted.argtypes = [vp, C.c_int]
        L.gsr_debug_enable_trace.argtypes = [vp, u32]
        L.gsr_debug_compositor_config.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32]
        L.gsr_debug_pipeline.argtypes = [vp, C.c_int32]
        L.gsr_sorter_create.argtypes = [C.c_int32, C.c_uint64, C.POINTER(vp)]
        L.gsr_sorter_destroy.argtypes = [vp]
        L.gsr_sorter_sort_device.argtypes = [vp, vp, vp, C.c_uint64, vp]
        L.gsr_sort_pairs_host.argtypes = [C.c_int32, C.POINTER(u32), C.POINTER(u32), C.c_uint64]
        L.gsr_sorter_last_ms.argtypes = [vp, fp]
        L.gsr_error_string.argtypes = [C.c_int]
        L.gsr_error_string.restype = C.c_char_p
        L.gsr_last_error.restype = C.c_char_p
        L.gsr_version.restype = C.c_char_p
        for name in EXPORTS:
            fn = getattr(L, name)
            if fn.restype is C.c_int and name not in ("gsr_device_count",):
                pass
        _lib = L
    return _lib


def check(code: int, where: str) -> None:
    if code != GSR_OK:
        raise GsrError(code, where)
