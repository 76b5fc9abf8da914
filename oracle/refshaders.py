"""Run the reference's OWN compute shaders on the CPU (oracle/_ref/libgsr_refshaders.so) -- the pin for the oracle.

TEST INFRASTRUCTURE ONLY (same import rule as oracle/oracle.py).  The library is the reference's six .glsl files
compiled for the CPU by oracle/glsl_cpu/build_ref.py; this module is the host side: it allocates the buffers of
`init_gpu()` (util/gaussian_splatting_rasterizer.gd:79-90) and issues the dispatches of `rasterize()` (:122-160) in
the same order with the same push constants, indirect dispatch sizes read from `grid_dimensions` like the GPU would.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
import sys
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(_HERE, "glsl_cpu"))
try:
    import build_ref as _build_ref
finally:
    sys.path.pop(0)

RADIX = 256                      # gaussian_splatting_rasterizer.gd:5-8 / radix_sort_*.glsl
PARTITION_SIZE = 8 * 512
TILE_SIZE = 16
RECORD_DTYPE = np.dtype(
    [("image_pos", "<f4", 2), ("pos_xy", "<f4", 2), ("conic", "<f4", 3), ("pos_z", "<f4"), ("color", "<f4", 4)]
)

_libs: dict[bool, C.CDLL] = {}


def available() -> bool:
    """True when the libraries exist (prebuilt) or can be built (reference present)."""
    try:
        return _build_ref.build()
    except Exception:
        return False


def _lib(libm: bool) -> C.CDLL:
    if libm not in _libs:
        if not _build_ref.build():
            raise RuntimeError("oracle/_ref/libgsr_refshaders*.so missing and GSR_REFERENCE_DIR does not name the reference to build it")
        if not libm:
            from . import oracle as _oracle   # makes sure libgsr_oracle.so (orc_test_exp/pow) exists
            _oracle.build()
        L = C.CDLL(_build_ref.lib_path(libm))
        for s in _build_ref.SHADERS:
            f = getattr(L, f"refshader_{s}_dispatch")
            f.restype = C.c_int
            f.argtypes = [C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_void_p, C.c_size_t,
                          C.c_size_t]
            getattr(L, f"refshader_{s}_bindings").restype = C.c_int
            getattr(L, f"refshader_{s}_set_shared_fill").argtypes = [C.c_uint]
        _libs[libm] = L
    return _libs[libm]


def set_shared_fill(word: int, libm: bool = False) -> None:
    """Value every word of `shared` storage holds when a workgroup starts (undefined in GLSL; it matters for
    gsplat_boundaries.glsl:36, which reads a shared word that no invocation of workgroup 0 wrote)."""
    L = _lib(libm)
    for s in _build_ref.SHADERS:
        getattr(L, f"refshader_{s}_set_shared_fill")(int(word) & 0xFFFFFFFF)


def create_push_constant(data) -> bytes:
    """util/render_context.gd:117-130: 4 bytes per entry (s32 for int/bool, f32 for float), zero-padded to 16."""
    raw = b"".join(struct.pack("<f", v) if isinstance(v, float) else struct.pack("<i", int(v)) for v in data)
    return raw + b"\0" * (-len(raw) % 16)


@dataclass
class ReferenceFrame:
    rgba: np.ndarray          # (H, W, 4) float32 -- the rgba32f render texture
    records: np.ndarray       # culled_splats, RECORD_DTYPE[n]
    keys_unsorted: np.ndarray
    values_unsorted: np.ndarray
    keys: np.ndarray          # sorted, first M of sort_keys
    values: np.ndarray
    bounds: np.ndarray        # (T, 2) uint32
    duplicates: int           # histogram[0] = sort_buffer_size
    grid_dims: np.ndarray     # the 6 indirect-dispatch words
    pick: np.ndarray          # tile_splat_pos (4 floats)


class ReferencePipeline:
    """The reference's rasterizer object, CPU-executed.  splat60: the 60-float std430 Splat records."""

    def __init__(self, splat60: np.ndarray, width: int, height: int, libm: bool = False):
        self.L = _lib(libm)
        self.splats = np.ascontiguousarray(splat60, dtype=np.float32).reshape(-1, 60).copy()
        self.n = n = self.splats.shape[0]
        self.w, self.h = int(width), int(height)
        self.tile_dims = ((self.w + TILE_SIZE - 1) // TILE_SIZE, (self.h + TILE_SIZE - 1) // TILE_SIZE)
        # --- init_gpu(), :79-90 ---
        self.cap = cap = n * 10                                   # num_sort_elements_max
        num_partitions = (cap + PARTITION_SIZE - 1) // PARTITION_SIZE
        self.culled = np.zeros(n, dtype=RECORD_DTYPE)             # point_cloud.size * 12*4
        self.grid_dims = np.ones(6, dtype=np.uint32)              # block_dims.fill(1)
        self.histogram = np.zeros(1 + 1 + 4 * RADIX + num_partitions * RADIX, dtype=np.uint32)   # 4 + (1 + 4R + P*R)*4 bytes
        self.sort_keys = np.zeros(max(2 * cap, 1), dtype=np.uint32)
        self.sort_values = np.zeros(max(2 * cap, 1), dtype=np.uint32)
        self.tile_bounds = np.zeros((self.tile_dims[0] * self.tile_dims[1], 2), dtype=np.uint32)
        self.tile_splat_pos = np.zeros(4, dtype=np.float32)
        self.render_texture = np.zeros((self.h, self.w, 4), dtype=np.float32)
        self.uniforms = np.zeros(8, dtype=np.float32)

    def _dispatch(self, shader: str, groups, buffers, push: bytes = b""):
        nb = len(buffers)
        ptrs = (C.c_void_p * nb)(*[b.ctypes.data for b in buffers])
        sizes = (C.c_size_t * nb)(*[b.nbytes for b in buffers])
        pc = C.create_string_buffer(push, max(len(push), 16))
        f = getattr(self.L, f"refshader_{shader}_dispatch")
        assert getattr(self.L, f"refshader_{shader}_bindings")() == nb, shader
        rc = f(int(groups[0]), int(groups[1]), int(groups[2]), ptrs, sizes, C.cast(pc, C.c_void_p), self.w, self.h)
        assert rc == 0

    def rasterize(self, camera_push_constants, uniforms32: bytes, heatmap: float = 0.0, target_tile: int = -1,
                  stop_after: str | None = None) -> ReferenceFrame:
        """camera_push_constants: 32 floats (view, projection); uniforms32: the 32-byte std140 block :126 writes."""
        vp = np.ascontiguousarray(camera_push_constants, dtype=np.float32).reshape(32)
        self.uniforms[:] = np.frombuffer(bytes(uniforms32), dtype=np.float32)          # buffer_update :126
        self.histogram[: 1 + 4 * RADIX] = 0                                              # buffer_clear :127
        self.tile_bounds[:] = 0                                                          # buffer_clear :128
        # :134-137 projection, ceili(point_cloud.size/256.0) groups (:103)
        self._dispatch("gsplat_projection", ((self.n + 255) // 256, 1, 1),
                       [self.splats, self.culled, self.histogram, self.sort_keys, self.sort_values, self.grid_dims, self.uniforms],
                       vp.tobytes())
        m = int(self.histogram[0])
        ku, vu = self.sort_keys[: min(m, self.cap)].copy(), self.sort_values[: min(m, self.cap)].copy()
        # :141-149 four sort passes; upsweep/downsweep indirect on grid_dimensions[0:3], spine on RADIX groups
        for p in range(4):
            push = create_push_constant([p, self.cap * (p % 2), self.cap * (1 - (p % 2))])
            g = tuple(int(x) for x in self.grid_dims[0:3])
            self._dispatch("radix_sort_upsweep", g, [self.histogram, self.sort_keys], push)
            self._dispatch("radix_sort_spine", (RADIX, 1, 1), [self.histogram], push)
            self._dispatch("radix_sort_downsweep", g, [self.histogram, self.sort_keys, self.sort_values], push)
        # :153-155 boundaries, indirect on grid_dimensions[3:6]
        self._dispatch("gsplat_boundaries", tuple(int(x) for x in self.grid_dims[3:6]),
                       [self.histogram, self.sort_keys, self.tile_bounds])
        # :158-159 render
        self._dispatch("gsplat_render", (self.tile_dims[0], self.tile_dims[1], 1),
                       [self.culled, self.sort_values, self.tile_bounds, self.tile_splat_pos, self.render_texture],
                       create_push_constant([float(heatmap), int(target_tile)]))
        mm = min(m, self.cap)
        return ReferenceFrame(self.render_texture.copy(), self.culled.copy(), ku, vu, self.sort_keys[:mm].copy(),
                              self.sort_values[:mm].copy(), self.tile_bounds.copy(), m, self.grid_dims.copy(),
                              self.tile_splat_pos.copy())


def sort_pairs(keys, values, cap=None, libm: bool = False):
    """The three radix-sort shaders x 4 passes on their own (rasterizer.gd:141-149)."""
    keys = np.asarray(keys, dtype=np.uint32)
    values = np.asarray(values, dtype=np.uint32)
    n = keys.size
    cap = int(cap if cap is not None else max(n, 1))
    L = _lib(libm)
    num_partitions = (cap + PARTITION_SIZE - 1) // PARTITION_SIZE
    hist = np.zeros(1 + 1 + 4 * RADIX + num_partitions * RADIX, dtype=np.uint32)
    k = np.zeros(2 * cap, dtype=np.uint32)
    v = np.zeros(2 * cap, dtype=np.uint32)
    k[:n], v[:n] = keys, values
    hist[0] = n
    groups = ((n + PARTITION_SIZE - 1) // PARTITION_SIZE, 1, 1)

    def run(shader, g, bufs, push):
        ptrs = (C.c_void_p * len(bufs))(*[b.ctypes.data for b in bufs])
        sizes = (C.c_size_t * len(bufs))(*[b.nbytes for b in bufs])
        pc = C.create_string_buffer(push, 16)
        assert getattr(L, f"refshader_{shader}_dispatch")(g[0], g[1], g[2], ptrs, sizes, C.cast(pc, C.c_void_p), 0, 0) == 0

    for p in range(4):
        push = create_push_constant([p, cap * (p % 2), cap * (1 - (p % 2))])
        run("radix_sort_upsweep", groups, [hist, k], push)
        run("radix_sort_spine", (RADIX, 1, 1), [hist], push)
        run("radix_sort_downsweep", groups, [hist, k, v], push)
    return k[:n].copy(), v[:n].copy()
