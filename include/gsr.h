/*
 * gsr.h -- C-ABI of libgsr.so: the B200-native (sm_100a) forward 3D-Gaussian-splatting rasterizer that
 * replaces the body of 2Retr0/GodotGaussianSplatting's `GaussianSplattingRasterizer`
 * (util/gaussian_splatting_rasterizer.gd) plus the six compute shaders it dispatches
 * (the .glsl files of resources/shaders/compute) and the RenderingDevice wrapper (util/render_context.gd).
 *
 * The reference has no native/FFI boundary of its own: its "plugin API" is the GDScript class.  Each
 * entry point below cites the reference interface it replaces (paths relative to the reference root).
 * A Godot host binds these through a GDExtension shim or C# P/Invoke (see INTEGRATION.md); this repo's
 * tests and bench bind them with Python ctypes (godotgaussiansplatting_b200/_lib.py).
 *
 * Conventions: plain C, opaque handle, `int` status returns (0 = GSR_OK), no exceptions cross the
 * boundary, no torch/CUDA types in signatures (device pointers and streams travel as void*).
 * All calls on one handle must be serialised by the caller (the reference calls everything from the
 * render thread: main.gd:122,152,156).  There is NO CPU fallback: every entry point fails with
 * GSR_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef GSR_H_
#define GSR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSR_API __attribute__((visibility("default")))

/* ---- status codes ---- */
enum {
    GSR_OK = 0,
    GSR_ERR_INVALID = 1,  /* bad argument / out-of-range size */
    GSR_ERR_CUDA = 2,     /* CUDA runtime failure, or no usable device (see gsr_last_error) */
    GSR_ERR_OOM = 3,      /* device allocation failed */
    GSR_ERR_STATE = 4,    /* call order violated (e.g. render before resize) */
    GSR_ERR_OVERFLOW = 5  /* duplicate list exceeded capacity (main.gd:100 "(buffer overflow!)") */
};

/* ---- gsr_config.flags ---- */
#define GSR_FLAG_REFERENCE_QUIRKS 0x1u /* reproduce gsplat_boundaries.glsl:47-49 tile-range quirks (Q10); default */
#define GSR_FLAG_FIXED_RANGES     0x2u /* corrected tile ranges instead (every occupied tile gets [start,end)) */
#define GSR_FLAG_FAST_REJECT      0x4u /* sharded (row-interleaved) contexts: force the conservative early reject + CTA-level compaction
                                          in the projection (exact; selected automatically from 6 ranks, where it is faster) */

#define GSR_FLAG_STATIC_CAPACITY  0x8u /* keep the reference's fixed duplicate capacity factor*N and truncate on overflow (rasterizer.gd:79,
                                          main.gd:100).  Default: the capacity starts at factor*N and GROWS -- every frame's M reaches a
                                          pinned host mirror without a host sync and the buffers are enlarged once M passes half of them;
                                          gsr_render with a host pointer re-renders a frame that still overflowed, so it never returns a
                                          truncated frame; an asynchronous frame that overflowed is flagged (gsr_stats.overflow /
                                          gsr_frame_record.overflow) and the next one has room */

#define GSR_FLAG_UNCONTRACTED_BLEND 0x10u /* debug: evaluate gsplat_render.glsl:84-90 with one rounding per GLSL operator (no fma anywhere).
                                            The default contracts at the five GLSL-legal points of the gsr spec (DESIGN.md section 4); without
                                            contraction the frame is bit-identical to the reference's own shader text executed on the CPU
                                            (oracle/_ref; oracle.set_blend_contraction(False)). */

/* ---- gsr_debug_copy selectors (parity taps; not on the frame path) ---- */
enum {
    GSR_BUF_RECORDS = 0, /* 48 B RasterizeData per splat id (gsplat_projection.glsl:42-48), max_splats entries */
    GSR_BUF_KEYS = 1,    /* sorted keys, M entries (descriptors['sort_keys'] half 0) */
    GSR_BUF_VALUES = 2,  /* sorted values, M entries (descriptors['sort_values'] half 0) */
    GSR_BUF_BOUNDS = 3,  /* uvec2 per tile (descriptors['tile_bounds']) */
    GSR_BUF_KEYS_UNSORTED = 4,  /* keys in emission order (only valid if flags keep them; see gsr_debug_keep_unsorted) */
    GSR_BUF_VALUES_UNSORTED = 5,
    GSR_BUF_FRAMEBUFFER = 6,  /* RGBA32F W*H (descriptors['render_texture']) */
    GSR_BUF_COMPOSITOR_TRACE = 7,       /* schedule trace of the last frame's compositor (gsr_debug_enable_trace) */
    GSR_BUF_COMPOSITOR_TRACE_COUNT = 8  /* number of trace items written (uint32) */
};

typedef struct gsr_ctx gsr_ctx;       /* one rasterizer = one GaussianSplattingRasterizer instance */
typedef struct gsr_sorter gsr_sorter; /* stand-alone radix sorter (config c5 microbench) */

typedef struct gsr_config {
    int32_t device;               /* CUDA ordinal (RenderingServer.get_rendering_device(), rasterizer.gd:70) */
    uint32_t flags;               /* GSR_FLAG_*; 0 = GSR_FLAG_REFERENCE_QUIRKS */
    uint64_t max_splats;          /* point_cloud.size (rasterizer.gd:79,83) */
    uint32_t dup_capacity_factor; /* initial sort capacity = factor * max_splats; 0 -> 10 (rasterizer.gd:79); grows on demand */
    uint32_t reserved;
} gsr_config;

typedef struct gsr_stats {
    uint64_t num_splats;  /* highest uploaded splat index + 1 */
    uint64_t duplicates;  /* M = histogram[0] of the reference (main.gd:98) -- true count, may exceed capacity */
    uint64_t visible;     /* V: splats that passed the cull and touch >= 1 tile */
    uint64_t capacity;    /* sort capacity in pairs */
    int64_t last_tile;    /* largest tile id touched by any visible splat (-1 if none) */
    uint32_t overflow;    /* 1 if duplicates > capacity in the last frame */
    uint32_t width, height, tiles_x, tiles_y;
    uint32_t band_y0, band_y1;  /* tile-row band rendered by this context */
    uint32_t kernel_launches;   /* kernels launched by the last gsr_render */
    float stage_ms[5];    /* 'Projection','Sort','Boundaries','Render' (rasterizer.gd:139,150,155,160) + total */
    uint64_t staged;      /* C: instances actually staged by the compositor (sum of consumed chunk sizes) */
} gsr_stats;

/* One entry of the per-frame history ring (the last GSR_HISTORY_FRAMES frames rendered by a context). */
#define GSR_HISTORY_FRAMES 512
typedef struct gsr_frame_record {
    uint64_t frame_index; /* 0-based count of gsr_render calls on this context */
    uint64_t duplicates;  /* M */
    uint64_t visible;     /* V */
    uint64_t staged;      /* C */
    uint32_t overflow;
    uint32_t reserved;
    float stage_ms[5];    /* Projection, Sort, Boundaries, Render, total (= their sum) -- GPU time between CUDA events around every stage */
    float front_ms;       /* the part of Projection that ran on the front stream (clear + projection kernel): overlapped with the previous
                             frame's compositor when frames are enqueued back to back, so the frame period is shorter than `total` */
} gsr_frame_record;

/* ---- lifecycle: replaces _init/init_gpu/cleanup_gpu (rasterizer.gd:59-120) and RenderingContext
 *      (render_context.gd:35-51).  Allocates every buffer of rasterizer.gd:83-92 (SoA instead of AoS). ---- */
GSR_API int gsr_create(const gsr_config *cfg, gsr_ctx **out);
GSR_API int gsr_destroy(gsr_ctx *ctx);

/* Use an existing CUDA stream (cudaStream_t as void*; NULL = the context's own stream).  The host that
 * owns the GPU work queue (Godot's render thread; torch's current stream in bench.py) passes its stream. */
GSR_API int gsr_set_stream(gsr_ctx *ctx, void *cuda_stream);

/* ---- splat upload: replaces device.buffer_update(buffer, i*STRUCT_SIZE*stride*4, ...) of
 *      PlyFile.load_gaussian_splats (util/ply_file.gd:71).  `splat60` = `count` std430 Splat structs of
 *      60 floats (gsplat_projection.glsl:33-40) in host memory; converted to SoA planes on the device.
 *      May be called repeatedly with disjoint or overlapping ranges (chunked async load). ---- */
GSR_API int gsr_upload_splats_aos(gsr_ctx *ctx, const float *splat60, uint64_t first, uint64_t count);

/* Same, but from RAW PLY vertices (scope row f1): `ply` = `count` vertices of `nprops` float32 each in the standard 3DGS
 * order (x,y,z,nx,ny,nz,f_dc_0..2,f_rest_0..44,opacity,scale_0..2,rot_0..3,...).  The per-splat preprocessing of
 * PlyFile.load_gaussian_splats (util/ply_file.gd:44-69: exp(scale), quaternion -> R, Sigma = R S^2 R^T, sigmoid(opacity),
 * SH re-interleave) runs on the device and writes the SoA planes directly; `creation_time` stamps the chunk (:40,47). */
GSR_API int gsr_upload_ply_raw(gsr_ctx *ctx, const float *ply, uint32_t nprops, uint64_t first, uint64_t count, float creation_time);

/* ---- texture_size setter (rasterizer.gd:26-48): reallocates tile_bounds + render_texture ---- */
GSR_API int gsr_resize(gsr_ctx *ctx, int32_t width, int32_t height);

/* Multi-GPU tile-row sharding (no counterpart in the single-device reference): this context renders tile
 * rows [row_begin, row_end) only; keys keep the global tile id.  (0, tiles_y) restores the full frame. */
GSR_API int gsr_set_band(gsr_ctx *ctx, int32_t row_begin, int32_t row_end);

/* Cyclic tile-row ownership for balanced multi-GPU sharding: this context owns the tile rows with
 * row % row_mod == row_rem (inside its band).  row_mod > 1 selects the FAST sharded mode: the projection rejects, with a
 * conservative radius bound, splats that cannot touch an owned row, so it no longer knows the frame-global last
 * occupied tile that the reference's tile-range quirk (gsplat_boundaries.glsl:47-49) depends on.  Instead every rank
 * leaves its local last occupied tile + 1 in the int32 at gsr_band_sync_word(); the host all-reduces that word (MAX,
 * in place, on the render stream) after the frame and calls gsr_band_fixup, which blanks the one affected tile on the
 * rank that owns it.  (1, 0) restores the exact single-context behaviour. */
GSR_API int gsr_set_row_interleave(gsr_ctx *ctx, int32_t row_rem, int32_t row_mod);
GSR_API void *gsr_band_sync_word(gsr_ctx *ctx);
GSR_API int gsr_band_fixup(gsr_ctx *ctx);

/* Fused compositor + framebuffer gather over NVLink peer memory (replaces the NCCL gather of SURVEY 8e): the presenting
 * rank exports CUDA-IPC handles of its two frames (2 x 64 bytes); every other rank imports them, after which its
 * compositor stores its tile-row band straight into the presenting rank's memory.  In this mode gsr_render_async is
 * called with a NULL host pointer on every rank (frames alternate between the two buffers in lockstep), the ranks
 * synchronise per frame with any 4-byte collective, and the presenting rank calls gsr_readback_async. */
GSR_API int gsr_peer_export_framebuffers(gsr_ctx *ctx, void *handles128);
GSR_API int gsr_peer_import_framebuffers(gsr_ctx *ctx, const void *handles128);

/* ---- rasterize() (rasterizer.gd:122-160).
 *      view_proj: the 128-byte push constant of update_camera_matrices (rasterizer.gd:181-193):
 *                 view_matrix then projection_matrix, GLSL column-major.
 *      uniforms:  the 32-byte uniform block of rasterizer.gd:126, byte-identical:
 *                 float camera_pos[3], float model_scale, int32 width, int32 height, float time, pad.
 *                 (width/height must equal the gsr_resize values.)
 *      heatmap_factor: float(should_enable_heatmap) (rasterizer.gd:158).
 *      out_rgba32f_host: NULL (frame stays on the device, like the reference's Texture2DRD) or a host
 *                 buffer of width*height*4 floats that receives the frame (synchronous).
 *      Enqueues on the context's stream and returns without a host sync when out_rgba32f_host is NULL. */
GSR_API int gsr_render(gsr_ctx *ctx, const float view_proj[32], const void *uniforms32, float heatmap_factor,
                       float *out_rgba32f_host);

/* ---- multiview (stereo / XR): several cameras of one splat cloud in one frame.  No reference counterpart: an OpenXR host
 *      (Godot's XRInterface: get_view_count(), get_transform_for_view(), get_projection_for_view()) renders every view of a frame
 *      into one layer of a texture array.  The splats stay resident once; every splat is read once per frame and projected
 *      for all K cameras; one sort and one compositor launch serve all views.
 *      Layer v of a K-view frame is bit-identical to what gsr_render of camera v produces in a single-view context with the same
 *      flags (incl. the Q10 tile-range quirks, applied per view, GSR_FLAG_FIXED_RANGES, GSR_FLAG_UNCONTRACTED_BLEND, heat-map and
 *      load-in animation).
 *      gsr_set_views(ctx, K), 1 <= K <= GSR_MAX_VIEWS (default 1): reallocates the K-layer frames, tile bounds and record tables.
 *        GSR_ERR_INVALID (context unchanged) when K * tiles > 65536 (the sort key's 16-bit tile id: 4 views at 1920x1080, 2 at
 *        3840x2160); GSR_ERR_STATE in a context with a shard group, peer frames, a band or row interleave, or overlap on -- and those
 *        calls return GSR_ERR_STATE while K > 1.  gsr_resize applies the same K * tiles check.
 *      In a K > 1 context: gsr_render / gsr_render_async* return GSR_ERR_STATE (use the calls below); the frame is K layers of
 *        W*H RGBA32F pixels, layer v at pixel offset v*W*H (a VK_IMAGE_VIEW_TYPE_2D_ARRAY image of K layers); gsr_framebuffer_device_ptr
 *        is layer 0, gsr_set_framebuffer_external needs K layers, gsr_present_device / gsr_readback_async convert or copy all K
 *        layers; gsr_pick takes tile ids in [0, K*T) (view = tile_id / T); gsr_get_stats / gsr_get_frame_history report M, V and C
 *        summed over the views and last_tile in that concatenated id space; the gsr_debug_copy taps cover all views (K*T bounds,
 *        K record tables of max_splats records, the K-layer frame).
 *      view_proj: K push constants of 32 floats (any projection, incl. the asymmetric per-eye frusta of XR).
 *      uniforms:  K uniform blocks of 32 bytes; they must agree on model_scale, width, height and time (else GSR_ERR_INVALID) --
 *                 only camera_pos differs between views. ---- */
#define GSR_MAX_VIEWS 4
GSR_API int gsr_set_views(gsr_ctx *ctx, int32_t num_views);
/* out_rgba32f_host: NULL (frame stays on the device) or K*W*H*4 floats, layer-major; synchronous like gsr_render. */
GSR_API int gsr_render_views(gsr_ctx *ctx, const float *view_proj /* K x 32 */, const void *uniforms /* K x 32 B */,
                             float heatmap_factor, float *out_rgba32f_host);
/* Pipelined read-back of all K layers (gsr_render_async_fmt): pinned_host holds K x gsr_output_bytes(format, W, H) bytes. */
GSR_API int gsr_render_views_async(gsr_ctx *ctx, const float *view_proj, const void *uniforms, float heatmap_factor,
                                   void *pinned_host, int32_t format);

/* Pipelined host read-back: enqueue the frame and an asynchronous device->host copy into `pinned_host` (page-locked
 * memory; with pageable memory the copy degrades to a synchronous one).  Frames alternate between two internal
 * framebuffers and the copy runs on a separate stream, so the read-back of frame i overlaps the kernels of frame i+1.
 * gsr_stream_join makes the render stream wait for all copies enqueued so far (so that an event recorded on the
 * render stream afterwards covers them); gsr_sync blocks the host until renders and copies are complete. */
GSR_API int gsr_render_async(gsr_ctx *ctx, const float view_proj[32], const void *uniforms32, float heatmap_factor,
                             float *pinned_host);
/* Same, but the host frame is RGB32F (width*height*3 floats): the alpha channel of the reference's output is the
 * constant 1.0 (gsplat_render.glsl:101), so it is packed away on the device before the PCIe transfer (-25 % bytes). */
GSR_API int gsr_render_async_rgb(gsr_ctx *ctx, const float view_proj[32], const void *uniforms32, float heatmap_factor,
                                 float *pinned_host_rgb);
/* ---- presentation hand-off (scope row f3; resources/shaders/spatial/main.gdshader:7-19, rasterizer.gd:41,48,92,101).
 *      The reference keeps an RGBA32F image and converts sRGB -> linear in the fragment shader that samples it.  A consumer that
 *      wants fewer bytes (PCIe read-back, the gather message) or the converted values asks for them here; the conversion is fused
 *      into the copy-out kernel.  format = GSR_OUT_* optionally OR-ed with GSR_OUT_SRGB_TO_LINEAR (rgb channels only). ---- */
enum {
    GSR_OUT_RGBA32F = 0, /* 16 B/pixel: the reference's texture, bit for bit */
    GSR_OUT_RGB32F = 1,  /* 12 B/pixel: alpha is the constant 1.0 (gsplat_render.glsl:101) */
    GSR_OUT_RGBA16F = 2, /*  8 B/pixel: IEEE binary16, round to nearest even */
    GSR_OUT_RGBA8 = 3    /*  4 B/pixel: UNORM8 = rint(clamp(x, 0, 1) * 255) */
};
#define GSR_OUT_SRGB_TO_LINEAR 0x100 /* apply main.gdshader:7-11 srgb_to_linear() to r,g,b first (pow = the library's deterministic pow) */
GSR_API size_t gsr_output_bytes(int32_t format, int32_t width, int32_t height);
/* gsr_render_async with a converted host frame (gsr_output_bytes(format, w, h) bytes of page-locked memory). */
GSR_API int gsr_render_async_fmt(gsr_ctx *ctx, const float view_proj[32], const void *uniforms32, float heatmap_factor,
                                 void *pinned_host, int32_t format);
/* Read the most recently rendered library-owned frame back to page-locked host memory on the copy stream, ordered
 * after everything enqueued on the render stream so far (shard group: after every rank's rows have landed).
 * format: GSR_OUT_* (0 = RGBA32F, 1 = RGB32F -- the former `rgb_only` argument). */
GSR_API int gsr_readback_async(gsr_ctx *ctx, void *pinned_host, int32_t format);
/* Converted copy of the most recent frame into caller-owned DEVICE memory, on the render stream, no host involvement: the
 * zero-copy hand-off to an image the embedder imported from its graphics API (Vulkan VK_KHR_external_memory_fd ->
 * cudaImportExternalMemory -> cudaExternalMemoryGetMappedBuffer; see INTEGRATION.md). */
GSR_API int gsr_present_device(gsr_ctx *ctx, void *dst_device, int32_t format);
GSR_API int gsr_stream_join(gsr_ctx *ctx);

/* ---- Multi-GPU shard group (no reference counterpart -- the reference is single-device; SURVEY 8e).  One context per GPU,
 *      in one process (a thread per GPU) or in one process per GPU.  The frame path of an attached group uses neither the
 *      host nor NCCL: per frame every rank (1) projects ITS slice of the splats (cull, EWA, SH: once per splat in the whole group) and
 *      stores every (key, value) pair and every 48-byte record into the memory of the rank that owns the pair's tile row
 *      (cyclic rows: row % world == rank) with peer stores over NVLink/NVSwitch, in splat-id order per destination, (2) packs,
 *      sorts and scans the pairs it received, (3) composites its rows straight into the presenting rank's (rank 0) frame, or
 *      keeps them (gsr_group_set_present); sequence-numbered flag words behind one system-scope fence per kernel order all of
 *      it on the devices.
 *      Results are bit-identical to the single-GPU frame (same rects, same emission order, exact Q10 bookkeeping).
 *        every rank:  gsr_resize; gsr_group_export(ctx, blob)            -> exchange the blobs (any transport)
 *                     gsr_group_attach(ctx, rank, world, all_blobs)       -> barrier once (any transport)
 *        per frame:   gsr_render_async(ctx, vp, uniforms, heat, NULL) on every rank (same frame order everywhere);
 *                     rank 0: gsr_readback_async(ctx, pinned, format) and/or gsr_present_device / gsr_framebuffer_device_ptr
 *      gsr_resize detaches (export / attach again).  A lost peer makes the bounded device-side waits expire: gsr_sync then
 *      returns GSR_ERR_STATE instead of the GPU hanging. ---- */
#define GSR_GROUP_BLOB_BYTES 320
#define GSR_GROUP_MAX_RANKS 16
GSR_API int gsr_group_export(gsr_ctx *ctx, void *blob /* GSR_GROUP_BLOB_BYTES */);
GSR_API int gsr_group_attach(gsr_ctx *ctx, int32_t rank, int32_t world, const void *blobs /* world x GSR_GROUP_BLOB_BYTES, rank order */);
GSR_API int gsr_group_detach(gsr_ctx *ctx);
/* Where an attached group presents (same value on every rank; default 0):
 *   0  rows are composited into rank 0's frames over NVLink -- the frame is complete on ONE device (display GPU, gsr_present_device,
 *      gsr_readback_async on rank 0);
 *   1  every rank keeps its rows in its own frames and reads them back itself with gsr_readback_rows_async into one full-frame
 *      RGBA32F host image that is page-locked in every rank's process (shared memory): a host consumer gets the frame over
 *      world PCIe links instead of one, and no frame data crosses NVLink at all. */
GSR_API int gsr_group_set_present(gsr_ctx *ctx, int32_t rows_local);
GSR_API int gsr_readback_rows_async(gsr_ctx *ctx, void *host_frame_rgba32f);
GSR_API int gsr_sync(gsr_ctx *ctx);

/* Device pointer of the RGBA32F frame (render_texture.texture_rd_rid, rasterizer.gd:48,101); row-major W*H. */
GSR_API void *gsr_framebuffer_device_ptr(gsr_ctx *ctx);
/* Render into caller-owned device memory instead (>= width*height*16 bytes; NULL restores the internal one). */
GSR_API int gsr_set_framebuffer_external(gsr_ctx *ctx, void *device_ptr);

/* ---- get_splat_position() (rasterizer.gd:162-171): re-dispatches the compositor for `tile_id` and reads the
 *      16-byte tile_splat_pos buffer (gsplat_render.glsl:33-36,105-110).  out_xyzn = splat_pos.xyz,
 *      num_tile_splats -- persistent across calls exactly like the reference's storage buffer.
 *      GSR_ERR_STATE before the first gsr_render at the current size (no tile ranges exist yet). ---- */
GSR_API int gsr_pick(gsr_ctx *ctx, uint32_t tile_id, float heatmap_factor, float out_xyzn[4]);

/* ---- update_debug_info() (main.gd:93-119): M, overflow, per-stage GPU ms.  Synchronises the stream. ---- */
GSR_API int gsr_get_stats(gsr_ctx *ctx, gsr_stats *out);

/* Per-frame GPU timestamps + counters of the most recent frames, oldest first (capture_timestamp/
 * get_captured_timestamp_gpu_time, rasterizer.gd:135-160, main.gd:106-119).  Synchronises the stream once. */
GSR_API int gsr_get_frame_history(gsr_ctx *ctx, uint32_t max_frames, gsr_frame_record *out, uint32_t *n_out);

/* ---- parity taps: copy an internal buffer to host (synchronises).  bytes = size of dst. ---- */
GSR_API int gsr_debug_copy(gsr_ctx *ctx, int which, void *dst, size_t bytes);
/* Record, for every work item of the compositor, {tile<<32|SM id, start ns, end ns, first_chunk<<32|chunks<<1|finished}
 * (4 x uint64 per item, %globaltimer).  max_items = 0 disables.  Profiling aid; not on the frame path by default. */
GSR_API int gsr_debug_enable_trace(gsr_ctx *ctx, uint32_t max_items);
/* Scheduling of the compositor's persistent grid (results never depend on it): resident CTAs per SM (0 = as many as fit; default 2),
 * longest-chain-first ticket order (default on), and the sparse-frame rule of that order pass: with at most
 * sparse_tiles_per_sm * SMs occupied tiles only one CTA per SM works (default 5; 0 = never). */
GSR_API int gsr_debug_compositor_config(gsr_ctx *ctx, int32_t ctas_per_sm, int32_t longest_first, int32_t sparse_tiles_per_sm);
/* Front / back overlap of consecutive frames (results never depend on it): 1 = a frame's clear + projection run on a second
 * stream, released when the previous frame's tile ranges are done, i.e. beside that frame's compositor; 0 or -1 (default) = every
 * kernel of a frame on the render stream, frames strictly one after the other.  Measured on B200 (DESIGN.md section 6): one GPU,
 * c3: neutral (the two kernels compete for the same issue slots); shard group of 4, c3: +10 % device-resident and end to end;
 * shard group of 4, c4: +10 % device-resident but -35 % with the rows-local read-back -- hence off by default. */
GSR_API int gsr_debug_pipeline(gsr_ctx *ctx, int32_t overlap);
/* Keep an unsorted copy of the emitted pairs each frame (costs 8*M bytes of traffic; off by default). */
GSR_API int gsr_debug_keep_unsorted(gsr_ctx *ctx, int enable);

/* ---- stand-alone radix sort (config c5; replaces radix_sort_{upsweep,spine,downsweep}.glsl x 4 passes,
 *      rasterizer.gd:143-149).  Stable LSD sort of 32-bit keys (+ optional 32-bit values), 4 x 8-bit digits. ---- */
GSR_API int gsr_sorter_create(int32_t device, uint64_t max_n, gsr_sorter **out);
GSR_API int gsr_sorter_destroy(gsr_sorter *s);
/* Device-resident sort: keys/values are device pointers (values may be NULL); result in place.
 * cuda_stream: cudaStream_t as void* (NULL = default stream).  No host sync. */
GSR_API int gsr_sorter_sort_device(gsr_sorter *s, void *d_keys, void *d_values, uint64_t n, void *cuda_stream);
/* Host convenience: copies in, sorts on the GPU, copies out (values may be NULL). */
GSR_API int gsr_sort_pairs_host(int32_t device, uint32_t *keys, uint32_t *values, uint64_t n);
/* ms of the last gsr_sorter_sort_device call measured with CUDA events on its stream (synchronises). */
GSR_API int gsr_sorter_last_ms(gsr_sorter *s, float *ms);

/* ---- misc ---- */
GSR_API const char *gsr_error_string(int code);
GSR_API const char *gsr_last_error(void); /* thread-local detail of the last failure */
GSR_API int gsr_device_count(void);
GSR_API const char *gsr_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GSR_H_ */
