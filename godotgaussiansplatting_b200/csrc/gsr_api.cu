// gsr_api.cu -- the C-ABI of libgsr.so (include/gsr.h): context, buffers, per-frame sequencing.
//
// Host-side counterpart of GaussianSplattingRasterizer.init_gpu / rasterize / get_splat_position /
// cleanup_gpu (util/gaussian_splatting_rasterizer.gd:65-171) and of RenderingContext
// (util/render_context.gd).  Fifteen compute dispatches with full barriers per frame in the reference
// become 1 + 5 + 1 + 1 kernel launches on one CUDA stream, with no host synchronisation on the frame path.
#include <stdarg.h>
#include <stdlib.h>
#include <stddef.h>
#include <string.h>
#include <unistd.h>

#include <new>

#include "common.cuh"

namespace gsr {

static thread_local char g_last_error[512] = "";

void set_last_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof g_last_error, fmt, ap);
    va_end(ap);
}

}  // namespace gsr

using namespace gsr;

constexpr int EV_PER_FRAME = 7;

struct gsr_ctx {
    int device = 0;
    uint32_t flags = 0;
    uint64_t max_splats = 0, capacity = 0, plane_stride = 0, num_splats = 0;
    uint64_t cap_stride = 0;     // capacity rounded up to 1024 pairs: distance between the three pair buffers (keeps each 16-byte aligned)
    cudaStream_t stream = nullptr, own_stream = nullptr;
    float4 *soa = nullptr;       // 15 planes x plane_stride
    float4 *records = nullptr;   // 3 float4 per splat id; two tables (consecutive frames alternate: front / back overlap)
    float4 *records2 = nullptr;
    uint32_t *keys = nullptr;    // 3 * capacity: sort input of even frames | of odd frames | ping-pong partner (rasterizer.gd:88 has two halves)
    uint32_t *vals = nullptr;    // 3 * capacity
    uint32_t *keys_cur = nullptr, *vals_cur = nullptr;   // sorted pairs of the most recent frame
    float4 *records_cur = nullptr;                       // record table the most recent frame composited from
    // front / back overlap: the projection of frame f+1 (front: HBM-bound) runs on its own stream beside the compositor of frame f
    // (back: FMA-pipe / chain bound) when the host enqueues frames back to back (gsr_render_async).  gsr_debug_pipeline(ctx, 0) = serial.
    cudaStream_t front_stream = nullptr;
    cudaEvent_t front_gate = nullptr;    // recorded after the tile ranges of the most recent frame (nullptr: nothing to wait for)
    int overlap = -1;                    // -1 = default = off (measured: DESIGN.md section 6; on helps c3 on 4 GPUs by 10 %, not one GPU, and hurt c4's read-back leg)
    SortWorkspace sort;
    FrameState *ring = nullptr;  // GSR_HISTORY_FRAMES slots; slot = frame_counter % GSR_HISTORY_FRAMES
    FrameState *frame = nullptr; // slot of the most recent frame
    unsigned long long *lookback = nullptr;  // one word per projection block, cleared every frame
    uint32_t lookback_blocks = 0;
    uint64_t frame_counter = 0;
    uint2 *bounds = nullptr;     // followed in the same allocation by the compositor queue (one memset per frame)
    uint32_t *comp_order = nullptr, *comp_hint = nullptr;   // longest-chain-first ticket order of the compositor + last frame's consumed chunks
    int comp_ctas_per_sm = 2, comp_order_mode = 1, comp_max_ctas = 1, comp_sparse_per_sm = 5;   // scheduling of the compositor's persistent grid (gsr_debug_compositor_config)
    uint64_t comp_hint_key = 0;   // ownership (band, rows) the hints were recorded under: a change invalidates them
    FrameState *pick_frame = nullptr;  // queue counters of the single-tile pick launch
    ulonglong4 *trace = nullptr;       // GSR_BUF_COMPOSITOR_TRACE (debug; allocated by gsr_debug_enable_trace)
    uint32_t *trace_count = nullptr;
    uint32_t trace_cap = 0;
    float4 *fb = nullptr, *fb_ext = nullptr;
    float4 *fb2 = nullptr;                       // second frame for pipelined read-back (gsr_render_async)
    void *stage[2] = {nullptr, nullptr};         // converted copies of the two frames (GSR_OUT_* other than RGBA32F), lazily allocated (16 B/pixel)
    float4 *fb_last = nullptr;                   // frame written by the most recent render
    cudaStream_t copy_stream = nullptr;          // D2H read-back overlaps the next frame's kernels
    cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    bool copied_valid[2] = {false, false};
    uint64_t async_counter = 0;
    // multi-GPU peer mode: every rank's compositor stores its band straight into the presenting rank's two frames
    bool peer_mode = false, peer_opened = false;
    float4 *peer_fb[2] = {nullptr, nullptr};
    uint64_t peer_counter = 0;
    float4 *pick = nullptr;
    float4 *staging = nullptr;
    uint64_t staging_splats = 0;
    uint32_t *unsorted_keys = nullptr, *unsorted_vals = nullptr;
    bool keep_unsorted = false;
    int width = 0, height = 0, tiles_x = 0, tiles_y = 0, band_y0 = 0, band_y1 = 0;
    bool band_set = false;
    int row_mod = 1, row_rem = 0;   // cyclic tile-row ownership (gsr_set_row_interleave): fast sharded mode when row_mod > 1
    int32_t *sync_word = nullptr;   // local (then all-reduced) last occupied tile + 1
    // multi-GPU shard group (gsr_group_export / gsr_group_attach): NCCL-free frame path, see group.cu
    struct Group {
        void *arena = nullptr;            // this rank's arena: flag page | receive segments (2 parities x keys, values) | records (2 parities)
        uint64_t rx_capacity = 0;         // pairs per receive buffer (all sources together); seg_cap = rx_capacity / world
        int rank = 0, world = 0;          // world > 1 <=> attached
        char *peer_arena[GROUP_MAX] = {};    // every rank's arena (peer pointers)
        GroupFlags *flags[GROUP_MAX] = {};   // every rank's flag page
        float4 *root_fb[2] = {nullptr, nullptr};  // the presenting rank's two frames
        void *opened[3 * GROUP_MAX] = {};    // IPC mappings to close
        int n_opened = 0;
        int present_rows = 0;             // 1: every rank keeps its rows in its own frames and reads them back itself (gsr_group_set_present)
        uint32_t seq = 0;                 // frames rendered by the group so far (lockstep on all ranks)
        uint64_t slice = 0;               // splats per rank (256-aligned)
        uint32_t seg_cap = 0;             // pairs one source may send to one destination per frame
    } grp;
    cudaEvent_t *ev = nullptr;   // [GSR_HISTORY_FRAMES][EV_PER_FRAME]: front start, front end | back start, received, sorted, ranges, rendered
    // dynamic duplicate capacity (replaces the reference's static 10 x N, rasterizer.gd:79 "FIXME: This should not be a static
    // value!"): every frame's M travels to a pinned host mirror without a host sync; the capacity grows ahead of need
    FrameState *host_ring = nullptr;       // pinned mirror of `ring`
    cudaEvent_t *ev_stat = nullptr;        // [GSR_HISTORY_FRAMES] recorded after the slot's copy
    uint64_t stats_polled = 0;             // frames whose mirror has been examined
    uint64_t m_high = 0;                   // high-water mark of M over the examined frames
    uint64_t capacity_max = 0;
    bool ev_valid = false;
    uint32_t last_launches = 0;
    int sm_count = 0;
    // multiview frame (gsr_set_views): K layers of W*H pixels, K*T tile bounds, K record tables of 3 * max_splats float4 per table
    int num_views = 1;
    uint64_t cap_factor = 10;    // gsr_config.dup_capacity_factor: the initial capacity is num_views * factor * max_splats
};

struct gsr_sorter {
    int device = 0;
    SortWorkspace ws;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool timed = false;
};

namespace {

int use_device(int device) {
    GSR_CUDA_TRY(cudaSetDevice(device));
    return GSR_OK;
}

int check_device(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_last_error("no CUDA device available (%s); libgsr has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count=0");
        return GSR_ERR_CUDA;
    }
    if (device < 0 || device >= count) {
        set_last_error("device ordinal %d out of range [0,%d)", device, count);
        return GSR_ERR_INVALID;
    }
    cudaDeviceProp prop;
    GSR_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_last_error("device %d is sm_%d%d; libgsr is built for sm_100a only", device, prop.major, prop.minor);
        return GSR_ERR_CUDA;
    }
    return GSR_OK;
}

void group_detach(gsr_ctx *c) {
    if (c->front_stream) cudaStreamSynchronize(c->front_stream);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    for (int i = 0; i < c->grp.n_opened; ++i) cudaIpcCloseMemHandle(c->grp.opened[i]);
    c->grp.n_opened = 0;
    if (c->grp.world > 1) { c->row_mod = 1; c->row_rem = 0; }
    c->grp.world = 0; c->grp.rank = 0; c->grp.seq = 0; c->grp.present_rows = 0;
    c->grp.root_fb[0] = c->grp.root_fb[1] = nullptr;
}

float4 *framebuffer(gsr_ctx *c) { return c->fb_ext ? c->fb_ext : (c->fb_last ? c->fb_last : c->fb); }
// pixels of a frame (all layers) and tiles of a frame (all views)
size_t frame_pixels(const gsr_ctx *c) { return (size_t)c->width * c->height * (size_t)c->num_views; }
size_t frame_tiles(const gsr_ctx *c) { return (size_t)c->tiles_x * c->tiles_y * (size_t)c->num_views; }
int refuse_multiview(const char *what) {
    set_last_error("%s: unavailable in a multiview context (gsr_set_views > 1)", what);
    return GSR_ERR_STATE;
}

void free_ctx(gsr_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->front_stream) { cudaStreamSynchronize(c->front_stream); cudaStreamDestroy(c->front_stream); }
    cudaFree(c->soa); cudaFree(c->records); cudaFree(c->records2); cudaFree(c->keys); cudaFree(c->vals);
    sort_workspace_destroy(c->sort);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->peer_opened) { cudaIpcCloseMemHandle(c->peer_fb[0]); cudaIpcCloseMemHandle(c->peer_fb[1]); }
    cudaFree(c->stage[0]); cudaFree(c->stage[1]);
    cudaFree(c->ring); cudaFree(c->lookback); cudaFree(c->bounds); cudaFree(c->comp_order); cudaFree(c->comp_hint); cudaFree(c->pick_frame); cudaFree(c->fb); cudaFree(c->fb2); cudaFree(c->pick); cudaFree(c->staging);
    for (int i = 0; i < 2; ++i) { if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]); if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]); }
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    cudaFree(c->sync_word);
    for (int i = 0; i < c->grp.n_opened; ++i) cudaIpcCloseMemHandle(c->grp.opened[i]);
    cudaFree(c->grp.arena);
    cudaFree(c->unsorted_keys); cudaFree(c->unsorted_vals); cudaFree(c->trace); cudaFree(c->trace_count);
    if (c->ev) {
        for (int i = 0; i < GSR_HISTORY_FRAMES * EV_PER_FRAME; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
        delete[] c->ev;
    }
    if (c->ev_stat) {
        for (int i = 0; i < GSR_HISTORY_FRAMES; ++i) if (c->ev_stat[i]) cudaEventDestroy(c->ev_stat[i]);
        delete[] c->ev_stat;
    }
    if (c->host_ring) cudaFreeHost(c->host_ring);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

}  // namespace

extern "C" {

GSR_API const char *gsr_error_string(int code) {
    switch (code) {
        case GSR_OK: return "ok";
        case GSR_ERR_INVALID: return "invalid argument";
        case GSR_ERR_CUDA: return "CUDA failure or no usable sm_100 device (no CPU fallback exists)";
        case GSR_ERR_OOM: return "device out of memory";
        case GSR_ERR_STATE: return "call order violated";
        case GSR_ERR_OVERFLOW: return "duplicate list exceeded capacity";
        default: return "unknown error";
    }
}
GSR_API const char *gsr_last_error(void) { return g_last_error; }
GSR_API const char *gsr_version(void) { return "gsr 0.1.0 (sm_100a)"; }
GSR_API int gsr_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

GSR_API int gsr_create(const gsr_config *cfg, gsr_ctx **out) {
    if (!cfg || !out || cfg->max_splats == 0) { set_last_error("gsr_create: null config/out or max_splats == 0"); return GSR_ERR_INVALID; }
    *out = nullptr;
    int rc = check_device(cfg->device);
    if (rc) return rc;
    if ((rc = use_device(cfg->device))) return rc;
    if (cfg->max_splats >= (1ull << 32) - 256ull) { set_last_error("max_splats must be < 2^32-256"); return GSR_ERR_INVALID; }
    gsr_ctx *c = new (std::nothrow) gsr_ctx();
    if (!c) return GSR_ERR_OOM;
    c->device = cfg->device;
    c->flags = cfg->flags;
    if (!(c->flags & (GSR_FLAG_REFERENCE_QUIRKS | GSR_FLAG_FIXED_RANGES))) c->flags |= GSR_FLAG_REFERENCE_QUIRKS;
    c->max_splats = cfg->max_splats;
    const uint64_t factor = cfg->dup_capacity_factor ? cfg->dup_capacity_factor : 10;  // rasterizer.gd:79
    c->cap_factor = factor;
    c->capacity_max = (1ull << 30) - 1;  // look-back words carry 30-bit counts
    c->capacity = c->max_splats * factor;
    if (c->capacity > c->capacity_max) c->capacity = c->capacity_max;
    c->plane_stride = (c->max_splats + 255ull) & ~255ull;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, c->device);
    if ((rc = composite_max_ctas_per_sm(&c->comp_max_ctas))) { delete c; return rc; }

#define TRY_ALLOC(ptr, bytes)                                                                      \
    do {                                                                                           \
        cudaError_t _e = cudaMalloc((void **)&(ptr), (bytes));                                     \
        if (_e != cudaSuccess) {                                                                   \
            set_last_error("cudaMalloc(%s, %llu B) -> %s", #ptr, (unsigned long long)(bytes), cudaGetErrorString(_e)); \
            free_ctx(c);                                                                           \
            return _e == cudaErrorMemoryAllocation ? GSR_ERR_OOM : GSR_ERR_CUDA;                   \
        }                                                                                          \
    } while (0)

    cudaError_t se;
    {
        int least = 0, greatest = 0;
        cudaDeviceGetStreamPriorityRange(&least, &greatest);
        se = cudaStreamCreateWithPriority(&c->own_stream, cudaStreamNonBlocking, greatest);
    }
    if (se != cudaSuccess) { set_last_error("cudaStreamCreate -> %s", cudaGetErrorString(se)); free_ctx(c); return GSR_ERR_CUDA; }
    c->stream = c->own_stream;
    se = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (se == cudaSuccess) {   // the front stream yields to the render stream wherever the host gave that one a higher priority
        int least = 0, greatest = 0;
        cudaDeviceGetStreamPriorityRange(&least, &greatest);
        se = cudaStreamCreateWithPriority(&c->front_stream, cudaStreamNonBlocking, least);
    }
    for (int i = 0; i < 2 && se == cudaSuccess; ++i) {
        se = cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming);
        if (se == cudaSuccess) se = cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming);
    }
    if (se != cudaSuccess) { set_last_error("copy stream/events -> %s", cudaGetErrorString(se)); free_ctx(c); return GSR_ERR_CUDA; }
    TRY_ALLOC(c->soa, sizeof(float4) * NUM_PLANES * c->plane_stride);
    TRY_ALLOC(c->records, sizeof(float4) * 3ull * c->max_splats);
    TRY_ALLOC(c->records2, sizeof(float4) * 3ull * c->max_splats);
    c->cap_stride = (c->capacity + 1023ull) & ~1023ull;
    TRY_ALLOC(c->keys, sizeof(uint32_t) * 3ull * c->cap_stride);
    TRY_ALLOC(c->vals, sizeof(uint32_t) * 3ull * c->cap_stride);
    c->keys_cur = c->keys; c->vals_cur = c->vals; c->records_cur = c->records;
    c->lookback_blocks = projection_num_blocks((uint32_t)c->max_splats);  // one scan link per CTA
    TRY_ALLOC(c->ring, sizeof(FrameState) * GSR_HISTORY_FRAMES);
    TRY_ALLOC(c->lookback, sizeof(unsigned long long) * ((size_t)c->lookback_blocks + 2u * GROUP_MAX * GROUP_MAX));  // scatter mode: (N/G/256 + 1) x G links
    c->frame = c->ring;
    TRY_ALLOC(c->pick, sizeof(float4));
    TRY_ALLOC(c->sync_word, sizeof(int32_t));
    c->staging_splats = c->max_splats < (1ull << 18) ? c->max_splats : (1ull << 18);
    TRY_ALLOC(c->staging, sizeof(float4) * NUM_PLANES * c->staging_splats);
#undef TRY_ALLOC
    rc = sort_workspace_create(c->sort, c->capacity, /*need_alt_buffers=*/false);
    if (rc) { free_ctx(c); return rc; }
    c->ev = new (std::nothrow) cudaEvent_t[GSR_HISTORY_FRAMES * EV_PER_FRAME]();
    if (!c->ev) { free_ctx(c); return GSR_ERR_OOM; }
    for (int i = 0; i < GSR_HISTORY_FRAMES * EV_PER_FRAME; ++i) {
        if (cudaEventCreate(&c->ev[i]) != cudaSuccess) { set_last_error("cudaEventCreate failed"); free_ctx(c); return GSR_ERR_CUDA; }
    }
    c->ev_stat = new (std::nothrow) cudaEvent_t[GSR_HISTORY_FRAMES]();
    if (!c->ev_stat) { free_ctx(c); return GSR_ERR_OOM; }
    for (int i = 0; i < GSR_HISTORY_FRAMES; ++i) {
        if (cudaEventCreateWithFlags(&c->ev_stat[i], cudaEventDisableTiming) != cudaSuccess) { set_last_error("cudaEventCreate failed"); free_ctx(c); return GSR_ERR_CUDA; }
    }
    if (cudaHostAlloc((void **)&c->host_ring, sizeof(FrameState) * GSR_HISTORY_FRAMES, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
        set_last_error("cudaHostAlloc(frame mirror) failed"); c->host_ring = nullptr; free_ctx(c); return GSR_ERR_OOM;
    }
    memset(c->host_ring, 0, sizeof(FrameState) * GSR_HISTORY_FRAMES);
    cudaMemsetAsync(c->soa, 0, sizeof(float4) * NUM_PLANES * c->plane_stride, c->stream);
    cudaMemsetAsync(c->records, 0, sizeof(float4) * 3ull * c->max_splats, c->stream);
    cudaMemsetAsync(c->records2, 0, sizeof(float4) * 3ull * c->max_splats, c->stream);
    cudaMemsetAsync(c->pick, 0, sizeof(float4), c->stream);
    cudaMemsetAsync(c->sync_word, 0, sizeof(int32_t), c->stream);
    cudaMemsetAsync(c->ring, 0, sizeof(FrameState) * GSR_HISTORY_FRAMES, c->stream);
    // load every kernel now: with lazy module loading a FIRST launch may have to synchronise with the device, which must not
    // happen on the frame path (and would deadlock a group whose ranks share one process: a wait kernel spins meanwhile)
    if ((rc = preload_group_kernels()) || (rc = preload_projection_kernels()) || (rc = preload_sort_kernels()) || (rc = preload_ranges_kernels()) ||
        (rc = preload_ingest_kernels()) || (rc = preload_present_kernels()) || (rc = preload_composite_kernels())) { free_ctx(c); return rc; }
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { set_last_error("init sync -> %s", cudaGetErrorString(e)); free_ctx(c); return GSR_ERR_CUDA; }
    *out = c;
    return GSR_OK;
}

GSR_API int gsr_destroy(gsr_ctx *ctx) {
    free_ctx(ctx);
    return GSR_OK;
}

GSR_API int gsr_set_stream(gsr_ctx *c, void *cuda_stream) {
    if (!c) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    c->ev_valid = false; c->front_gate = nullptr;
    return GSR_OK;
}

GSR_API int gsr_upload_splats_aos(gsr_ctx *c, const float *splat60, uint64_t first, uint64_t count) {
    if (!c || (!splat60 && count)) return GSR_ERR_INVALID;
    if (count > c->max_splats || first > c->max_splats - count) { set_last_error("upload range [%llu,%llu) exceeds max_splats %llu", (unsigned long long)first, (unsigned long long)(first + count), (unsigned long long)c->max_splats); return GSR_ERR_INVALID; }
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));   // a projection in flight reads the planes this call rewrites
    uint64_t done = 0;
    while (done < count) {
        const uint64_t m = (count - done) < c->staging_splats ? (count - done) : c->staging_splats;
        GSR_CUDA_TRY(cudaMemcpyAsync(c->staging, splat60 + (done * 60ull), m * 240ull, cudaMemcpyHostToDevice, c->stream));
        if ((rc = launch_aos_to_soa(c->staging, m, c->soa, c->plane_stride, first + done, c->stream))) return rc;
        done += m;
    }
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));  // the caller may free/reuse splat60 (buffer_update semantics)
    if (first + count > c->num_splats) c->num_splats = first + count;
    return GSR_OK;
}

GSR_API int gsr_upload_ply_raw(gsr_ctx *c, const float *ply, uint32_t nprops, uint64_t first, uint64_t count, float creation_time) {
    if (!c || (!ply && count)) return GSR_ERR_INVALID;
    if (nprops < 62 || nprops > 256) { set_last_error("gsr_upload_ply_raw: %u properties; need the 62 standard 3DGS floats (x..rot_3) first", nprops); return GSR_ERR_INVALID; }
    if (count > c->max_splats || first > c->max_splats - count) { set_last_error("upload range [%llu,%llu) exceeds max_splats %llu", (unsigned long long)first, (unsigned long long)(first + count), (unsigned long long)c->max_splats); return GSR_ERR_INVALID; }
    int rc = use_device(c->device);
    if (rc) return rc;
    const uint64_t staging_floats = c->staging_splats * 60ull;  // the AoS staging buffer, reused for raw vertices
    const uint64_t per = staging_floats / nprops;
    if (per == 0) { set_last_error("gsr_upload_ply_raw: staging buffer too small"); return GSR_ERR_INVALID; }
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));   // a projection in flight reads the planes this call rewrites
    uint64_t done = 0;
    while (done < count) {
        const uint64_t m = (count - done) < per ? (count - done) : per;
        GSR_CUDA_TRY(cudaMemcpyAsync(c->staging, ply + done * nprops, m * nprops * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        if ((rc = launch_ply_to_soa(reinterpret_cast<const float *>(c->staging), nprops, m, creation_time, c->soa, c->plane_stride, first + done, c->stream))) return rc;
        done += m;
    }
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (first + count > c->num_splats) c->num_splats = first + count;
    return GSR_OK;
}

GSR_API int gsr_resize(gsr_ctx *c, int32_t width, int32_t height) {
    if (!c || width < 1 || height < 1) { set_last_error("gsr_resize: bad size %dx%d", width, height); return GSR_ERR_INVALID; }
    const int tx = (width + TILE - 1) / TILE, ty = (height + TILE - 1) / TILE;
    if ((int64_t)tx * ty * c->num_views > 65536) {  // tile id must fit the 16 key bits above the depth code (gsplat_projection.glsl:222)
        set_last_error("gsr_resize: %d views x %d tiles exceed the 16-bit tile id of the sort key", c->num_views, tx * ty);
        return GSR_ERR_INVALID;
    }
    const size_t K = (size_t)c->num_views;
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->front_gate = nullptr;
    c->width = c->height = c->tiles_x = c->tiles_y = 0;  // a failure below leaves the context in the "before gsr_resize" state
    cudaFree(c->bounds); c->bounds = nullptr;
    cudaFree(c->comp_order); c->comp_order = nullptr;
    cudaFree(c->comp_hint); c->comp_hint = nullptr;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    cudaFree(c->fb); c->fb = nullptr;
    cudaFree(c->fb2); c->fb2 = nullptr;
    cudaFree(c->stage[0]); cudaFree(c->stage[1]); c->stage[0] = c->stage[1] = nullptr;
    c->fb_last = nullptr; c->copied_valid[0] = c->copied_valid[1] = false;
    // peer mode refers to the frames freed above (exported) or to another process's frames of the old size (imported): drop it.
    // The host must export / import again after a resize (every rank resizes, then the presenting rank re-exports).
    if (c->peer_opened) { cudaIpcCloseMemHandle(c->peer_fb[0]); cudaIpcCloseMemHandle(c->peer_fb[1]); c->peer_opened = false; }
    c->peer_mode = false; c->peer_fb[0] = c->peer_fb[1] = nullptr; c->peer_counter = 0; c->async_counter = 0;
    group_detach(c);   // same for a shard group: every rank resizes, exports and attaches again
    GSR_CUDA_TRY(cudaMalloc((void **)&c->bounds, sizeof(uint2) * (size_t)tx * ty * K));
    GSR_CUDA_TRY(cudaMalloc((void **)&c->comp_order, sizeof(uint32_t) * (size_t)tx * ty * K));
    GSR_CUDA_TRY(cudaMalloc((void **)&c->comp_hint, sizeof(uint32_t) * (size_t)tx * ty * K));
    GSR_CUDA_TRY(cudaMemsetAsync(c->comp_hint, 0, sizeof(uint32_t) * (size_t)tx * ty * K, c->stream));
    c->comp_hint_key = 0;
    if (!c->pick_frame) GSR_CUDA_TRY(cudaMalloc((void **)&c->pick_frame, sizeof(FrameState)));
    GSR_CUDA_TRY(cudaMalloc((void **)&c->fb, sizeof(float4) * (size_t)width * height * K));
    GSR_CUDA_TRY(cudaMalloc((void **)&c->fb2, sizeof(float4) * (size_t)width * height * K));
    GSR_CUDA_TRY(cudaMemsetAsync(c->fb, 0, sizeof(float4) * (size_t)width * height * K, c->stream));
    GSR_CUDA_TRY(cudaMemsetAsync(c->fb2, 0, sizeof(float4) * (size_t)width * height * K, c->stream));
    c->width = width; c->height = height; c->tiles_x = tx; c->tiles_y = ty;
    if (!c->band_set) { c->band_y0 = 0; c->band_y1 = ty; }
    if (c->band_y1 > ty) c->band_y1 = ty;
    if (c->band_y0 > c->band_y1) c->band_y0 = c->band_y1;
    return GSR_OK;
}

GSR_API int gsr_set_row_interleave(gsr_ctx *c, int32_t row_rem, int32_t row_mod) {
    if (!c || row_mod < 1 || row_rem < 0 || row_rem >= row_mod) { set_last_error("gsr_set_row_interleave: need 0 <= rem < mod"); return GSR_ERR_INVALID; }
    if (c->num_views > 1 && row_mod > 1) return refuse_multiview("gsr_set_row_interleave");
    c->row_mod = row_mod; c->row_rem = row_rem;
    return GSR_OK;
}

GSR_API void *gsr_band_sync_word(gsr_ctx *c) { return c ? (void *)c->sync_word : nullptr; }

GSR_API int gsr_band_fixup(gsr_ctx *c) {
    if (!c) return GSR_ERR_INVALID;
    if (c->row_mod <= 1 || !c->fb_last) return GSR_OK;  // exact modes resolve the quirk inside tile_ranges_kernel
    if (c->flags & GSR_FLAG_FIXED_RANGES) return GSR_OK;
    int rc = use_device(c->device);
    if (rc) return rc;
    return launch_band_fixup(c->sync_word, c->fb_last, c->width, c->height, c->tiles_x, c->tiles_x * c->tiles_y, c->band_y0, c->band_y1,
                             c->row_mod, c->row_rem, c->stream);
}

GSR_API int gsr_set_band(gsr_ctx *c, int32_t row_begin, int32_t row_end) {
    if (!c || c->tiles_y == 0) { set_last_error("gsr_set_band before gsr_resize"); return GSR_ERR_STATE; }
    if (row_begin < 0 || row_end > c->tiles_y || row_begin > row_end) { set_last_error("band [%d,%d) outside [0,%d]", row_begin, row_end, c->tiles_y); return GSR_ERR_INVALID; }
    if (c->num_views > 1 && !(row_begin == 0 && row_end == c->tiles_y)) return refuse_multiview("gsr_set_band");
    c->band_y0 = row_begin; c->band_y1 = row_end;
    c->band_set = !(row_begin == 0 && row_end == c->tiles_y);
    return GSR_OK;
}

static int grow_capacity(gsr_ctx *c, uint64_t want);

GSR_API int gsr_set_views(gsr_ctx *c, int32_t num_views) {
    if (!c || num_views < 1 || num_views > GSR_MAX_VIEWS) { set_last_error("gsr_set_views: need a context and 1 <= views <= %d", GSR_MAX_VIEWS); return GSR_ERR_INVALID; }
    if ((int64_t)c->tiles_x * c->tiles_y * num_views > 65536) {
        set_last_error("gsr_set_views: %d views x %d tiles exceed the 16-bit tile id of the sort key", num_views, c->tiles_x * c->tiles_y);
        return GSR_ERR_INVALID;
    }
    if (num_views > 1 && (c->grp.world > 1 || c->peer_mode || c->band_set || !(c->band_y0 == 0 && c->band_y1 == c->tiles_y) || c->row_mod > 1 ||
                          c->overlap > 0)) {
        set_last_error("gsr_set_views: multiview needs a single-GPU full-frame context (no shard group, peer frames, band, row interleave or overlap)");
        return GSR_ERR_STATE;
    }
    if (num_views == c->num_views) return GSR_OK;
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    // one record table per view, in each of the two alternating sets
    cudaFree(c->records); cudaFree(c->records2);
    c->records = c->records2 = c->records_cur = nullptr;
    const size_t rec_bytes = sizeof(float4) * 3ull * c->max_splats * (size_t)num_views;
    GSR_CUDA_TRY(cudaMalloc((void **)&c->records, rec_bytes));
    GSR_CUDA_TRY(cudaMalloc((void **)&c->records2, rec_bytes));
    GSR_CUDA_TRY(cudaMemsetAsync(c->records, 0, rec_bytes, c->stream));
    GSR_CUDA_TRY(cudaMemsetAsync(c->records2, 0, rec_bytes, c->stream));
    c->records_cur = c->records;
    c->num_views = num_views;
    // K-layer frames, K*T bounds / compositor order / hints (the hints are dropped)
    if (c->width > 0 && (rc = gsr_resize(c, c->width, c->height))) return rc;
    // every view brings its own duplicates: start from K x factor x N, like K single-view contexts (grows on demand as before)
    return grow_capacity(c, (uint64_t)num_views * c->cap_factor * c->max_splats);
}

// Per-frame constants of the projection: project_covariance's focal / limit terms and the norm bound of the conservative reject.
static void frame_constants(const float *view_proj, const Uniforms &u, ProjectionArgs &pa) {
    {   // per-frame constants of project_covariance, same IEEE binary32 operations as gsplat_projection.glsl:127-133
        const float tfi0 = view_proj[16 + 0], tfi1 = view_proj[16 + 5];
        const volatile float hw = (float)u.dims[0] * 0.5f, hh = (float)u.dims[1] * 0.5f;
        const volatile float f0 = hw * tfi0, f1 = hh * tfi1;
        const volatile float t0 = 1.0f / tfi0, t1 = 1.0f / tfi1;
        const volatile float n0 = -t0, n1 = -t1;
        pa.focal_base[0] = f0; pa.focal_base[1] = f1;
        pa.lim_lo[0] = n0 * 1.3f; pa.lim_lo[1] = n1 * 1.3f;
        pa.lim_hi[0] = t0 * 1.3f; pa.lim_hi[1] = t1 * 1.3f;
    }
    {   // |W|_2^2 <= |W^T W|_inf (largest absolute row sum of the Gram matrix); exactly 1 for a rigid camera
        float g[3][3];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                g[i][j] = 0.0f;
                for (int r = 0; r < 3; ++r) g[i][j] += view_proj[4 * i + r] * view_proj[4 * j + r];
            }
        float nrm = 0.0f;
        for (int i = 0; i < 3; ++i) {
            float row = 0.0f;
            for (int j = 0; j < 3; ++j) row += g[i][j] < 0.0f ? -g[i][j] : g[i][j];
            nrm = row > nrm ? row : nrm;
        }
        pa.w_frob2 = nrm * 1.0001f;
    }
}

// ---- dynamic duplicate capacity ------------------------------------------------------------------------------------------
static int grow_capacity(gsr_ctx *c, uint64_t want) {
    if (want > c->capacity_max) want = c->capacity_max;
    if (want <= c->capacity) return GSR_OK;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    c->front_gate = nullptr;
    cudaFree(c->keys); cudaFree(c->vals); c->keys = c->vals = c->keys_cur = c->vals_cur = nullptr;
    sort_workspace_destroy(c->sort);
    const bool unsorted = c->unsorted_keys != nullptr;
    cudaFree(c->unsorted_keys); cudaFree(c->unsorted_vals); c->unsorted_keys = c->unsorted_vals = nullptr;
    c->capacity = want;
    c->cap_stride = (c->capacity + 1023ull) & ~1023ull;
    GSR_CUDA_TRY(cudaMalloc((void **)&c->keys, sizeof(uint32_t) * 3ull * c->cap_stride));
    GSR_CUDA_TRY(cudaMalloc((void **)&c->vals, sizeof(uint32_t) * 3ull * c->cap_stride));
    c->keys_cur = c->keys; c->vals_cur = c->vals;
    if (unsorted) {
        GSR_CUDA_TRY(cudaMalloc((void **)&c->unsorted_keys, sizeof(uint32_t) * c->capacity));
        GSR_CUDA_TRY(cudaMalloc((void **)&c->unsorted_vals, sizeof(uint32_t) * c->capacity));
    }
    return sort_workspace_create(c->sort, c->capacity, /*need_alt_buffers=*/false);
}

// Examine the mirrors of the frames that have completed since the last call (no host sync: event queries) and grow the
// capacity once M has used more than half of it -- an overflow then needs M to more than double from one frame to the next.
static int track_capacity(gsr_ctx *c) {
    if (c->flags & GSR_FLAG_STATIC_CAPACITY) return GSR_OK;
    while (c->stats_polled < c->frame_counter) {
        if (c->frame_counter - c->stats_polled > GSR_HISTORY_FRAMES) { c->stats_polled = c->frame_counter - GSR_HISTORY_FRAMES; continue; }
        const uint32_t slot = (uint32_t)(c->stats_polled % GSR_HISTORY_FRAMES);
        if (cudaEventQuery(c->ev_stat[slot]) != cudaSuccess) { cudaGetLastError(); break; }
        const uint64_t m = c->host_ring[slot].dup_total;
        if (m > c->m_high) c->m_high = m;
        c->stats_polled += 1;
    }
    if (c->m_high * 2ull > c->capacity && c->capacity < c->capacity_max) return grow_capacity(c, c->m_high * 3ull);
    return GSR_OK;
}

struct GroupFrame { uint32_t seq; int parity; int rows_local; };

// GPU time of one frame's stages from its events: 'Projection' = front part (clear + projection kernel, on the front stream when frames
// overlap) + receive (group mode: segment wait + gather); total = the sum of the stages = GPU time attributable to the frame (with
// overlap the frame PERIOD is shorter than that: the front part runs beside the previous frame's compositor).
static int stage_times(gsr_ctx *c, uint32_t slot, float out[5], float *front_ms) {
    cudaEvent_t *ev = c->ev + EV_PER_FRAME * slot;
    float front = 0.f, recv = 0.f;
    GSR_CUDA_TRY(cudaEventElapsedTime(&front, ev[0], ev[1]));
    GSR_CUDA_TRY(cudaEventElapsedTime(&recv, ev[2], ev[3]));
    out[0] = front + recv;
    for (int i = 1; i < 4; ++i) GSR_CUDA_TRY(cudaEventElapsedTime(&out[i], ev[2 + i], ev[3 + i]));
    out[4] = out[0] + out[1] + out[2] + out[3];
    if (front_ms) *front_ms = front;
    return GSR_OK;
}

// arena layout (identical on every rank of a group: same max_splats, same rx_capacity)
// (`parity` = frame phase seq % GROUP_PHASES)
static size_t arena_rx_keys_off(uint64_t cap, int parity) { return GROUP_FLAGS_BYTES + sizeof(uint32_t) * cap * (size_t)parity; }
static size_t arena_rx_vals_off(uint64_t cap, int parity) { return GROUP_FLAGS_BYTES + sizeof(uint32_t) * cap * (size_t)(GROUP_PHASES + parity); }
static size_t arena_records_off(uint64_t cap, uint64_t max_splats, int parity) { return GROUP_FLAGS_BYTES + sizeof(uint32_t) * cap * 2 * GROUP_PHASES + sizeof(float4) * 3ull * max_splats * (size_t)parity; }
static size_t arena_bytes(uint64_t cap, uint64_t max_splats) { return arena_records_off(cap, max_splats, GROUP_PHASES); }

static GroupPeers group_peers(const gsr_ctx *c, int parity) {
    (void)parity;
    GroupPeers p;
    memset(&p, 0, sizeof p);
    p.world = c->grp.world; p.rank = c->grp.rank;
    for (int r = 0; r < c->grp.world; ++r) p.flags[r] = c->grp.flags[r];
    return p;
}

static int render_enqueue(gsr_ctx *c, const float *view_proj, const void *uniforms32, float heatmap_factor, float4 *target = nullptr,
                          const GroupFrame *gf = nullptr) {
    if (!c || !view_proj || !uniforms32) return GSR_ERR_INVALID;
    if (c->width == 0) { set_last_error("gsr_render before gsr_resize"); return GSR_ERR_STATE; }
    const int K = c->num_views;   // view_proj / uniforms32: K push constants / uniform blocks
    Uniforms u;
    memcpy(&u, uniforms32, sizeof u);
    if (u.dims[0] != c->width || u.dims[1] != c->height) {
        set_last_error("uniform dims %dx%d differ from gsr_resize %dx%d", u.dims[0], u.dims[1], c->width, c->height);
        return GSR_ERR_INVALID;
    }
    for (int v = 1; v < K; ++v) {   // the fused projection shares the time factors, scaled covariance and opacity between views
        Uniforms uv;
        memcpy(&uv, static_cast<const char *>(uniforms32) + sizeof(Uniforms) * v, sizeof uv);
        if (memcmp(&uv.model_scale, &u.model_scale, sizeof u.model_scale) || memcmp(uv.dims, u.dims, sizeof u.dims) || memcmp(&uv.time, &u.time, sizeof u.time)) {
            set_last_error("uniform block of view %d differs from view 0 in model_scale, width, height or time", v);
            return GSR_ERR_INVALID;
        }
    }
    int rc = use_device(c->device);
    if (rc) return rc;
    if ((rc = track_capacity(c))) return rc;
    cudaStream_t s = c->stream;
    // Front / back overlap.  The front part of a frame (clear + projection: HBM-bound) needs nothing from the frame before it, the back
    // part (sort, ranges, compositor) nothing from the frame after it.  With overlap on, the front part runs on its own stream and
    // is released when the PREVIOUS frame's tile ranges are done: it then shares the GPU with that frame's compositor (FMA-pipe /
    // chain bound, 1-2 small CTAs per SM), which leaves the memory system idle.  Consecutive frames alternate between two sort
    // inputs and two record tables; the back part waits for its own front part.  A host that renders one frame at a time
    // (gsr_render) sees the same kernels in the same order.
    const bool overlap = c->overlap > 0 && c->front_stream != nullptr;
    cudaStream_t fs = overlap ? c->front_stream : s;
    int launches = 0;
    const uint32_t slot = (uint32_t)(c->frame_counter % GSR_HISTORY_FRAMES);
    c->frame = c->ring + slot;
    cudaEvent_t *ev = c->ev + EV_PER_FRAME * slot;
    const int half = (int)(c->frame_counter & 1u);
    uint32_t *keys_in = c->keys + (size_t)half * c->cap_stride, *vals_in = c->vals + (size_t)half * c->cap_stride;
    uint32_t *keys_alt = c->keys + 2ull * c->cap_stride, *vals_alt = c->vals + 2ull * c->cap_stride;
    float4 *records = half ? c->records2 : c->records;
    const uint32_t n_tiles = (uint32_t)frame_tiles(c);

    // ---- front: rasterizer.gd:127-128 (clear M = this frame's history slot + the scan links), then the projection ----
    if (overlap && c->front_gate) GSR_CUDA_TRY(cudaStreamWaitEvent(fs, c->front_gate, 0));
    {
        uint32_t links = projection_num_blocks((uint32_t)c->max_splats);
        if (gf) {
            const uint64_t first = (uint64_t)c->grp.rank * c->grp.slice;
            const uint64_t count = first < c->max_splats ? ((c->max_splats - first) < c->grp.slice ? (c->max_splats - first) : c->grp.slice) : 0;
            links = projection_scatter_blocks((uint32_t)count) * (uint32_t)c->grp.world;
        }
        // serial: one kernel clears the tile bounds as well; overlapped: the bounds belong to the back part (the previous frame's
        // compositor may still read them)
        if ((rc = launch_frame_clear(c->frame, c->lookback, links, overlap ? nullptr : c->bounds, overlap ? 0u : n_tiles, fs))) return rc;
        launches += 1;
    }
    GSR_CUDA_TRY(cudaEventRecord(ev[0], fs));  // 'Start'

    ProjectionArgs pa;
    // the reference dispatches over splat_buffer.length() = point_cloud.size every frame (rasterizer.gd:83,134), i.e. also over the
    // zero-initialised structs of splats the loader has not delivered yet: so does libgsr (the SoA planes start zeroed)
    pa.soa = c->soa; pa.plane_stride = c->plane_stride; pa.num_splats = (uint32_t)c->max_splats;
    memcpy(pa.vp, view_proj, sizeof pa.vp);
    pa.u = u;
    frame_constants(view_proj, u, pa);
    const bool fast = c->row_mod > 1 && !gf;   // group mode is exact: the frame-global last tile travels with the pairs
    pa.band_y0 = c->band_y0; pa.band_y1 = c->band_y1;
    pa.row_mod = c->row_mod; pa.row_rem = c->row_rem;
    // Conservative early reject + compaction of the survivors over 1024-splat CTAs (projection_sharded_kernel): exact, and
    // measured on B200 (c3, one rank of G emulated): G=8 0.39 vs 0.46 ms, G=4 equal, G=2 slower (with two ranks nearly every
    // splat's conservative extent touches both).  So: on by default from 6 ranks, or on request (GSR_FLAG_FAST_REJECT).
    const bool want_reject = (c->flags & GSR_FLAG_FAST_REJECT) != 0 || c->row_mod >= 6;
    pa.fast_reject = (want_reject && fast) ? 1 : 0;
    pa.fast_mode = fast ? 1 : 0;
    // full frame: 12 of 32 lanes (below that, per-lane 128-bit gathers move fewer bytes); sharded: few lanes of a warp land in
    // this rank's rows and the latency-bound gather path was measured slower than fetching the whole 6 KB slice (0.60 vs 0.46 ms)
    pa.sh_bulk_min = (fast || c->row_mod > 1) ? 1 : 12;
    pa.records = records; pa.keys = keys_in; pa.values = vals_in; pa.capacity = (uint32_t)c->capacity;
    pa.lookback = c->lookback; pa.frame = c->frame;
    if (gf) {
        // group mode: the projection is sharded by SPLATS.  This rank projects its slice and stores every pair and record into the
        // memory of the rank that owns it (peer stores over NVLink); the back part then waits for the other sources' flags and packs
        // what it received -- its own rows' pairs of ALL splats, in splat-id order -- into the sort input.
        const int G = c->grp.world;
        ScatterPeers sp;
        memset(&sp, 0, sizeof sp);
        sp.world = G; sp.rank = c->grp.rank; sp.parity = gf->parity; sp.seq = gf->seq;
        const uint64_t first = (uint64_t)c->grp.rank * c->grp.slice;
        sp.first = (uint32_t)(first < c->max_splats ? first : c->max_splats);
        sp.count = (uint32_t)(first < c->max_splats ? ((c->max_splats - first) < c->grp.slice ? (c->max_splats - first) : c->grp.slice) : 0);
        sp.seg_cap = c->grp.seg_cap;
        for (int d = 0; d < G; ++d) {
            char *ar = c->grp.peer_arena[d];
            sp.records[d] = reinterpret_cast<float4 *>(ar + arena_records_off(c->grp.rx_capacity, c->max_splats, gf->parity));
            sp.keys[d] = reinterpret_cast<uint32_t *>(ar + arena_rx_keys_off(c->grp.rx_capacity, gf->parity)) + (size_t)c->grp.rank * c->grp.seg_cap;
            sp.values[d] = reinterpret_cast<uint32_t *>(ar + arena_rx_vals_off(c->grp.rx_capacity, gf->parity)) + (size_t)c->grp.rank * c->grp.seg_cap;
            sp.flags[d] = c->grp.flags[d];
        }
        sp.lookback = c->lookback;
        if ((rc = launch_projection_scatter(pa, sp, fs))) return rc;
        launches += 1;
    } else if (K > 1) {
        ViewsArgs va;
        memset(&va, 0, sizeof va);
        va.num_views = K; va.tiles_per_view = (uint32_t)(c->tiles_x * c->tiles_y);
        for (int v = 0; v < K; ++v) {
            ProjectionArgs &pv = va.view[v];
            pv = pa;
            memcpy(pv.vp, view_proj + 32 * v, sizeof pv.vp);
            memcpy(&pv.u, static_cast<const char *>(uniforms32) + sizeof(Uniforms) * v, sizeof pv.u);
            frame_constants(view_proj + 32 * v, pv.u, pv);
            pv.records = records + 3ull * c->max_splats * (uint64_t)v;
        }
        if ((rc = launch_projection_views(va, fs))) return rc;
        launches += pa.num_splats ? 1 : 0;
    } else {
        if ((rc = launch_projection(pa, fs))) return rc;
        launches += pa.num_splats ? 1 : 0;
    }
    GSR_CUDA_TRY(cudaEventRecord(ev[1], fs));  // end of the front part

    // ---- back ----
    if (overlap) {
        GSR_CUDA_TRY(cudaStreamWaitEvent(s, ev[1], 0));
        if ((rc = launch_frame_clear(nullptr, nullptr, 0u, c->bounds, n_tiles, s))) return rc;
        launches += 1;
    }
    GSR_CUDA_TRY(cudaEventRecord(ev[2], s));
    if (gf) {
        const int G = c->grp.world;
        char *mine = c->grp.peer_arena[c->grp.rank];
        if ((rc = launch_group_wait_segments(c->grp.flags[c->grp.rank], gf->parity, G, gf->seq, c->grp.seg_cap, (uint32_t)c->capacity, c->frame, s))) return rc;
        if ((rc = launch_gather_segments(c->grp.flags[c->grp.rank], G, c->grp.seg_cap,
                                         reinterpret_cast<const uint32_t *>(mine + arena_rx_keys_off(c->grp.rx_capacity, gf->parity)),
                                         reinterpret_cast<const uint32_t *>(mine + arena_rx_vals_off(c->grp.rx_capacity, gf->parity)), keys_in, vals_in,
                                         c->sm_count * 8, s))) return rc;
        records = reinterpret_cast<float4 *>(mine + arena_records_off(c->grp.rx_capacity, c->max_splats, gf->parity));
        launches += 2;
    }
    c->keys_cur = keys_in; c->vals_cur = vals_in; c->records_cur = records;
    GSR_CUDA_TRY(cudaEventRecord(ev[3], s));  // 'Projection' = front + receive

    if (c->keep_unsorted) {
        GSR_CUDA_TRY(cudaMemcpyAsync(c->unsorted_keys, keys_in, sizeof(uint32_t) * c->capacity, cudaMemcpyDeviceToDevice, s));
        GSR_CUDA_TRY(cudaMemcpyAsync(c->unsorted_vals, vals_in, sizeof(uint32_t) * c->capacity, cudaMemcpyDeviceToDevice, s));
    }
    const uint32_t *m_ptr = reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(c->frame) + offsetof(FrameState, dup_sorted));
    if ((rc = sort_pairs_device(c->sort, keys_in, vals_in, m_ptr, keys_alt, vals_alt, s, &launches))) return rc;
    GSR_CUDA_TRY(cudaEventRecord(ev[4], s));  // 'Sort'

    const int sharded = fast ? 2 : ((!(c->band_y0 == 0 && c->band_y1 == c->tiles_y) || c->row_mod > 1) ? 1 : 0);
    if (fast) GSR_CUDA_TRY(cudaMemsetAsync(c->sync_word, 0, sizeof(int32_t), s));
    const int quirks = (c->flags & GSR_FLAG_FIXED_RANGES) ? 0 : 1;
    if (K > 1) rc = launch_tile_ranges_views(keys_in, c->frame, c->bounds, (uint32_t)(c->tiles_x * c->tiles_y), quirks, c->sm_count * 8, s);
    else rc = launch_tile_ranges(keys_in, c->frame, c->bounds, n_tiles, quirks, sharded, fast ? c->sync_word : nullptr, c->sm_count * 8, s);
    if (rc) return rc;
    launches += 1;
    GSR_CUDA_TRY(cudaEventRecord(ev[5], s));  // 'Boundaries'
    c->front_gate = ev[5];   // the next frame's front part may start here, beside this frame's compositor

    CompositeArgs ca;
    float4 *out_fb = c->fb_ext ? c->fb_ext : (target ? target : c->fb);
    // a pipelined read-back of this buffer may still be in flight on the copy stream (gsr_render_async followed by gsr_render)
    for (int i = 0; i < 2; ++i) {
        const float4 *owned = c->peer_mode ? c->peer_fb[i] : (i ? c->fb2 : c->fb);
        if (c->copied_valid[i] && owned == out_fb) GSR_CUDA_TRY(cudaStreamWaitEvent(s, c->ev_copied[i], 0));
    }
    c->fb_last = out_fb;
    ca.records = records; ca.values = vals_in; ca.bounds = c->bounds; ca.out = out_fb;
    ca.width = c->width; ca.height = c->height; ca.tiles_x = c->tiles_x;
    {   // owned tile rows: band rows with row % row_mod == row_rem
        int first = c->band_y0 + ((c->row_rem - c->band_y0 % c->row_mod) + c->row_mod) % c->row_mod;
        int nrows = first < c->band_y1 ? (c->band_y1 - 1 - first) / c->row_mod + 1 : 0;
        ca.tile_begin = first * c->tiles_x;
        ca.row_step = c->row_mod;
        ca.num_tiles = nrows * c->tiles_x * K;   // K > 1: full frame (no band, no rows), so the owned tiles are all K*T
    }
    ca.tiles_per_view = K > 1 ? c->tiles_x * c->tiles_y : 0;
    ca.layer_stride = (uint64_t)c->width * c->height;
    ca.record_stride = 3ull * c->max_splats;
    ca.heatmap_factor = heatmap_factor;
    ca.target_tile_id = 0xFFFFFFFFu;  // rasterizer.gd:158
    ca.pick = c->pick;
    ca.frame = c->frame; ca.count_staged = 1;
    ca.order = nullptr; ca.consumed = c->comp_hint;
    ca.ctas_per_sm = c->comp_ctas_per_sm < c->comp_max_ctas ? c->comp_ctas_per_sm : c->comp_max_ctas; ca.sm_count = c->sm_count;
    ca.contract = (c->flags & GSR_FLAG_UNCONTRACTED_BLEND) ? 0 : 1;
    {   // the hints describe the owned-tile indexing of the frame that wrote them: drop them when the ownership changes
        const uint64_t key = ((uint64_t)(uint32_t)ca.tile_begin << 32) ^ ((uint64_t)(uint32_t)ca.row_step << 24) ^ (uint64_t)(uint32_t)ca.num_tiles;
        if (key != c->comp_hint_key) { GSR_CUDA_TRY(cudaMemsetAsync(c->comp_hint, 0, sizeof(uint32_t) * frame_tiles(c), s)); c->comp_hint_key = key; }
    }
    if (c->comp_order_mode && ca.num_tiles > 0) {   // longest chains first: the long sequential chains start at once instead of in the tail
        if ((rc = launch_tile_order(c->bounds, ca.tile_begin, ca.row_step, ca.tiles_x, ca.num_tiles, c->comp_hint, c->comp_order, c->frame,
                                    (uint32_t)(c->comp_sparse_per_sm * c->sm_count), (uint32_t)c->sm_count, s))) return rc;
        ca.order = c->comp_order;
        launches += 1;
    }
    ca.trace = c->trace; ca.trace_count = c->trace_count; ca.trace_cap = c->trace_cap;
    if (c->trace) GSR_CUDA_TRY(cudaMemsetAsync(c->trace_count, 0, sizeof(uint32_t), s));
    if (gf && !gf->rows_local && c->grp.rank != 0 && gf->seq >= 3u) {   // the presenting rank must have consumed the frame that used this slot
        if ((rc = launch_group_wait_released(c->grp.flags[c->grp.rank], gf->seq - 2u, s))) return rc;
        launches += 1;
    }
    if ((rc = launch_composite(ca, s))) return rc;
    launches += ca.num_tiles > 0 ? 1 : 0;
    if (gf && !gf->rows_local) {   // rows have landed in the presenting rank's frame: tell it (system-scope flag store after the kernel boundary)
        if ((rc = launch_group_signal_done(group_peers(c, gf->parity), 0, c->grp.rank, gf->seq, s))) return rc;
        launches += 1;
    }
    GSR_CUDA_TRY(cudaEventRecord(ev[6], s));  // 'Render'
    // this frame's counters (M, overflow, C) to the pinned mirror: what track_capacity() reads without ever syncing
    // (a 16-byte-store kernel into mapped pinned memory, NOT a cudaMemcpyAsync: a D2H copy on the render stream would queue behind the
    // frame read-back on the copy engine and serialise the two streams)
    if ((rc = launch_publish_frame_state(c->frame, c->host_ring + slot, s))) return rc;
    GSR_CUDA_TRY(cudaEventRecord(c->ev_stat[slot], s));
    c->ev_valid = true;
    c->frame_counter += 1;
    c->last_launches = (uint32_t)launches;
    return GSR_OK;
}

static int render_sync_impl(gsr_ctx *c, const float *view_proj, const void *uniforms32, float heatmap_factor, float *out_host) {
    if (c && c->grp.world > 1) { set_last_error("gsr_render: a context attached to a group renders with gsr_render_async (all ranks, same frame)"); return GSR_ERR_STATE; }
    int rc = render_enqueue(c, view_proj, uniforms32, heatmap_factor);
    if (rc) return rc;
    if (out_host) {
        // synchronous path: a frame that overflowed the duplicate capacity is never returned -- grow and render it again
        // (the reference truncates silently: rasterizer.gd:79, main.gd:100; GSR_FLAG_STATIC_CAPACITY keeps that behaviour)
        for (int attempt = 0; attempt < 8 && !(c->flags & GSR_FLAG_STATIC_CAPACITY); ++attempt) {
            const uint32_t slot = (uint32_t)((c->frame_counter - 1) % GSR_HISTORY_FRAMES);
            GSR_CUDA_TRY(cudaEventSynchronize(c->ev_stat[slot]));
            const FrameState &fs = c->host_ring[slot];
            if (!fs.overflow || c->capacity >= c->capacity_max) break;
            if ((rc = grow_capacity(c, fs.dup_total + fs.dup_total / 4ull + 1024ull))) return rc;
            if ((rc = render_enqueue(c, view_proj, uniforms32, heatmap_factor))) return rc;
        }
        GSR_CUDA_TRY(cudaMemcpyAsync(out_host, framebuffer(c), sizeof(float4) * frame_pixels(c), cudaMemcpyDeviceToHost, c->stream));
        GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    }
    return GSR_OK;
}

GSR_API int gsr_render(gsr_ctx *c, const float view_proj[32], const void *uniforms32, float heatmap_factor, float *out_host) {
    if (c && c->num_views > 1) return refuse_multiview("gsr_render (use gsr_render_views)");
    return render_sync_impl(c, view_proj, uniforms32, heatmap_factor, out_host);
}

GSR_API int gsr_render_views(gsr_ctx *c, const float *view_proj, const void *uniforms, float heatmap_factor, float *out_host) {
    return render_sync_impl(c, view_proj, uniforms, heatmap_factor, out_host);
}

static int readback_enqueue(gsr_ctx *c, float4 *frame, int slot, void *pinned_host, int format, uint32_t group_seq = 0) {
    const size_t pixels = frame_pixels(c);
    const size_t bpp = present_bytes_per_pixel(format);
    if (!bpp) { set_last_error("unknown output format 0x%x", format); return GSR_ERR_INVALID; }
    int rc;
    const bool convert = format != GSR_OUT_RGBA32F;
    if (convert && !c->stage[slot]) GSR_CUDA_TRY(cudaMalloc(&c->stage[slot], sizeof(float4) * pixels + 64));
    GSR_CUDA_TRY(cudaEventRecord(c->ev_done[slot], c->stream));
    GSR_CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->ev_done[slot], 0));
    // group mode: the other ranks' rows arrive over NVLink; their done flags gate the copy (device-side wait on the copy stream)
    if (group_seq && (rc = launch_group_wait_done(c->grp.flags[c->grp.rank], c->grp.world, group_seq, c->copy_stream))) return rc;
    if (convert) {
        if ((rc = launch_present(frame, c->stage[slot], pixels, format, c->copy_stream))) return rc;
        GSR_CUDA_TRY(cudaMemcpyAsync(pinned_host, c->stage[slot], bpp * pixels, cudaMemcpyDeviceToHost, c->copy_stream));
    } else {
        GSR_CUDA_TRY(cudaMemcpyAsync(pinned_host, frame, sizeof(float4) * pixels, cudaMemcpyDeviceToHost, c->copy_stream));
    }
    GSR_CUDA_TRY(cudaEventRecord(c->ev_copied[slot], c->copy_stream));
    c->copied_valid[slot] = true;
    return GSR_OK;
}

static int render_async_impl(gsr_ctx *c, const float *view_proj, const void *uniforms32, float heatmap_factor, void *pinned_host, int format) {
    if (!c) return GSR_ERR_INVALID;
    if (c->grp.world > 1) {   // shard group: every rank enqueues the same frame; rows land in the presenting rank's frames
        if (pinned_host) { set_last_error("group mode: render with a NULL host pointer on every rank, then gsr_readback_async on rank 0"); return GSR_ERR_STATE; }
        int rc = use_device(c->device);
        if (rc) return rc;
        GroupFrame gf;
        gf.seq = c->grp.seq + 1u; gf.parity = (int)(gf.seq % (uint32_t)GROUP_PHASES);
        const int slot = (int)((gf.seq - 1u) & 1u);
        gf.rows_local = c->grp.present_rows;
        float4 *target = c->grp.root_fb[slot];
        if (gf.rows_local) {   // every rank presents its own rows (host consumer, one PCIe link per GPU): only its own read-back gates the slot
            target = slot ? c->fb2 : c->fb;   // (render_enqueue orders the compositor after the slot's read-back)
        } else if (c->grp.rank == 0) {
            if (c->copied_valid[slot]) GSR_CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_copied[slot], 0));
            if (gf.seq >= 3u && (rc = launch_group_release(group_peers(c, gf.parity), c->grp.world, gf.seq - 2u, c->stream))) return rc;
        }
        if ((rc = render_enqueue(c, view_proj, uniforms32, heatmap_factor, target, &gf))) return rc;
        c->grp.seq = gf.seq;
        return GSR_OK;
    }
    if (c->peer_mode) {  // frames alternate between the presenting rank's two frames; read-back is a separate call
        if (pinned_host) { set_last_error("peer mode: render with a NULL host pointer, then gsr_readback_async on the presenting rank"); return GSR_ERR_STATE; }
        int rc = use_device(c->device);
        if (rc) return rc;
        const int slot = (int)(c->peer_counter & 1u);
        if (c->copied_valid[slot]) GSR_CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_copied[slot], 0));
        if ((rc = render_enqueue(c, view_proj, uniforms32, heatmap_factor, c->peer_fb[slot]))) return rc;
        c->peer_counter += 1;
        return GSR_OK;
    }
    if (!pinned_host || c->fb_ext) {  // nothing to read back, or the caller owns the frame memory: plain enqueue
        if (format != GSR_OUT_RGBA32F && pinned_host) { set_last_error("converted read-back is unavailable with an external framebuffer"); return GSR_ERR_STATE; }
        int rc = render_enqueue(c, view_proj, uniforms32, heatmap_factor);
        if (rc) return rc;
        if (pinned_host)
            GSR_CUDA_TRY(cudaMemcpyAsync(pinned_host, framebuffer(c), sizeof(float4) * frame_pixels(c), cudaMemcpyDeviceToHost, c->stream));
        return GSR_OK;
    }
    // Pipelined read-back: frames alternate between two device framebuffers; the D2H copy of frame i runs on the
    // copy stream while the render stream already works on frame i+1.  Frame i+2 waits for copy i before it
    // overwrites the same buffer.
    int rc = use_device(c->device);
    if (rc) return rc;
    const int slot = (int)(c->async_counter & 1u);
    float4 *target = slot ? c->fb2 : c->fb;   // (render_enqueue orders the compositor after the slot's read-back; sort and ranges need not wait)
    if ((rc = render_enqueue(c, view_proj, uniforms32, heatmap_factor, target))) return rc;
    if ((rc = readback_enqueue(c, target, slot, pinned_host, format))) return rc;
    c->async_counter += 1;
    return GSR_OK;
}

GSR_API int gsr_render_async(gsr_ctx *c, const float view_proj[32], const void *uniforms32, float heatmap_factor, float *pinned_host) {
    if (c && c->num_views > 1) return refuse_multiview("gsr_render_async (use gsr_render_views_async)");
    return render_async_impl(c, view_proj, uniforms32, heatmap_factor, pinned_host, GSR_OUT_RGBA32F);
}

GSR_API int gsr_render_async_rgb(gsr_ctx *c, const float view_proj[32], const void *uniforms32, float heatmap_factor, float *pinned_host_rgb) {
    if (c && c->num_views > 1) return refuse_multiview("gsr_render_async_rgb (use gsr_render_views_async)");
    return render_async_impl(c, view_proj, uniforms32, heatmap_factor, pinned_host_rgb, GSR_OUT_RGB32F);
}

GSR_API int gsr_render_async_fmt(gsr_ctx *c, const float view_proj[32], const void *uniforms32, float heatmap_factor, void *pinned_host, int32_t format) {
    if (c && c->num_views > 1) return refuse_multiview("gsr_render_async_fmt (use gsr_render_views_async)");
    if (!present_bytes_per_pixel(format)) { set_last_error("unknown output format 0x%x", format); return GSR_ERR_INVALID; }
    return render_async_impl(c, view_proj, uniforms32, heatmap_factor, pinned_host, format);
}

GSR_API int gsr_render_views_async(gsr_ctx *c, const float *view_proj, const void *uniforms, float heatmap_factor, void *pinned_host, int32_t format) {
    if (!present_bytes_per_pixel(format)) { set_last_error("unknown output format 0x%x", format); return GSR_ERR_INVALID; }
    return render_async_impl(c, view_proj, uniforms, heatmap_factor, pinned_host, format);
}

GSR_API size_t gsr_output_bytes(int32_t format, int32_t width, int32_t height) {
    return (width > 0 && height > 0) ? present_bytes_per_pixel(format) * (size_t)width * (size_t)height : 0;
}

// Converted copy of the most recent frame into CALLER-OWNED DEVICE memory on the render stream: the hand-off to an imported
// external image / buffer (Vulkan VK_KHR_external_memory via cudaImportExternalMemory, done by the embedder) without touching the host.
GSR_API int gsr_present_device(gsr_ctx *c, void *dst_device, int32_t format) {
    if (!c || !dst_device) return GSR_ERR_INVALID;
    if (!c->fb_last && !c->fb_ext) { set_last_error("gsr_present_device: no frame rendered yet"); return GSR_ERR_STATE; }
    if (!present_bytes_per_pixel(format)) { set_last_error("unknown output format 0x%x", format); return GSR_ERR_INVALID; }
    int rc = use_device(c->device);
    if (rc) return rc;
    if (c->grp.world > 1) {   // the other ranks' rows must have landed (device-side wait, same stream)
        if (c->grp.rank != 0) { set_last_error("gsr_present_device: only rank 0 of a group presents the frame"); return GSR_ERR_STATE; }
        if ((rc = launch_group_wait_done(c->grp.flags[0], c->grp.world, c->grp.seq, c->stream))) return rc;
    }
    return launch_present(framebuffer(c), dst_device, (uint64_t)frame_pixels(c), format, c->stream);
}

GSR_API int gsr_readback_async(gsr_ctx *c, void *pinned_host, int32_t format) {
    if (!c || !pinned_host) return GSR_ERR_INVALID;
    if (!c->fb_last || c->fb_ext) { set_last_error("gsr_readback_async: no library-owned frame rendered yet"); return GSR_ERR_STATE; }
    int rc = use_device(c->device);
    if (rc) return rc;
    if (c->grp.world > 1) {
        if (c->grp.rank != 0) { set_last_error("gsr_readback_async: only rank 0 of a group presents the frame"); return GSR_ERR_STATE; }
        return readback_enqueue(c, c->fb_last, (int)((c->grp.seq - 1u) & 1u), pinned_host, format, c->grp.seq);
    }
    const int slot = (c->fb_last == c->fb2 || (c->peer_mode && c->fb_last == c->peer_fb[1])) ? 1 : 0;
    return readback_enqueue(c, c->fb_last, slot, pinned_host, format);
}

GSR_API int gsr_group_set_present(gsr_ctx *c, int32_t rows_local) {
    if (!c) return GSR_ERR_INVALID;
    if (c->grp.world <= 1) { set_last_error("gsr_group_set_present: attach the group first"); return GSR_ERR_STATE; }
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    c->grp.present_rows = rows_local != 0;
    c->copied_valid[0] = c->copied_valid[1] = false;
    return GSR_OK;
}

// Rows-local presentation: this rank's tile rows (row % world == rank) of the most recent frame -> the same rows of a full-frame
// RGBA32F host image (`host_frame` = address of pixel (0,0); page-locked in THIS process), on this rank's copy stream and PCIe link.
GSR_API int gsr_readback_rows_async(gsr_ctx *c, void *host_frame) {
    if (!c || !host_frame) return GSR_ERR_INVALID;
    if (c->grp.world <= 1 || !c->grp.present_rows || !c->fb_last) { set_last_error("gsr_readback_rows_async: needs an attached group in rows-local presentation and a rendered frame"); return GSR_ERR_STATE; }
    int rc = use_device(c->device);
    if (rc) return rc;
    const int slot = (int)((c->grp.seq - 1u) & 1u);
    const size_t row_bytes = sizeof(float4) * (size_t)c->width, slab = row_bytes * TILE;
    const int G = c->grp.world, r = c->grp.rank;
    GSR_CUDA_TRY(cudaEventRecord(c->ev_done[slot], c->stream));
    GSR_CUDA_TRY(cudaStreamWaitEvent(c->copy_stream, c->ev_done[slot], 0));
    const int full_rows = c->height / TILE;                        // tile rows that are 16 pixel rows high
    const int n_full = r < full_rows ? (full_rows - 1 - r) / G + 1 : 0;
    const char *src = reinterpret_cast<const char *>(c->fb_last);
    char *dst = static_cast<char *>(host_frame);
    if (n_full) GSR_CUDA_TRY(cudaMemcpy2DAsync(dst + (size_t)r * slab, (size_t)G * slab, src + (size_t)r * slab, (size_t)G * slab, slab, (size_t)n_full,
                                               cudaMemcpyDeviceToHost, c->copy_stream));
    if (c->height % TILE && full_rows % G == r)                    // the ragged last tile row, if this rank owns it
        GSR_CUDA_TRY(cudaMemcpyAsync(dst + (size_t)full_rows * slab, src + (size_t)full_rows * slab, row_bytes * (size_t)(c->height % TILE), cudaMemcpyDeviceToHost, c->copy_stream));
    GSR_CUDA_TRY(cudaEventRecord(c->ev_copied[slot], c->copy_stream));
    c->copied_valid[slot] = true;
    return GSR_OK;
}

GSR_API int gsr_peer_export_framebuffers(gsr_ctx *c, void *handles128) {
    if (!c || !handles128) return GSR_ERR_INVALID;
    if (c->num_views > 1) return refuse_multiview("gsr_peer_export_framebuffers");
    if (!c->fb || !c->fb2 || c->fb_ext) { set_last_error("gsr_peer_export_framebuffers: call gsr_resize first (library-owned frames only)"); return GSR_ERR_STATE; }
    int rc = use_device(c->device);
    if (rc) return rc;
    cudaIpcMemHandle_t h[2];
    GSR_CUDA_TRY(cudaIpcGetMemHandle(&h[0], c->fb));
    GSR_CUDA_TRY(cudaIpcGetMemHandle(&h[1], c->fb2));
    memcpy(handles128, h, sizeof h);
    c->peer_fb[0] = c->fb; c->peer_fb[1] = c->fb2;
    c->peer_mode = true;
    return GSR_OK;
}

GSR_API int gsr_peer_import_framebuffers(gsr_ctx *c, const void *handles128) {
    if (!c || !handles128) return GSR_ERR_INVALID;
    if (c->num_views > 1) return refuse_multiview("gsr_peer_import_framebuffers");
    int rc = use_device(c->device);
    if (rc) return rc;
    cudaIpcMemHandle_t h[2];
    memcpy(h, handles128, sizeof h);
    GSR_CUDA_TRY(cudaIpcOpenMemHandle((void **)&c->peer_fb[0], h[0], cudaIpcMemLazyEnablePeerAccess));
    GSR_CUDA_TRY(cudaIpcOpenMemHandle((void **)&c->peer_fb[1], h[1], cudaIpcMemLazyEnablePeerAccess));
    c->peer_mode = true; c->peer_opened = true;
    return GSR_OK;
}

// ---- multi-GPU shard group: one context per GPU (processes or threads), NCCL-free frame path (group.cu) ----
namespace {
struct GroupBlob {   // what gsr_group_export hands to the other ranks (any transport; 320 bytes)
    uint32_t magic, version;
    uint64_t pid;
    int32_t device, width, height, pad;
    uint64_t max_splats, rx_capacity;
    void *arena, *fb[2];
    cudaIpcMemHandle_t h_arena, h_fb[2];
    unsigned char reserved[GSR_GROUP_BLOB_BYTES - 264];
};
static_assert(sizeof(GroupBlob) == GSR_GROUP_BLOB_BYTES, "blob layout");
constexpr uint32_t GROUP_MAGIC = 0x47535247u;  // "GRSG"

}  // namespace

GSR_API int gsr_group_export(gsr_ctx *c, void *blob) {
    if (!c || !blob) return GSR_ERR_INVALID;
    if (c->num_views > 1) return refuse_multiview("gsr_group_export");
    if (!c->fb || !c->fb2 || c->fb_ext) { set_last_error("gsr_group_export: call gsr_resize first (library-owned frames only)"); return GSR_ERR_STATE; }
    int rc = use_device(c->device);
    if (rc) return rc;
    if (!c->grp.arena) {
        c->grp.rx_capacity = (c->capacity + 1023ull) & ~1023ull;   // the receive segments of all sources together hold as many pairs as one sort input
        const size_t bytes = arena_bytes(c->grp.rx_capacity, c->max_splats);
        cudaError_t e = cudaMalloc(&c->grp.arena, bytes);
        if (e != cudaSuccess) { set_last_error("cudaMalloc(group arena, %zu B) -> %s", bytes, cudaGetErrorString(e)); c->grp.arena = nullptr; return GSR_ERR_OOM; }
        GSR_CUDA_TRY(cudaMemset(c->grp.arena, 0, bytes));
    }
    GroupBlob b;
    memset(&b, 0, sizeof b);
    b.magic = GROUP_MAGIC; b.version = 1; b.pid = (uint64_t)getpid();
    b.device = c->device; b.width = c->width; b.height = c->height;
    b.max_splats = c->max_splats; b.rx_capacity = c->grp.rx_capacity;
    b.arena = c->grp.arena; b.fb[0] = c->fb; b.fb[1] = c->fb2;
    // IPC handles are needed only by ranks living in other processes; a failure here surfaces there (zero handle)
    if (cudaIpcGetMemHandle(&b.h_arena, c->grp.arena) != cudaSuccess || cudaIpcGetMemHandle(&b.h_fb[0], c->fb) != cudaSuccess ||
        cudaIpcGetMemHandle(&b.h_fb[1], c->fb2) != cudaSuccess) {
        cudaGetLastError();
        memset(&b.h_arena, 0, sizeof b.h_arena); memset(b.h_fb, 0, sizeof b.h_fb);
    }
    memcpy(blob, &b, sizeof b);
    return GSR_OK;
}

GSR_API int gsr_group_attach(gsr_ctx *c, int32_t rank, int32_t world, const void *blobs) {
    if (!c || !blobs || world < 1 || world > GROUP_MAX || rank < 0 || rank >= world) { set_last_error("gsr_group_attach: need 0 <= rank < world <= %d", GROUP_MAX); return GSR_ERR_INVALID; }
    if (!c->grp.arena || !c->fb) { set_last_error("gsr_group_attach before gsr_group_export"); return GSR_ERR_STATE; }
    if (c->num_views > 1) return refuse_multiview("gsr_group_attach");
    int rc = use_device(c->device);
    if (rc) return rc;
    group_detach(c);
    if (world == 1) return GSR_OK;
    const GroupBlob *B = reinterpret_cast<const GroupBlob *>(blobs);
    const uint64_t slice = (((c->max_splats + (uint64_t)world - 1) / (uint64_t)world) + 255ull) & ~255ull;
    for (int r = 0; r < world; ++r) {
        if (B[r].magic != GROUP_MAGIC || B[r].version != 1) { set_last_error("gsr_group_attach: blob %d is not a gsr_group_export blob", r); return GSR_ERR_INVALID; }
        if (B[r].max_splats != c->max_splats || B[r].width != c->width || B[r].height != c->height || B[r].rx_capacity != c->grp.rx_capacity) {
            set_last_error("gsr_group_attach: rank %d was created with a different scene / frame size", r);
            return GSR_ERR_INVALID;
        }
    }
    if (B[rank].arena != c->grp.arena || B[rank].pid != (uint64_t)getpid()) { set_last_error("gsr_group_attach: blob %d is not this context's export", rank); return GSR_ERR_INVALID; }
    auto fail = [&](const char *what, int r, cudaError_t e) {
        set_last_error("gsr_group_attach: %s of rank %d -> %s", what, r, cudaGetErrorString(e));
        group_detach(c);
        return GSR_ERR_CUDA;
    };
    for (int r = 0; r < world; ++r) {
        char *arena = nullptr;
        float4 *fb[2] = {nullptr, nullptr};
        if (r == rank) {
            arena = (char *)c->grp.arena; fb[0] = c->fb; fb[1] = c->fb2;
        } else if (B[r].pid == (uint64_t)getpid()) {   // same process (one thread per GPU, the GDExtension case): plain peer pointers
            if (B[r].device != c->device) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, c->device, B[r].device);
                if (!can) return fail("no peer access to the device", r, cudaErrorPeerAccessUnsupported);
                cudaError_t e = cudaDeviceEnablePeerAccess(B[r].device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail("cudaDeviceEnablePeerAccess", r, e);
                cudaGetLastError();
            }
            arena = (char *)B[r].arena; fb[0] = (float4 *)B[r].fb[0]; fb[1] = (float4 *)B[r].fb[1];
        } else {                                       // another process: CUDA IPC mappings
            cudaError_t e = cudaIpcOpenMemHandle((void **)&arena, B[r].h_arena, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) return fail("cudaIpcOpenMemHandle(arena)", r, e);
            c->grp.opened[c->grp.n_opened++] = arena;
            if (r == 0) {
                for (int k = 0; k < 2; ++k) {
                    e = cudaIpcOpenMemHandle((void **)&fb[k], B[r].h_fb[k], cudaIpcMemLazyEnablePeerAccess);
                    if (e != cudaSuccess) return fail("cudaIpcOpenMemHandle(frame)", r, e);
                    c->grp.opened[c->grp.n_opened++] = fb[k];
                }
            }
        }
        c->grp.flags[r] = reinterpret_cast<GroupFlags *>(arena);
        c->grp.peer_arena[r] = arena;
        if (r == 0) { c->grp.root_fb[0] = fb[0]; c->grp.root_fb[1] = fb[1]; }
    }
    GSR_CUDA_TRY(cudaMemsetAsync(c->grp.arena, 0, GROUP_FLAGS_BYTES, c->stream));   // flags start at seq 0 (all ranks attach, then barrier)
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->grp.rank = rank; c->grp.world = world; c->grp.slice = slice; c->grp.seq = 0;
    c->grp.seg_cap = (uint32_t)(c->grp.rx_capacity / (uint64_t)world) & ~3u;   // segments start 16-byte aligned
    c->row_mod = world; c->row_rem = rank;   // cyclic tile rows: balanced by construction
    c->band_y0 = 0; c->band_y1 = c->tiles_y; c->band_set = false;
    c->copied_valid[0] = c->copied_valid[1] = false;
    return GSR_OK;
}

GSR_API int gsr_group_detach(gsr_ctx *c) {
    if (!c) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    group_detach(c);
    return GSR_OK;
}

GSR_API int gsr_stream_join(gsr_ctx *c) {
    if (!c) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    for (int i = 0; i < 2; ++i)
        if (c->copied_valid[i]) GSR_CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_copied[i], 0));
    return GSR_OK;
}

GSR_API int gsr_sync(gsr_ctx *c) {
    if (!c) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->copy_stream));
    if (c->grp.world > 1) {   // a device-side wait of the group protocol gave up (peer lost / frames enqueued out of lockstep)
        uint32_t err = 0;
        GSR_CUDA_TRY(cudaMemcpy(&err, &c->grp.flags[c->grp.rank]->error, sizeof err, cudaMemcpyDeviceToHost));
        if (err) {
            cudaMemset(&c->grp.flags[c->grp.rank]->error, 0, sizeof err);
            set_last_error("group: a device-side wait timed out (%s)", err == 1 ? "segments of a peer" : "done / released flag");
            return GSR_ERR_STATE;
        }
    }
    return GSR_OK;
}

GSR_API void *gsr_framebuffer_device_ptr(gsr_ctx *c) { return c ? (void *)framebuffer(c) : nullptr; }

GSR_API int gsr_set_framebuffer_external(gsr_ctx *c, void *device_ptr) {
    if (!c) return GSR_ERR_INVALID;
    c->fb_ext = (float4 *)device_ptr;
    return GSR_OK;
}

GSR_API int gsr_pick(gsr_ctx *c, uint32_t tile_id, float heatmap_factor, float out_xyzn[4]) {
    if (!c || !out_xyzn) return GSR_ERR_INVALID;
    if (c->width == 0) { set_last_error("gsr_pick before gsr_resize"); return GSR_ERR_STATE; }
    if (c->frame_counter == 0 || !c->fb_last) { set_last_error("gsr_pick before the first gsr_render at this size"); return GSR_ERR_STATE; }
    int rc = use_device(c->device);
    if (rc) return rc;
    const uint32_t T = (uint32_t)(c->tiles_x * c->tiles_y);
    const uint32_t t0 = (uint32_t)(c->band_y0 * c->tiles_x), t1 = (uint32_t)(c->band_y1 * c->tiles_x);
    const bool owned = c->num_views > 1 ? tile_id < T * (uint32_t)c->num_views   // multiview: full frames, tile ids of all views
                                        : (tile_id < T && tile_id >= t0 && tile_id < t1 && (int)(tile_id / (uint32_t)c->tiles_x) % c->row_mod == c->row_rem);
    if (owned) {
        CompositeArgs ca;
        ca.records = c->records_cur; ca.values = c->vals_cur; ca.bounds = c->bounds; ca.out = framebuffer(c);
        ca.width = c->width; ca.height = c->height; ca.tiles_x = c->tiles_x;
        ca.tile_begin = (int32_t)tile_id; ca.num_tiles = 1; ca.row_step = 1;
        ca.heatmap_factor = heatmap_factor; ca.target_tile_id = tile_id; ca.pick = c->pick;
        ca.frame = c->pick_frame; ca.count_staged = 0;  // own queue counters; slot 0 of the queue, state slot 0
        ca.order = nullptr; ca.consumed = nullptr; ca.ctas_per_sm = 1; ca.sm_count = c->sm_count;
        ca.contract = (c->flags & GSR_FLAG_UNCONTRACTED_BLEND) ? 0 : 1;
        ca.trace = nullptr; ca.trace_count = nullptr; ca.trace_cap = 0;
        ca.tiles_per_view = c->num_views > 1 ? (int32_t)T : 0;
        ca.layer_stride = (uint64_t)c->width * c->height; ca.record_stride = 3ull * c->max_splats;
        for (int i = 0; i < 2; ++i)   // the re-dispatch rewrites the tile's pixels: not under a read-back in flight
            if (c->copied_valid[i]) GSR_CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_copied[i], 0));
        GSR_CUDA_TRY(cudaMemsetAsync(c->pick_frame, 0, sizeof(FrameState), c->stream));
        if ((rc = launch_composite(ca, c->stream))) return rc;
    }
    GSR_CUDA_TRY(cudaMemcpyAsync(out_xyzn, c->pick, sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return GSR_OK;
}

GSR_API int gsr_get_stats(gsr_ctx *c, gsr_stats *out) {
    if (!c || !out) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    memset(out, 0, sizeof *out);
    FrameState fs;
    GSR_CUDA_TRY(cudaMemcpyAsync(&fs, c->frame, sizeof fs, cudaMemcpyDeviceToHost, c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    out->num_splats = c->num_splats;
    out->duplicates = fs.dup_total;
    out->visible = fs.visible;
    out->capacity = c->capacity;
    out->last_tile = (int64_t)fs.last_tile_plus1 - 1;
    out->overflow = fs.overflow;
    out->width = (uint32_t)c->width; out->height = (uint32_t)c->height;
    out->tiles_x = (uint32_t)c->tiles_x; out->tiles_y = (uint32_t)c->tiles_y;
    out->band_y0 = (uint32_t)c->band_y0; out->band_y1 = (uint32_t)c->band_y1;
    out->kernel_launches = c->last_launches;
    out->staged = fs.staged;
    if (c->ev_valid && c->frame_counter > 0) {
        if ((rc = stage_times(c, (uint32_t)((c->frame_counter - 1) % GSR_HISTORY_FRAMES), out->stage_ms, nullptr))) return rc;
    }
    return GSR_OK;
}

GSR_API int gsr_get_frame_history(gsr_ctx *c, uint32_t max_frames, gsr_frame_record *out, uint32_t *n_out) {
    if (!c || !out || !n_out) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    *n_out = 0;
    if (!c->ev_valid || c->frame_counter == 0) return GSR_OK;
    uint64_t n = c->frame_counter < GSR_HISTORY_FRAMES ? c->frame_counter : GSR_HISTORY_FRAMES;
    if (n > max_frames) n = max_frames;
    static thread_local FrameState host_ring[GSR_HISTORY_FRAMES];
    GSR_CUDA_TRY(cudaMemcpyAsync(host_ring, c->ring, sizeof(FrameState) * GSR_HISTORY_FRAMES, cudaMemcpyDeviceToHost, c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t fi = c->frame_counter - n + k;
        const uint32_t slot = (uint32_t)(fi % GSR_HISTORY_FRAMES);
        const FrameState &fs = host_ring[slot];
        gsr_frame_record &r = out[k];
        memset(&r, 0, sizeof r);
        r.frame_index = fi; r.duplicates = fs.dup_total; r.visible = fs.visible; r.staged = fs.staged; r.overflow = fs.overflow;
        if ((rc = stage_times(c, slot, r.stage_ms, &r.front_ms))) return rc;
    }
    *n_out = (uint32_t)n;
    return GSR_OK;
}

GSR_API int gsr_debug_keep_unsorted(gsr_ctx *c, int enable) {
    if (!c) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    if (enable && !c->unsorted_keys) {
        GSR_CUDA_TRY(cudaMalloc((void **)&c->unsorted_keys, sizeof(uint32_t) * c->capacity));
        GSR_CUDA_TRY(cudaMalloc((void **)&c->unsorted_vals, sizeof(uint32_t) * c->capacity));
    }
    c->keep_unsorted = enable != 0;
    return GSR_OK;
}

GSR_API int gsr_debug_compositor_config(gsr_ctx *c, int32_t ctas_per_sm, int32_t longest_first, int32_t sparse_tiles_per_sm) {
    if (!c || ctas_per_sm < 0 || sparse_tiles_per_sm < 0) return GSR_ERR_INVALID;
    c->comp_ctas_per_sm = ctas_per_sm ? ctas_per_sm : c->comp_max_ctas; c->comp_order_mode = longest_first != 0; c->comp_sparse_per_sm = sparse_tiles_per_sm;
    return GSR_OK;
}

GSR_API int gsr_debug_pipeline(gsr_ctx *c, int32_t overlap) {
    if (!c) return GSR_ERR_INVALID;
    if (c->num_views > 1 && overlap > 0) return refuse_multiview("gsr_debug_pipeline (overlap)");
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->front_stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->overlap = overlap < 0 ? -1 : (overlap != 0); c->front_gate = nullptr;
    return GSR_OK;
}

GSR_API int gsr_debug_enable_trace(gsr_ctx *c, uint32_t max_items) {
    if (!c) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    cudaFree(c->trace); cudaFree(c->trace_count);
    c->trace = nullptr; c->trace_count = nullptr; c->trace_cap = 0;
    if (max_items) {
        GSR_CUDA_TRY(cudaMalloc((void **)&c->trace, sizeof(ulonglong4) * (size_t)max_items + 32));
        GSR_CUDA_TRY(cudaMalloc((void **)&c->trace_count, sizeof(uint32_t)));
        GSR_CUDA_TRY(cudaMemset(c->trace_count, 0, sizeof(uint32_t)));
        c->trace_cap = max_items;
    }
    return GSR_OK;
}

GSR_API int gsr_debug_copy(gsr_ctx *c, int which, void *dst, size_t bytes) {
    if (!c || !dst) return GSR_ERR_INVALID;
    int rc = use_device(c->device);
    if (rc) return rc;
    const void *src = nullptr;
    size_t avail = 0;
    switch (which) {
        case GSR_BUF_RECORDS: src = c->records_cur; avail = sizeof(float4) * 3ull * c->max_splats * (size_t)c->num_views; break;
        case GSR_BUF_KEYS: src = c->keys_cur; avail = sizeof(uint32_t) * c->capacity; break;
        case GSR_BUF_VALUES: src = c->vals_cur; avail = sizeof(uint32_t) * c->capacity; break;
        case GSR_BUF_BOUNDS: src = c->bounds; avail = sizeof(uint2) * frame_tiles(c); break;
        case GSR_BUF_KEYS_UNSORTED: src = c->unsorted_keys; avail = c->unsorted_keys ? sizeof(uint32_t) * c->capacity : 0; break;
        case GSR_BUF_VALUES_UNSORTED: src = c->unsorted_vals; avail = c->unsorted_vals ? sizeof(uint32_t) * c->capacity : 0; break;
        case GSR_BUF_FRAMEBUFFER: src = framebuffer(c); avail = sizeof(float4) * frame_pixels(c); break;
        case GSR_BUF_COMPOSITOR_TRACE: src = c->trace; avail = c->trace ? sizeof(ulonglong4) * (size_t)c->trace_cap : 0; break;
        case GSR_BUF_COMPOSITOR_TRACE_COUNT: src = c->trace_count; avail = c->trace_count ? sizeof(uint32_t) : 0; break;
        default: set_last_error("gsr_debug_copy: unknown buffer %d", which); return GSR_ERR_INVALID;
    }
    if (!src || bytes > avail) { set_last_error("gsr_debug_copy(%d): %zu bytes requested, %zu available", which, bytes, avail); return GSR_ERR_INVALID; }
    GSR_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    GSR_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return GSR_OK;
}

// ---------------------------------------------------------------------------------------------------
// stand-alone sorter
// ---------------------------------------------------------------------------------------------------
GSR_API int gsr_sorter_create(int32_t device, uint64_t max_n, gsr_sorter **out) {
    if (!out || max_n == 0) return GSR_ERR_INVALID;
    *out = nullptr;
    int rc = check_device(device);
    if (rc) return rc;
    if ((rc = use_device(device))) return rc;
    gsr_sorter *s = new (std::nothrow) gsr_sorter();
    if (!s) return GSR_ERR_OOM;
    s->device = device;
    rc = sort_workspace_create(s->ws, max_n, /*need_alt_buffers=*/true);
    if (rc == GSR_OK && (cudaEventCreate(&s->e0) != cudaSuccess || cudaEventCreate(&s->e1) != cudaSuccess)) rc = GSR_ERR_CUDA;
    if (rc) { sort_workspace_destroy(s->ws); delete s; return rc; }
    *out = s;
    return GSR_OK;
}

GSR_API int gsr_sorter_destroy(gsr_sorter *s) {
    if (!s) return GSR_OK;
    cudaSetDevice(s->device);
    cudaDeviceSynchronize();
    sort_workspace_destroy(s->ws);
    if (s->e0) cudaEventDestroy(s->e0);
    if (s->e1) cudaEventDestroy(s->e1);
    delete s;
    return GSR_OK;
}

GSR_API int gsr_sorter_sort_device(gsr_sorter *s, void *d_keys, void *d_values, uint64_t n, void *cuda_stream) {
    if (!s || (!d_keys && n)) return GSR_ERR_INVALID;
    if (n > s->ws.max_n) { set_last_error("sort of %llu exceeds sorter capacity %llu", (unsigned long long)n, (unsigned long long)s->ws.max_n); return GSR_ERR_INVALID; }
    int rc = use_device(s->device);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const uint32_t n32 = (uint32_t)n;
    GSR_CUDA_TRY(cudaMemcpyAsync(s->ws.n_dev, &n32, sizeof n32, cudaMemcpyHostToDevice, st));
    GSR_CUDA_TRY(cudaEventRecord(s->e0, st));
    int launches = 0;
    rc = sort_pairs_device(s->ws, (uint32_t *)d_keys, (uint32_t *)d_values, s->ws.n_dev, s->ws.alt_keys, d_values ? s->ws.alt_vals : nullptr, st, &launches);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaEventRecord(s->e1, st));
    s->timed = true;
    return GSR_OK;
}

GSR_API int gsr_sorter_last_ms(gsr_sorter *s, float *ms) {
    if (!s || !ms || !s->timed) return GSR_ERR_STATE;
    int rc = use_device(s->device);
    if (rc) return rc;
    GSR_CUDA_TRY(cudaEventSynchronize(s->e1));
    GSR_CUDA_TRY(cudaEventElapsedTime(ms, s->e0, s->e1));
    return GSR_OK;
}

GSR_API int gsr_sort_pairs_host(int32_t device, uint32_t *keys, uint32_t *values, uint64_t n) {
    if (n == 0) return GSR_OK;
    if (!keys) return GSR_ERR_INVALID;
    gsr_sorter *s = nullptr;
    int rc = gsr_sorter_create(device, n, &s);
    if (rc) return rc;
    uint32_t *dk = nullptr, *dv = nullptr;
    cudaError_t e = cudaMalloc((void **)&dk, 4 * n);
    if (e == cudaSuccess && values) e = cudaMalloc((void **)&dv, 4 * n);
    if (e == cudaSuccess) e = cudaMemcpy(dk, keys, 4 * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && values) e = cudaMemcpy(dv, values, 4 * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = gsr_sorter_sort_device(s, dk, dv, n, nullptr);
        if (rc == GSR_OK) e = cudaDeviceSynchronize();
    }
    if (e == cudaSuccess && rc == GSR_OK) e = cudaMemcpy(keys, dk, 4 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && rc == GSR_OK && values) e = cudaMemcpy(values, dv, 4 * n, cudaMemcpyDeviceToHost);
    cudaFree(dk); cudaFree(dv);
    gsr_sorter_destroy(s);
    if (e != cudaSuccess) { set_last_error("gsr_sort_pairs_host: %s", cudaGetErrorString(e)); return e == cudaErrorMemoryAllocation ? GSR_ERR_OOM : GSR_ERR_CUDA; }
    return rc;
}

}  // extern "C"
