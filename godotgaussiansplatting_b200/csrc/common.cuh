// common.cuh -- shared declarations of libgsr (sm_100a).  Product code: never includes anything from oracle/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gsr.h"

namespace gsr {

constexpr int TILE = 16;            // rasterizer.gd:4 TILE_SIZE
constexpr int NUM_PLANES = 15;      // 60-float Splat = 15 float4 planes in SoA
constexpr int PROJ_THREADS = 256;   // gsplat_projection.glsl:31 local_size_x

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
void set_last_error(const char *fmt, ...);

#define GSR_CUDA_TRY(expr)                                                                         \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            ::gsr::set_last_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return (_e == cudaErrorMemoryAllocation) ? GSR_ERR_OOM : GSR_ERR_CUDA;                 \
        }                                                                                          \
    } while (0)

// ---------------------------------------------------------------------------------------------
// "gsr deterministic math" (DESIGN.md section 4).  One IEEE binary32 op per operator, no implicit
// contraction (the library is compiled with -fmad=false), explicit __fmaf_rn where the spec says so.
// GLSL min/max/clamp semantics written out (gsplat_projection.glsl uses clamp/max).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float g_max(float x, float y) { return (x < y) ? y : x; }
__device__ __forceinline__ float g_min(float x, float y) { return (y < x) ? y : x; }
__device__ __forceinline__ float g_clamp(float x, float lo, float hi) { return g_min(g_max(x, lo), hi); }

// 2^t: clamp to [-127,128], round-half-even via the 1.5*2^23 magic constant, degree-6 polynomial on
// [-0.5,0.5] (Horner, fma), scale 2^n assembled in the exponent field (n=-127 -> 0, n=128 -> +inf).
__device__ __forceinline__ float det_exp2(float t) {
    const float MAGIC = 12582912.0f;
    float tc = g_min(g_max(t, -127.0f), 128.0f);
    float tm = __fadd_rn(tc, MAGIC);
    float nf = __fsub_rn(tm, MAGIC);
    float f = __fsub_rn(tc, nf);
    float p = 0x1.446c7ep-13f;
    p = __fmaf_rn(p, f, 0x1.5f48c8p-10f);
    p = __fmaf_rn(p, f, 0x1.3b29d8p-7f);
    p = __fmaf_rn(p, f, 0x1.c6aeccp-5f);
    p = __fmaf_rn(p, f, 0x1.ebfbe0p-3f);
    p = __fmaf_rn(p, f, 0x1.62e430p-1f);
    p = __fmaf_rn(p, f, 1.0f);
    uint32_t sbits = (__float_as_uint(tm) << 23) + 0x3F800000u;
    return __fmul_rn(p, __uint_as_float(sbits));
}

// GLSL exp(x) := 2^(x*log2e), log2e rounded to binary32.
__device__ __forceinline__ float det_exp(float x) { return det_exp2(__fmul_rn(x, 0x1.715476p+0f)); }

__device__ __forceinline__ float det_log2(float x) {
    int eadj = 0;
    if (x < 0x1p-126f) { x = __fmul_rn(x, 0x1p+32f); eadj = -32; }
    uint32_t u = __float_as_uint(x);
    int e = (int)(u >> 23) - 127;
    float m = __uint_as_float((u & 0x007FFFFFu) | 0x3F800000u);
    if (m >= 0x1.6a09e6p+0f) { m = __fmul_rn(m, 0.5f); e += 1; }
    float s = __fdiv_rn(__fsub_rn(m, 1.0f), __fadd_rn(m, 1.0f));
    float z = __fmul_rn(s, s);
    float g = 0x1.ba18b8p-2f;
    g = __fmaf_rn(g, z, 0x1.27471ep-1f);
    g = __fmaf_rn(g, z, 0x1.ec70e6p-1f);
    g = __fmaf_rn(g, z, 0x1.715476p+1f);
    return __fadd_rn((float)(e + eadj), __fmul_rn(s, g));
}

// GLSL pow(x,y) := exp2(y*log2(x)), pow(x<=0, y>0) := 0.
__device__ __forceinline__ float det_pow(float x, float y) {
    if (!(x > 0.0f)) return 0.0f;
    return det_exp2(__fmul_rn(y, det_log2(x)));
}

// ---------------------------------------------------------------------------------------------
// per-frame device state (one cudaMemsetAsync clears it; rasterizer.gd:127 clears histogram[0..1024])
// ---------------------------------------------------------------------------------------------
struct FrameState {
    unsigned long long dup_total;  // M, true count (histogram[0] of the reference)
    uint32_t dup_sorted;           // min(M, capacity): what the sort / ranges / compositor see
    uint32_t visible;              // V
    int32_t last_tile_plus1;       // 1 + largest tile id touched (0 = none); atomicMax target
    uint32_t overflow;
    uint32_t proj_ticket;          // dynamic block id for the projection look-back
    uint32_t pad0;
    unsigned long long staged;     // C: instances staged by the compositor (sum of consumed chunk sizes)
    uint32_t comp_head;            // compositor: next tile ticket of the persistent grid
    uint32_t comp_cta_limit;       // compositor: CTAs that may work (0 = all launched); set by tile_order_kernel for sparse frames
    uint32_t pad[4];
};
static_assert(sizeof(FrameState) == 64, "FrameState is one 64-byte slot of the history ring");

// Uniform block exactly as the reference uploads it (rasterizer.gd:126; gsplat_projection.glsl:75-80)
struct Uniforms {
    float camera_pos[3];
    float model_scale;
    int32_t dims[2];
    float time;
    float pad;
};
static_assert(sizeof(Uniforms) == 32, "uniform block must be 32 bytes");

// ---------------------------------------------------------------------------------------------
// radix sorter (radix_sort.cu)
// ---------------------------------------------------------------------------------------------
struct SortWorkspace {
    uint32_t *hist = nullptr;       // [4][256] global digit histograms
    uint32_t *status = nullptr;     // [4][max_tiles][256] decoupled look-back words
    uint32_t *tickets = nullptr;    // [4] dynamic tile counters (same allocation as hist)
    uint32_t *alt_keys = nullptr;   // ping-pong halves
    uint32_t *alt_vals = nullptr;
    uint32_t *n_dev = nullptr;      // device copy of n for the stand-alone sorter
    uint64_t max_n = 0;
    uint32_t max_tiles = 0;
    int grid_hist = 0, grid_sweep_pairs = 0, grid_sweep_keys = 0;
    size_t bytes() const;
};
int sort_workspace_create(SortWorkspace &ws, uint64_t max_n, bool need_alt_buffers);
void sort_workspace_destroy(SortWorkspace &ws);
// Sorts n (read on the device from *n_ptr, clamped to ws.max_n) pairs; 4 passes ping-pong between
// keys/vals and alt_keys/alt_vals (the reference's two buffer halves, rasterizer.gd:145), result back in
// keys/vals.  vals/alt_vals may be null (keys only).  *launches += kernels launched.
int sort_pairs_device(SortWorkspace &ws, uint32_t *keys, uint32_t *vals, const uint32_t *n_ptr, uint32_t *alt_keys,
                      uint32_t *alt_vals, cudaStream_t stream, int *launches);
uint32_t sort_tile_keys();

// ---------------------------------------------------------------------------------------------
// stage launchers (projection.cu, ranges.cu, compositor.cu, ingest.cu)
// ---------------------------------------------------------------------------------------------
struct ProjectionArgs {
    const float4 *soa;       // 15 planes of `plane_stride` float4 each
    uint64_t plane_stride;
    uint32_t num_splats;
    float vp[32];            // view_matrix, projection_matrix (GLSL column-major)
    Uniforms u;
    float focal_base[2];     // (dims*0.5) * (P00, P11)           gsplat_projection.glsl:127-128
    float lim_lo[2], lim_hi[2];  // -+ (1/(P00,P11)) * 1.3          gsplat_projection.glsl:129,133
    int32_t band_y0, band_y1;  // tile rows [band_y0, band_y1) ...
    int32_t row_mod, row_rem;  // ... of which this context owns those with row % row_mod == row_rem (1, 0 = all)
    int32_t fast_reject;       // sharded fast mode: conservative early reject of splats that cannot touch an owned row;
                               // last_tile is then the LOCAL last emitted tile (global one by all-reduce, gsr_band_fixup)
    int32_t sh_bulk_min;       // warps with at least this many emitting lanes fetch their SH planes with TMA bulk copies
    int32_t fast_mode;         // fast sharded mode (row_mod > 1): last_tile is the LOCAL last emitted tile
    float w_frob2;             // upper bound of |mat3(view_matrix)|_2^2 (for the early reject)
    float4 *records;         // 3 float4 per splat id (RasterizeData layout)
    uint32_t *keys, *values;
    uint32_t capacity;
    unsigned long long *lookback;  // one word per projection CTA (256 splats)
    FrameState *frame;
};
int launch_projection(const ProjectionArgs &a, cudaStream_t stream);

// Multiview frame (gsr_set_views): K cameras of one splat cloud in one projection.  view[v] carries camera v's matrices, uniform block
// and per-frame constants and its own record table; every other field is the same in all K entries (keys, values, capacity, look-back,
// frame state, splat planes).  View v's pairs carry the tile ids [v*T, (v+1)*T), so one sort orders all views.
struct ViewsArgs {
    ProjectionArgs view[GSR_MAX_VIEWS];
    int32_t num_views;
    uint32_t tiles_per_view;  // T
};
int launch_projection_views(const ViewsArgs &a, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// multi-GPU shard group (group.cu, gsr_group_attach): flag words + receive segments + record tables in every rank's arena
// ---------------------------------------------------------------------------------------------
constexpr int GROUP_MAX = 16;                                   // ranks per group (one NVSwitch domain)
// Receive segments and record tables exist three times (frame seq % 3): a source's scatter projection of frame f+1 runs while the
// destinations still composite frame f (front / back overlap, gsr_api.cu), and frame f-1's consumers are only known to be done
// through the chain  scatter(f+1) after own ranges(f) after all sources' scatter(f) after their ranges(f-1) after their compositor(f-2).
constexpr int GROUP_PHASES = 3;
#define GSR_GROUP_TIMEOUT_NS 2000000000ull                      // every device-side wait gives up after 2 s
struct GroupFlags {                                             // offset 0 of a rank's arena; written by the peers over NVLink
    // [frame phase = seq % 3][source rank][0] = seq << 32 | pairs the source sent to THIS rank's receive segment,
    //                                     [1] = seq << 32 | (largest tile id touched by the source's splats + 1)
    unsigned long long seg_meta[GROUP_PHASES][GROUP_MAX][2];
    uint32_t done[GROUP_MAX];               // presenting rank: done[r] = seq of the newest frame whose rows from rank r have landed
    uint32_t released;                      // set by the presenting rank: frames with seq <= released no longer need their slot
    uint32_t error;                         // local: a wait timed out (1 = segments of a peer, 2 = done / released)
    uint32_t scat_ticket;                   // local: CTAs of the scatter projection that have finished
    int32_t scat_last;                      // local: atomicMax target, last tile + 1 over this rank's slice
    unsigned long long seg_total[GROUP_MAX];  // local: pairs this rank sent to each destination this frame (scan total)
    uint32_t seg_prefix[GROUP_MAX + 1];     // local: exclusive prefix of the received (clamped) segment lengths, [world] = M of this rank
};
constexpr size_t GROUP_FLAGS_BYTES = 4096;                      // the receive segments and record tables follow the flag page
static_assert(sizeof(GroupFlags) <= GROUP_FLAGS_BYTES, "flag page");
struct GroupPeers {                                             // the same pointers on every rank, indexed by rank
    GroupFlags *flags[GROUP_MAX];
    int world, rank;
};
// What the scatter projection of one rank needs to know about the group: every destination's record table and receive segment
// (peer pointers) of the current frame phase (seq % 3; called parity below), and this rank's slice of the splats.
struct ScatterPeers {
    int world, rank, parity;
    uint32_t seq;
    uint32_t first, count;                  // this rank projects splats [first, first + count)
    uint32_t seg_cap;                       // pairs one source may send to one destination per frame
    float4 *records[GROUP_MAX];             // destination d's record table (3 float4 per splat id) of this parity
    uint32_t *keys[GROUP_MAX];              // destination d's receive segment for THIS source: pairs land at [0, seg_cap)
    uint32_t *values[GROUP_MAX];
    GroupFlags *flags[GROUP_MAX];
    unsigned long long *lookback;           // [blocks][world] scan links of this launch (zeroed)
};
// Projection sharded by SPLATS (group mode): rank r projects its slice with the full-frame maths of projection_kernel and emits every
// (key, value) pair and every record straight into the memory of the rank that owns the pair's tile row (row % world), in splat-id
// order per destination -- the all-to-all of SURVEY 8e's "alternative" fused into the kernel as peer stores over NVLink.
int launch_projection_scatter(const ProjectionArgs &a, const ScatterPeers &sp, cudaStream_t stream);
uint32_t projection_scatter_blocks(uint32_t count);
// destination side: wait for every source's segment of this frame, publish M / overflow / the frame-global last tile, then pack the
// world receive segments into the contiguous sort input (source-rank order = splat-id order)
int launch_group_wait_segments(GroupFlags *flags, int parity, int world, uint32_t seq, uint32_t seg_cap, uint32_t capacity, FrameState *frame, cudaStream_t stream);
int launch_gather_segments(const GroupFlags *flags, int world, uint32_t seg_cap, const uint32_t *rx_keys, const uint32_t *rx_vals, uint32_t *keys, uint32_t *vals,
                           int grid, cudaStream_t stream);
// 64-byte FrameState -> mapped pinned host memory with system-scope stores (no copy engine involved)
int launch_publish_frame_state(const FrameState *frame, FrameState *host_mapped, cudaStream_t stream);
int launch_group_wait_released(GroupFlags *flags, uint32_t need, cudaStream_t stream);
int launch_group_wait_done(GroupFlags *flags, int world, uint32_t seq, cudaStream_t stream);
int launch_group_signal_done(const GroupPeers &peers, int root, int rank, uint32_t seq, cudaStream_t stream);
int launch_group_release(const GroupPeers &peers, int world, uint32_t value, cudaStream_t stream);
uint32_t projection_num_blocks(uint32_t num_splats);

// sharded: 0 = full frame, 1 = exact sharded mode (global last tile known from the projection), 2 = fast sharded mode
// (local last tile -> *sync_word = tile + 1; the frame-global quirk is applied later by launch_band_fixup).
int launch_tile_ranges(const uint32_t *sorted_keys, const FrameState *frame, uint2 *bounds, uint32_t num_tiles,
                       int quirks, int sharded, int32_t *sync_word, int grid, cudaStream_t stream);
// Multiview frame: the same ranges per view over the concatenated tile ids (view = tile / tiles_per_view).  Each view's last key gets
// the single-view tail rule (Q10 with T-1 = the view's last tile); the plain end of a view's last tile is never written.
int launch_tile_ranges_views(const uint32_t *sorted_keys, const FrameState *frame, uint2 *bounds, uint32_t tiles_per_view, int quirks, int grid,
                             cudaStream_t stream);
int launch_band_fixup(const int32_t *global_last_plus1, float4 *out, int32_t width, int32_t height, int32_t tiles_x, int32_t num_tiles_total,
                      int32_t band_y0, int32_t band_y1, int32_t row_mod, int32_t row_rem, cudaStream_t stream);

struct CompositeArgs {
    const float4 *records;
    const uint32_t *values;
    const uint2 *bounds;
    float4 *out;             // W*H RGBA32F
    int32_t width, height, tiles_x;
    int32_t tile_begin;      // first tile id rendered (band_y0 * tiles_x, or the first owned row)
    int32_t row_step;        // distance in tile rows between consecutive owned rows (1 = contiguous band)
    int32_t num_tiles;       // tiles rendered
    float heatmap_factor;
    uint32_t target_tile_id; // 0xFFFFFFFF = none (rasterizer.gd:158)
    float4 *pick;            // tile_splat_pos buffer (gsplat_render.glsl:33-36)
    FrameState *frame;       // ticket counter (comp_head must be 0) + staged-instance counter
    int32_t count_staged;    // add this launch's consumed instances to frame->staged (0 for the pick re-dispatch)
    const uint32_t *order;   // optional: ticket k renders owned tile order[k] (longest chains first, launch_tile_order); nullptr = natural order
    uint32_t *consumed;      // optional [num_tiles]: chunks each owned tile blended before its stop rule fired | 1u << 31 (next frame's order hint)
    int32_t ctas_per_sm;     // resident CTAs per SM of the persistent grid
    int32_t sm_count;
    int32_t contract;        // 1: the gsr spec (explicit fma at the GLSL-legal contraction points); 0: no contraction (GSR_FLAG_UNCONTRACTED_BLEND)
    ulonglong4 *trace;       // optional schedule trace (debug): {tile<<32|smid, t0_ns, t1_ns, consumed<<32|list_chunks<<1|1}
    uint32_t *trace_count;
    uint32_t trace_cap;
    // multiview frame (zero = one view): tile id t renders tile t % tiles_per_view of view t / tiles_per_view, from record table
    // `records + view * record_stride` (float4s) into layer `out + view * layer_stride` (pixels)
    int32_t tiles_per_view;
    uint64_t layer_stride;
    uint64_t record_stride;
};
int launch_composite(const CompositeArgs &a, cudaStream_t stream);
int composite_max_ctas_per_sm(int *out);
// order[0 .. num_tiles) = owned-tile indices sorted by descending expected chain length: the chunk count the tile consumed in the
// previous frame (hint[k] with bit 31 set; the bit is cleared here) or, without a hint, its list length in chunks capped at
// `cap_chunks` (a list is rarely consumed beyond ~20 chunks).  Counting sort, one CTA.  Scheduling only: pixels do not depend on it.
// Sparse frames: when at most `sparse_tiles` owned tiles are occupied, frame->comp_cta_limit = sparse_cta_limit (one CTA per SM:
// a chain that has an SM to itself advances fastest); otherwise 0 = every launched CTA works.
int launch_tile_order(const uint2 *bounds, int32_t tile_begin, int32_t row_step, int32_t tiles_x, int32_t num_tiles, uint32_t *hint, uint32_t *order,
                      FrameState *frame, uint32_t sparse_tiles, uint32_t sparse_cta_limit, cudaStream_t stream);

int launch_ply_to_soa(const float *ply, uint32_t nprops, uint64_t count, float creation_time, float4 *soa, uint64_t plane_stride, uint64_t first,
                      cudaStream_t stream);
// present.cu: RGBA32F frame -> GSR_OUT_* (| GSR_OUT_SRGB_TO_LINEAR)
int launch_present(const float4 *rgba, void *out, uint64_t pixels, int format, cudaStream_t stream);
size_t present_bytes_per_pixel(int format);
int launch_aos_to_soa(const float4 *aos, uint64_t count, float4 *soa, uint64_t plane_stride, uint64_t first, cudaStream_t stream);

// cudaFuncGetAttributes on every kernel of a file: defeats lazy module loading before the first frame
int preload_group_kernels();
int preload_projection_kernels();
int preload_sort_kernels();
int preload_ranges_kernels();
int launch_frame_clear(FrameState *frame, unsigned long long *links, uint32_t n_links, uint2 *bounds, uint32_t n_bounds, cudaStream_t stream);
int preload_ingest_kernels();
int preload_present_kernels();
int preload_composite_kernels();

}  // namespace gsr
