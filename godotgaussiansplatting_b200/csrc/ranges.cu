// ranges.cu -- stage 3: tile-range scan.  Replaces gsplat_boundaries.glsl:23-50.
//
// Adjacent difference over the high 16 bits of the sorted keys -> uint2 bounds[tile] = (start, end).
// bounds is cleared to 0 before the launch (rasterizer.gd:128).  The element count M is read from
// FrameState on the device (the reference dispatches indirectly from grid_dims[3..5], rasterizer.gd:153).
//
// Reference quirks (Q10), reproduced when `quirks` != 0:
//   * the first occupied tile keeps start = 0 from the clear (correct by construction);
//   * every thread whose tile is T-1 stores bounds[T-1].y = M-1 (:47-49), dropping the final splat;
//   * the last OCCUPIED tile, when it is not tile T-1, never gets its end written and renders nothing
//     (gsplat_render.glsl:61: max(0, int(0 - start))).
// Sharded runs (`sharded` != 0): this context holds one tile-row band of the frame; its band-local last
// occupied tile is only "the frame's last occupied tile" if it equals FrameState.last_tile (computed by the
// projection over ALL splats); otherwise its end is M_local, exactly what the un-sharded scan would write.
#include "common.cuh"

namespace gsr {

namespace {

__device__ __forceinline__ void range_step(uint32_t id, uint32_t a, uint32_t b, uint32_t m, uint2 *__restrict__ bounds, uint32_t num_tiles, int quirks,
                                           int sharded, const FrameState *__restrict__ frame, int32_t *__restrict__ sync_word) {
    if (id > 0 && a != b) {   // gsplat_boundaries.glsl:39-42
        bounds[a].y = id;
        bounds[b].x = id;
    }
    if (id == m - 1) {  // tail rules for the last key's tile
        if (sync_word) *sync_word = (int32_t)b + 1;  // local last occupied tile (fast sharded mode: all-reduced by the host)
        if (quirks) {
            if (b == num_tiles - 1u) {
                if (m - 1u >= 1u) bounds[b].y = m - 1u;
            } else if (sharded == 2) {
                bounds[b].y = m;  // the frame-global "last occupied tile renders nothing" rule is applied by band_fixup_kernel
            } else if (sharded == 1 && (int32_t)b != frame->last_tile_plus1 - 1) {
                bounds[b].y = m;
            }
        } else {
            bounds[b].y = m;
        }
    }
}

// Four keys per thread and iteration from one 128-bit load (+ the predecessor of the first, an L1/L2 hit): the kernel is a pure
// streaming read of 4*M bytes and was latency-bound with one 4-byte load per thread (r01: 28 us for 38 MB).
__global__ void __launch_bounds__(256) tile_ranges_kernel(const uint32_t *__restrict__ keys, const FrameState *__restrict__ frame,
                                                          uint2 *__restrict__ bounds, uint32_t num_tiles, int quirks, int sharded,
                                                          int32_t *__restrict__ sync_word) {
    const uint32_t m = frame->dup_sorted;
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t quads = m >> 2;
    const uint4 *k4 = reinterpret_cast<const uint4 *>(keys);
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += stride) {
        const uint4 k = __ldg(k4 + q);
        const uint32_t id = q << 2;
        const uint32_t prev = id ? __ldg(keys + id - 1) >> 16 : 0u;
        const uint32_t t0 = k.x >> 16, t1 = k.y >> 16, t2 = k.z >> 16, t3 = k.w >> 16;
        range_step(id, prev, t0, m, bounds, num_tiles, quirks, sharded, frame, sync_word);
        range_step(id + 1, t0, t1, m, bounds, num_tiles, quirks, sharded, frame, sync_word);
        range_step(id + 2, t1, t2, m, bounds, num_tiles, quirks, sharded, frame, sync_word);
        range_step(id + 3, t2, t3, m, bounds, num_tiles, quirks, sharded, frame, sync_word);
    }
    for (uint32_t id = (quads << 2) + blockIdx.x * blockDim.x + threadIdx.x; id < m; id += stride) {   // ragged tail (< 4 keys)
        const uint32_t b = keys[id] >> 16;
        const uint32_t a = id ? keys[id - 1] >> 16 : 0u;
        range_step(id, a, b, m, bounds, num_tiles, quirks, sharded, frame, sync_word);
    }
}

// Multiview frame: keys carry tile ids v*T + tile.  A view's list is the single-view frame's list with every index offset by the
// view's first pair s_v, so the single-view rules apply per view: at a view boundary (key id-1 in view u, key id in a later view) the
// plain end of u's last tile is NOT written; u's last key instead gets the tail rule of range_step, where "m - 1 >= 1" (the view has
// at least two pairs) reads "key e-1 is in the same view"; the next view's first tile gets its start from the transition (a view
// starting at pair 0 keeps start 0 from the clear, as the single-view frame's first tile does).
__device__ __forceinline__ void view_tail(const uint32_t *__restrict__ keys, uint32_t e, uint32_t b, uint32_t T, uint2 *__restrict__ bounds, int quirks) {
    if (quirks) {
        if (b % T == T - 1u) {
            if (e >= 1u && (keys[e - 1] >> 16) / T == b / T) bounds[b].y = e;
        }
    } else {
        bounds[b].y = e + 1u;
    }
}

__device__ __forceinline__ void range_step_views(const uint32_t *__restrict__ keys, uint32_t id, uint32_t a, uint32_t b, uint32_t m, uint2 *__restrict__ bounds,
                                                 uint32_t T, int quirks) {
    if (id > 0 && a != b) {
        if (a / T == b / T) bounds[a].y = id;
        else view_tail(keys, id - 1u, a, T, bounds, quirks);
        bounds[b].x = id;
    }
    if (id == m - 1) view_tail(keys, id, b, T, bounds, quirks);
}

__global__ void __launch_bounds__(256) tile_ranges_views_kernel(const uint32_t *__restrict__ keys, const FrameState *__restrict__ frame,
                                                                uint2 *__restrict__ bounds, uint32_t tiles_per_view, int quirks) {
    const uint32_t m = frame->dup_sorted;
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t quads = m >> 2;
    const uint4 *k4 = reinterpret_cast<const uint4 *>(keys);
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += stride) {
        const uint4 k = __ldg(k4 + q);
        const uint32_t id = q << 2;
        const uint32_t prev = id ? __ldg(keys + id - 1) >> 16 : 0u;
        const uint32_t t0 = k.x >> 16, t1 = k.y >> 16, t2 = k.z >> 16, t3 = k.w >> 16;
        range_step_views(keys, id, prev, t0, m, bounds, tiles_per_view, quirks);
        range_step_views(keys, id + 1, t0, t1, m, bounds, tiles_per_view, quirks);
        range_step_views(keys, id + 2, t1, t2, m, bounds, tiles_per_view, quirks);
        range_step_views(keys, id + 3, t2, t3, m, bounds, tiles_per_view, quirks);
    }
    for (uint32_t id = (quads << 2) + blockIdx.x * blockDim.x + threadIdx.x; id < m; id += stride) {
        const uint32_t b = keys[id] >> 16;
        const uint32_t a = id ? keys[id - 1] >> 16 : 0u;
        range_step_views(keys, id, a, b, m, bounds, tiles_per_view, quirks);
    }
}

// Fast sharded mode, after the ranks have all-reduced (MAX) their local last occupied tile: the rank that owns the
// frame's last occupied tile L blanks it when L != T-1 -- in the reference that tile never gets its range end written
// (gsplat_boundaries.glsl:47-49) and therefore renders nothing: rgb = 0, heat-map term (1 - t) = 0, alpha = 1.
__global__ void __launch_bounds__(256) band_fixup_kernel(const int32_t *__restrict__ global_last_plus1, float4 *__restrict__ out, int32_t width,
                                                         int32_t height, int32_t tiles_x, int32_t num_tiles_total, int32_t band_y0, int32_t band_y1,
                                                         int32_t row_mod, int32_t row_rem) {
    const int32_t L = *global_last_plus1 - 1;
    if (L < 0 || L == num_tiles_total - 1) return;
    const int32_t ty = L / tiles_x, tx = L % tiles_x;
    if (ty < band_y0 || ty >= band_y1 || ty % row_mod != row_rem) return;  // another rank owns it
    const int32_t px = tx * TILE + (int32_t)(threadIdx.x & 15u), py = ty * TILE + (int32_t)(threadIdx.x >> 4);
    if (px < width && py < height) out[(uint64_t)py * (uint64_t)width + (uint64_t)px] = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
}

// Longest-chain-first order of the tiles a compositor launch owns (scheduling only: pixels do not depend on it).  One CTA: histogram
// of the expected chunk count in shared memory, descending exclusive scan, scatter.  Expected chunks = what the tile consumed in the
// previous frame when the compositor left a hint (bit 31 set), else min(list chunks, NO_HINT_CAP): beyond a few chunks the list
// length says little about where the tile-stop vote fires (measured on c3: lists of 16..360 chunks are all consumed to ~8 +- 4).
// Owned tile k <-> tile id exactly as in the compositor.
constexpr uint32_t ORDER_BINS = 64, ORDER_NO_HINT_CAP = 24;
__global__ void __launch_bounds__(1024) tile_order_kernel(const uint2 *__restrict__ bounds, int32_t tile_begin, int32_t row_step, int32_t tiles_x,
                                                          int32_t num_tiles, uint32_t *__restrict__ hint, uint32_t *__restrict__ order,
                                                          FrameState *__restrict__ frame, uint32_t sparse_tiles, uint32_t sparse_cta_limit) {
    __shared__ uint32_t s_hist[ORDER_BINS], s_base[ORDER_BINS];
    const uint32_t tid = threadIdx.x;
    if (tid < ORDER_BINS) s_hist[tid] = 0u;
    __syncthreads();
    auto bin_of = [&](int32_t k) -> uint32_t {
        const uint32_t tile = (uint32_t)tile_begin + ((uint32_t)k / (uint32_t)tiles_x) * (uint32_t)(row_step * tiles_x) + (uint32_t)k % (uint32_t)tiles_x;
        const uint2 b = bounds[tile];
        const int32_t d = (int32_t)(b.y - b.x);
        const uint32_t list = d > 0 ? ((uint32_t)d + 255u) >> 8 : 0u;
        uint32_t expect = list < ORDER_NO_HINT_CAP ? list : ORDER_NO_HINT_CAP;
        if (hint) {
            const uint32_t h = hint[k];
            if (h & 0x80000000u) {   // the chain can be at most one chunk longer per chunk the list grew; an empty list stays empty
                const uint32_t c = (h & 0x7FFFFFFFu) + 1u;
                expect = list < c ? list : c;
            }
        }
        return expect < ORDER_BINS - 1u ? expect : ORDER_BINS - 1u;
    };
    for (int32_t k = (int32_t)tid; k < num_tiles; k += 1024) atomicAdd(&s_hist[bin_of(k)], 1u);
    __syncthreads();
    if (tid == 0) {   // 64 bins: a serial descending scan is cheaper than a barrier tree
        uint32_t acc = 0u;
        for (int b = (int)ORDER_BINS - 1; b >= 0; --b) { s_base[b] = acc; acc += s_hist[b]; }
        // few chains (a sparse view, one rank's share of a multi-GPU frame): let each have an SM to itself
        if (frame) frame->comp_cta_limit = ((uint32_t)num_tiles - s_hist[0] <= sparse_tiles) ? sparse_cta_limit : 0u;
    }
    __syncthreads();
    for (int32_t k = (int32_t)tid; k < num_tiles; k += 1024) order[atomicAdd(&s_base[bin_of(k)], 1u)] = (uint32_t)k;
    __syncthreads();
    if (hint) for (int32_t k = (int32_t)tid; k < num_tiles; k += 1024) hint[k] &= 0x7FFFFFFFu;   // consumed: the compositor sets bit 31 again
}

// Start of a frame (rasterizer.gd:127-128): this frame's counters, the projection's scan links and the tile bounds back to zero.
// One kernel instead of three cudaMemsetAsync (fewer stream operations per frame); any of the three parts may be absent
// (overlapped frames clear the bounds at the start of the back part: gsr_api.cu).
__global__ void __launch_bounds__(256) frame_clear_kernel(unsigned long long *frame_words, uint32_t n_frame, unsigned long long *links, uint32_t n_links,
                                                            unsigned long long *bounds, uint32_t n_bounds) {
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t i0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (i0 < n_frame) frame_words[i0] = 0ull;
    for (uint32_t i = i0; i < n_links; i += stride) links[i] = 0ull;
    for (uint32_t i = i0; i < n_bounds; i += stride) bounds[i] = 0ull;
}

}  // namespace

#ifndef GSR_CPU_EMU  // tests/kernel_emu compiles the kernels above for the CPU; the launchers are CUDA only
int launch_frame_clear(FrameState *frame, unsigned long long *links, uint32_t n_links, uint2 *bounds, uint32_t n_bounds, cudaStream_t stream) {
    static_assert(sizeof(FrameState) % 8 == 0 && sizeof(uint2) == 8, "cleared as 64-bit words");
    const uint32_t most = n_links > n_bounds ? n_links : n_bounds;
    uint32_t grid = (most + 255u) / 256u;
    grid = grid < 1u ? 1u : (grid > 296u ? 296u : grid);
    frame_clear_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<unsigned long long *>(frame), frame ? (uint32_t)(sizeof(FrameState) / 8) : 0u, links, n_links,
                                                 reinterpret_cast<unsigned long long *>(bounds), n_bounds);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}

// Force-load this file's kernels (CUDA loads modules lazily; see gsr_create).
int preload_ranges_kernels() {
    cudaFuncAttributes fa;
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, tile_ranges_kernel));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, tile_ranges_views_kernel));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, band_fixup_kernel));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, tile_order_kernel));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, frame_clear_kernel));
    return GSR_OK;
}

int launch_tile_order(const uint2 *bounds, int32_t tile_begin, int32_t row_step, int32_t tiles_x, int32_t num_tiles, uint32_t *hint, uint32_t *order,
                      FrameState *frame, uint32_t sparse_tiles, uint32_t sparse_cta_limit, cudaStream_t stream) {
    if (num_tiles <= 0) return GSR_OK;
    tile_order_kernel<<<1, 1024, 0, stream>>>(bounds, tile_begin, row_step, tiles_x, num_tiles, hint, order, frame, sparse_tiles, sparse_cta_limit);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}

int launch_band_fixup(const int32_t *global_last_plus1, float4 *out, int32_t width, int32_t height, int32_t tiles_x, int32_t num_tiles_total,
                      int32_t band_y0, int32_t band_y1, int32_t row_mod, int32_t row_rem, cudaStream_t stream) {
    band_fixup_kernel<<<1, 256, 0, stream>>>(global_last_plus1, out, width, height, tiles_x, num_tiles_total, band_y0, band_y1, row_mod, row_rem);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}

int launch_tile_ranges(const uint32_t *sorted_keys, const FrameState *frame, uint2 *bounds, uint32_t num_tiles, int quirks,
                       int sharded, int32_t *sync_word, int grid, cudaStream_t stream) {
    tile_ranges_kernel<<<grid, 256, 0, stream>>>(sorted_keys, frame, bounds, num_tiles, quirks, sharded, sync_word);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}

int launch_tile_ranges_views(const uint32_t *sorted_keys, const FrameState *frame, uint2 *bounds, uint32_t tiles_per_view, int quirks, int grid,
                             cudaStream_t stream) {
    tile_ranges_views_kernel<<<grid, 256, 0, stream>>>(sorted_keys, frame, bounds, tiles_per_view, quirks);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}
#endif  // GSR_CPU_EMU

}  // namespace gsr
