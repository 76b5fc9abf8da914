// multiview_emu.cpp -- the multiview kernels of libgsr (projection_views_kernel, tile_ranges_views_kernel and the multiview
// composite_kernel) compiled for the CPU under the same shim as kernel_emu.cpp.
// TEST INFRASTRUCTURE: see cuda_shim.h.  Built by tests/test_multiview.py with the g++ flags of tests/kernel_emu/build.py.
#define GSR_CPU_EMU 1
#include <vector>

#include "cuda_shim.h"

namespace cuda_emu { dim g_block_dim{128, 1, 1}, g_grid_dim{1, 1, 1}; }
namespace gsr { void set_last_error(const char *, ...) {} }

#include "../../godotgaussiansplatting_b200/csrc/compositor.cu"
#include "../../godotgaussiansplatting_b200/csrc/ranges.cu"
#include "../../godotgaussiansplatting_b200/csrc/projection.cu"

namespace {
// the per-frame constants of gsr_api.cu frame_constants() (project_covariance's focal / limit terms), same IEEE operations
void view_constants(const float *vp, gsr::ProjectionArgs &pa) {
    const float tfi0 = vp[16 + 0], tfi1 = vp[16 + 5];
    const volatile float hw = (float)pa.u.dims[0] * 0.5f, hh = (float)pa.u.dims[1] * 0.5f;
    const volatile float f0 = hw * tfi0, f1 = hh * tfi1;
    const volatile float t0 = 1.0f / tfi0, t1 = 1.0f / tfi1;
    const volatile float n0 = -t0, n1 = -t1;
    pa.focal_base[0] = f0; pa.focal_base[1] = f1;
    pa.lim_lo[0] = n0 * 1.3f; pa.lim_lo[1] = n1 * 1.3f;
    pa.lim_hi[0] = t0 * 1.3f; pa.lim_hi[1] = t1 * 1.3f;
}
void views_body(void *p) { gsr::projection_views_kernel(*static_cast<const gsr::ViewsArgs *>(p)); }

struct RangesLaunch { const uint32_t *keys; const gsr::FrameState *frame; uint2 *bounds; uint32_t tpv; int quirks; };
void ranges_body(void *p) {
    const RangesLaunch *l = static_cast<const RangesLaunch *>(p);
    gsr::tile_ranges_views_kernel(l->keys, l->frame, l->bounds, l->tpv, l->quirks);
}

struct Launch { const gsr::CompositeArgs *args; int variant; };
void composite_body(void *p) {
    const Launch *l = static_cast<const Launch *>(p);
    if (l->variant == 1) gsr::composite_kernel<false, true>(*l->args);
    else gsr::composite_kernel<true, true>(*l->args);
}
}  // namespace

// K views (vps: K x 32 floats, uniforms: K x 32 bytes) of n splats; records: K tables of 3*n float4.  Returns M (true count).
extern "C" long long emu_projection_views(const void *soa, unsigned long long plane_stride, unsigned num_splats, int num_views, const float *vps,
                                          const void *uniforms, void *records, uint32_t *keys, uint32_t *values, unsigned capacity, int sh_bulk_min,
                                          unsigned *visible_out, int *last_tile_out) {
    if (num_views < 1 || num_views > GSR_MAX_VIEWS) return -1;
    gsr::ViewsArgs va;
    memset(&va, 0, sizeof va);
    gsr::FrameState frame;
    memset(&frame, 0, sizeof frame);
    const unsigned blocks = (num_splats + gsr::PROJ_THREADS - 1) / gsr::PROJ_THREADS;
    std::vector<unsigned long long> lookback(blocks ? blocks : 1, 0ull);
    va.num_views = num_views;
    for (int v = 0; v < num_views; ++v) {
        gsr::ProjectionArgs &pa = va.view[v];
        pa.soa = static_cast<const float4 *>(soa); pa.plane_stride = plane_stride; pa.num_splats = num_splats;
        memcpy(pa.vp, vps + 32 * v, sizeof pa.vp);
        memcpy(&pa.u, static_cast<const char *>(uniforms) + 32 * v, sizeof pa.u);
        view_constants(vps + 32 * v, pa);
        pa.band_y0 = 0; pa.band_y1 = (pa.u.dims[1] + 15) / 16; pa.row_mod = 1; pa.row_rem = 0;
        pa.sh_bulk_min = sh_bulk_min > 0 ? sh_bulk_min : 12;
        pa.records = static_cast<float4 *>(records) + 3ull * num_splats * (unsigned long long)v;
        pa.keys = keys; pa.values = values; pa.capacity = capacity;
        pa.lookback = lookback.data(); pa.frame = &frame;
    }
    va.tiles_per_view = (uint32_t)(((va.view[0].u.dims[0] + 15) / 16) * ((va.view[0].u.dims[1] + 15) / 16));
    cuda_emu::g_block_dim = cuda_emu::dim{(unsigned)gsr::PROJ_THREADS, 1, 1};
    cuda_emu::g_grid_dim = cuda_emu::dim{blocks, 1, 1};
    for (unsigned b = 0; b < blocks; ++b) glsl::run_workgroup(glsl::uvec3(b, 0, 0), glsl::uvec3((unsigned)gsr::PROJ_THREADS, 1, 1), &views_body, &va);
    cuda_emu::g_block_dim = cuda_emu::dim{128, 1, 1};
    cuda_emu::g_grid_dim = cuda_emu::dim{1, 1, 1};
    if (visible_out) *visible_out = frame.visible;
    if (last_tile_out) *last_tile_out = frame.last_tile_plus1 - 1;
    return (long long)frame.dup_total;
}

// bounds: num_views * tiles_per_view uint2, cleared here (rasterizer.gd:128); `grid` blocks of 256 threads, one after another
extern "C" int emu_tile_ranges_views(const uint32_t *sorted_keys, uint32_t m, uint32_t *bounds, uint32_t tiles_per_view, int num_views, int quirks, int grid) {
    gsr::FrameState frame;
    memset(&frame, 0, sizeof frame);
    frame.dup_total = m; frame.dup_sorted = m;
    memset(bounds, 0, sizeof(uint32_t) * 2 * (size_t)tiles_per_view * (size_t)num_views);
    RangesLaunch l{sorted_keys, &frame, reinterpret_cast<uint2 *>(bounds), tiles_per_view, quirks};
    cuda_emu::g_block_dim = cuda_emu::dim{256, 1, 1};
    cuda_emu::g_grid_dim = cuda_emu::dim{(unsigned)grid, 1, 1};
    for (int b = 0; b < grid; ++b) glsl::run_workgroup(glsl::uvec3((unsigned)b, 0, 0), glsl::uvec3(256, 1, 1), &ranges_body, &l);
    cuda_emu::g_block_dim = cuda_emu::dim{128, 1, 1};
    cuda_emu::g_grid_dim = cuda_emu::dim{1, 1, 1};
    return 0;
}

// One persistent block renders all K*T tiles in natural ticket order; records: K tables of 3*n float4, out: K layers of W*H RGBA32F.
extern "C" int emu_composite_views(int variant, const void *records, unsigned long long num_splats, const uint32_t *values, const uint32_t *bounds,
                                   float *out_rgba, int width, int height, int num_views, float heatmap_factor, uint32_t target_tile_id, float *pick4) {
    const int tiles_x = (width + 15) / 16, T = tiles_x * ((height + 15) / 16);
    gsr::FrameState frame;
    memset(&frame, 0, sizeof frame);
    gsr::CompositeArgs a;
    memset(&a, 0, sizeof a);
    a.records = static_cast<const float4 *>(records);
    a.values = values;
    a.bounds = reinterpret_cast<const uint2 *>(bounds);
    a.out = reinterpret_cast<float4 *>(out_rgba);
    a.width = width; a.height = height; a.tiles_x = tiles_x;
    a.tile_begin = 0; a.row_step = 1; a.num_tiles = T * num_views;
    a.heatmap_factor = heatmap_factor; a.target_tile_id = target_tile_id;
    a.pick = reinterpret_cast<float4 *>(pick4);
    a.frame = &frame; a.count_staged = 1;
    a.ctas_per_sm = 1; a.sm_count = 1; a.contract = variant == 1 ? 0 : 1;
    a.tiles_per_view = T; a.layer_stride = (uint64_t)width * (uint64_t)height; a.record_stride = 3ull * num_splats;
    Launch l{&a, variant};
    cuda_emu::g_block_dim = cuda_emu::dim{128, 1, 1};
    glsl::run_workgroup(glsl::uvec3(0, 0, 0), glsl::uvec3(128, 1, 1), &composite_body, &l);
    return frame.comp_head >= (uint32_t)a.num_tiles ? 0 : 1;
}
