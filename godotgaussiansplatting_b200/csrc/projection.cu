// projection.cu -- stage 1: projection + frustum cull + EWA 2-D covariance + SH colour + tile-key duplication.
//
// Replaces gsplat_projection.glsl:150-227 (one thread per splat).  Differences in *how*, not *what*:
//   * splat attributes are read from 15 SoA float4 planes (culled splats touch 16 B, not the 240-B AoS
//     struct; SH planes are only read for splats that actually emit keys);
//   * the single contended atomicAdd (:196) is replaced by a warp scan + decoupled look-back over the
//     projection warps (32 splats per link, no CTA barriers), so duplicate offsets are an exclusive prefix sum in splat-id order -- the
//     deterministic refinement of the reference's arbitrary atomic order (Q13);
//   * the per-thread serial emit loop (:219-226, up to hundreds of keys from one lane) is replaced by a
//     warp-cooperative emit: every output slot of the warp is produced by some lane (binary search
//     over the warp's 32 offsets), so writes are perfectly coalesced and load-balanced;
//   * M never leaves the GPU (the last warp of the scan stores it in FrameState) -- same as the reference, which
//     feeds it to indirect dispatches (:210-214).
// The arithmetic follows the "gsr deterministic math" contract (common.cuh): this file is compiled with
// -fmad=false, every operator below is one IEEE binary32 operation in GLSL parse order.
#include <string.h>

#include "common.cuh"

namespace gsr {

namespace {

constexpr float SH_C0 = 0.28209479177387814f;
constexpr float SH_C1 = 0.4886025119029199f;
constexpr float SH_C2_0 = 1.0925484305920792f;
constexpr float SH_C2_1 = 1.0925484305920792f;
constexpr float SH_C2_2 = 0.31539156525252005f;
constexpr float SH_C2_3 = 1.0925484305920792f;
constexpr float SH_C2_4 = 0.5462742152960396f;
constexpr float SH_C3_0 = 0.5900435899266435f;
constexpr float SH_C3_1 = 2.890611442640554f;
constexpr float SH_C3_2 = 0.4570457994644658f;
constexpr float SH_C3_3 = 0.3731763325901154f;
constexpr float SH_C3_4 = 0.4570457994644658f;
constexpr float SH_C3_5 = 1.445305721320277f;
constexpr float SH_C3_6 = 0.5900435899266435f;

#define LB_AGG (1ull << 62)
#define LB_PREFIX (2ull << 62)
#define LB_VAL ((1ull << 62) - 1ull)

struct Mat3 { float m[3][3]; };  // m[c][r], GLSL column-major

__device__ __forceinline__ float ease_out_cubic(float x) {  // gsplat_projection.glsl:87-90
    float a = 1.0f - x;
    return 1.0f - a * a * a;
}

__device__ __forceinline__ uint32_t warp_incl_scan_u32(uint32_t v, uint32_t lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= (uint32_t)o) v += t;
    }
    return v;
}

// Warp-parallel decoupled look-back over one 64-bit word per block.  Returns the exclusive prefix.
__device__ __forceinline__ unsigned long long lookback_exclusive(volatile unsigned long long *status, uint32_t bid,
                                                                 unsigned long long total, uint32_t lane) {
    // the caller has already published (bid == 0 ? PREFIX : AGGREGATE) | total
    if (bid == 0) return 0ull;
    unsigned long long excl = 0ull;
    int64_t start = (int64_t)bid - 1;
    while (true) {
        const int64_t t = start - (int64_t)lane;
        unsigned long long v = (t >= 0) ? status[t] : LB_PREFIX;
        while (__any_sync(0xffffffffu, (v >> 62) == 0ull)) {
            if ((v >> 62) == 0ull) v = status[t];
        }
        const uint32_t pmask = __ballot_sync(0xffffffffu, (v >> 62) == 2ull);
        const uint32_t first = pmask ? (uint32_t)(__ffs(pmask) - 1) : 32u;
        unsigned long long c = (lane <= first) ? (v & LB_VAL) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        excl += c;
        if (pmask) break;
        start -= 32;
    }
    if (lane == 0) status[bid] = LB_PREFIX | ((excl + total) & LB_VAL);
    return excl;
}

// ---- TMA (bulk async copy) + mbarrier helpers: SASS UBLKCP / SYNCS ----
#ifndef GSR_CPU_EMU
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}
#else  // tests/kernel_emu (CPU logic pre-flight): a bulk copy completes at once, so the barrier protocol is a no-op
inline void mbar_init(uint64_t *, uint32_t) {}
inline void fence_mbar_init() {}
inline void mbar_expect_tx(uint64_t *, uint32_t) {}
inline void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *) { memcpy(dst, src, bytes); }
inline void mbar_wait(uint64_t *, uint32_t) {}
#endif

// SH colour (gsplat_projection.glsl:94-121), streamed six planes (= 8 coefficients x RGB) at a time so that at
// most 24 coefficient registers are live.  `src[k * stride]` is SH plane k of this splat (shared slab or global).
template <bool FROM_SMEM>
__device__ __forceinline__ void sh_color(const float4 *src, uint64_t stride, float x, float y, float z, float col[3]) {
    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
    {
        float sh[24];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const float4 v = FROM_SMEM ? src[(uint64_t)k * stride] : __ldg(src + (uint64_t)k * stride);
            sh[4 * k + 0] = v.x; sh[4 * k + 1] = v.y; sh[4 * k + 2] = v.z; sh[4 * k + 3] = v.w;
        }
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
#define SHC(k) (sh[3 * (k) + ch])
            float r = 0.5f + SHC(0) * SH_C0;
            r = r - SHC(1) * SH_C1 * y;
            r = r + SHC(2) * SH_C1 * z;
            r = r - SHC(3) * SH_C1 * x;
            r = r + SHC(4) * SH_C2_0 * xy;
            r = r - SHC(5) * SH_C2_1 * yz;
            r = r + SHC(6) * SH_C2_2 * (2.0f * zz - xx - yy);
            r = r - SHC(7) * SH_C2_3 * xz;
#undef SHC
            col[ch] = r;
        }
    }
    {
        float sh[24];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const float4 v = FROM_SMEM ? src[(uint64_t)(6 + k) * stride] : __ldg(src + (uint64_t)(6 + k) * stride);
            sh[4 * k + 0] = v.x; sh[4 * k + 1] = v.y; sh[4 * k + 2] = v.z; sh[4 * k + 3] = v.w;
        }
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
#define SHC(k) (sh[3 * ((k) - 8) + ch])
            float r = col[ch];
            r = r + SHC(8) * SH_C2_4 * (xx - yy);
            r = r - SHC(9) * SH_C3_0 * y * (3.0f * xx - yy);
            r = r + SHC(10) * SH_C3_1 * x * yz;
            r = r - SHC(11) * SH_C3_2 * y * (4.0f * zz - xx - yy);
            r = r + SHC(12) * SH_C3_3 * z * (2.0f * zz - 3.0f * xx - 3.0f * yy);
            r = r - SHC(13) * SH_C3_4 * x * (4.0f * zz - xx - yy);
            r = r + SHC(14) * SH_C3_5 * z * (xx - yy);
            r = r - SHC(15) * SH_C3_6 * x * (xx - 3.0f * yy);
#undef SHC
            col[ch] = g_max(0.0f, r);
        }
    }
}

struct LaneOut {  // what one splat contributes (valid when n > 0)
    uint32_t n, x0, y0, w, depth;
    int32_t last_tile;
    float4 r0, r1;  // record words 0,1
    float opacity, vx, vy, vz;
};

// gsplat_projection.glsl:158-218 for one splat given its plane-0..2 values.  Returns false when the splat is culled (or,
// in fast sharded mode, provably outside this context's rows).  QUICK: stop after the cull + conservative reject.
template <bool QUICK>
__device__ __forceinline__ bool project_lane(const ProjectionArgs &a, const float4 pt, const float4 ca, const float4 cb, LaneOut &o) {
    const float *V = a.vp, *P = a.vp + 16;  // X[c][r] = X[4*c + r]
    const int W = a.u.dims[0], H = a.u.dims[1];
    const uint32_t gx = (uint32_t)((W + TILE - 1) / TILE), gy = (uint32_t)((H + TILE - 1) / TILE);
    const float ms = a.u.model_scale;
    o.n = 0; o.last_tile = -1;
            // :158-166 frustum cull
            const float sp0 = pt.x * ms, sp1 = pt.y * ms, sp2 = pt.z * ms;
            float view[4], clip[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) view[r] = ((V[0 + r] * sp0 + V[4 + r] * sp1) + V[8 + r] * sp2) + V[12 + r] * 1.0f;
#pragma unroll
            for (int r = 0; r < 4; ++r) clip[r] = ((P[0 + r] * view[0] + P[4 + r] * view[1]) + P[8 + r] * view[2]) + P[12 + r] * view[3];
            const float vb = clip[3] * 1.2f;
            if (clip[0] < -vb || clip[1] < -vb || clip[2] < 0.0f || clip[0] > vb || clip[1] > vb || clip[2] > clip[3]) return false;


            // :169-174 load-in animation
            const float splat_time = a.u.time - pt.w;
            const float tf = ease_out_cubic(g_clamp(splat_time, 0.0f, 1.0f));
            const float tfl = ease_out_cubic(g_clamp(splat_time - 0.35f, 0.0f, 1.0f));
            const float splat_opacity = cb.z * tfl * tfl;
            const float splat_scale = ms * (2.0f * (1.0f - tfl) + 1.0f * tfl);

            // per-frame constants (focal = dims*0.5*tan_fov_inv, +-tan_fov*1.3) are evaluated once on the host with
            // the same IEEE operations (ProjectionArgs::focal_base, lim_lo, lim_hi)
            const float z_inv = 1.0f / view[2];
            const float focal0 = a.focal_base[0] * z_inv, focal1 = a.focal_base[1] * z_inv;
            const float mx = g_clamp(view[0] * z_inv, a.lim_lo[0], a.lim_hi[0]);
            const float my = g_clamp(view[1] * z_inv, a.lim_lo[1], a.lim_hi[1]);
            const float ndc0 = clip[0] / clip[3], ndc1 = clip[1] / clip[3], ndc2 = clip[2] / clip[3];
            const float ipx = ((ndc0 + 1.0f) * 0.5f - 1.0f * (1.0f - tf)) * (float)(W - 1);
            const float ipy = ((ndc1 + 1.0f) * 0.5f - 0.75f * (1.0f - tf)) * (float)(H - 1);

            if (a.fast_reject) {
                // Sharded fast mode: a CONSERVATIVE radius decides whether the splat can touch a tile row this context
                // owns; if not, the exact math below would end in "nt == 0" anyway.  With e1 <= trace(cov_2d) + 0.32,
                // trace(J W S' W^T J^T) <= lambda_max(S') |J|_F^2 |W|_2^2 <= |S'|_F |J|_F^2 |W|_2^2 and pow(op, 0.2) <= max(1, op):
                //   radius <= max(1, op) * 2.5 * sqrt(|S'|_F |J|_F^2 |W|_2^2 + 0.92)        (w_norm2 >= |W|_2^2 from the host)
                const float sf2 = (ca.x * ca.x + ca.w * ca.w + cb.y * cb.y) + 2.0f * (ca.y * ca.y + ca.z * ca.z + cb.x * cb.x);
                const float lam = sqrtf(sf2) * splat_scale * splat_scale * 1.0001f;
                const float jf2 = focal0 * focal0 + focal1 * focal1 * (1.0f + mx * mx + my * my);
                const float rb = g_max(1.0f, splat_opacity) * 2.5f * sqrtf(lam * jf2 * a.w_frob2 + 0.92f) * 1.001f + 1.0f;
                const float fa = floorf((ipy - rb) * 0.0625f), fb = floorf((ipy + rb) * 0.0625f);
                if (fa == fa && fb == fb && fabsf(fa) < 1.0e9f && fabsf(fb) < 1.0e9f) {  // finite: otherwise let the exact path decide
                    int32_t lo = (int32_t)fa, hi = (int32_t)fb;
                    if (lo < a.band_y0) lo = a.band_y0;
                    if (hi > a.band_y1 - 1) hi = a.band_y1 - 1;
                    if (hi < lo) return false;
                    const int32_t first = lo + ((a.row_rem - lo % a.row_mod) + a.row_mod) % a.row_mod;
                    if (first > hi) return false;
                }
            }

            if (QUICK) return true;  // compaction pass: cull + conservative reject only

            // :124-142 project_covariance
            Mat3 cov3 = {{{ca.x, ca.y, ca.z}, {ca.y, ca.w, cb.x}, {ca.z, cb.x, cb.y}}};
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int r = 0; r < 3; ++r) cov3.m[c][r] = cov3.m[c][r] * splat_scale * splat_scale;
            // jacobian columns (focal.x, 0, -focal.y*mean.x), (0, focal.y, -focal.y*mean.y), 0 (:134-137).  gsr spec: the
            // structurally-zero terms of b = transpose(mat3(view)) * jacobian are skipped; only the three entries of
            // cov_2d = transpose(b) * cov_3d * b that :141 reads are formed.  B0[r] = b[0][r], B1[r] = b[1][r].
            const float j02 = -focal1 * mx, j12 = -focal1 * my;
            float B0[3], B1[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                B0[r] = V[4 * r + 0] * focal0 + V[4 * r + 2] * j02;
                B1[r] = V[4 * r + 1] * focal1 + V[4 * r + 2] * j12;
            }
            // t1 = transpose(b) * cov_3d: T0[c] = t1[c][0] = sum_k b[0][k]*cov3[c][k], T1[c] = t1[c][1]
            float T0[3], T1[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                T0[c] = (B0[0] * cov3.m[c][0] + B0[1] * cov3.m[c][1]) + B0[2] * cov3.m[c][2];
                T1[c] = (B1[0] * cov3.m[c][0] + B1[1] * cov3.m[c][1]) + B1[2] * cov3.m[c][2];
            }
            // cov_2d[c][r] = sum_k t1[k][r] * b[c][k]
            const float c2_00 = (T0[0] * B0[0] + T0[1] * B0[1]) + T0[2] * B0[2];
            const float c2_01 = (T1[0] * B0[0] + T1[1] * B0[1]) + T1[2] * B0[2];
            const float c2_11 = (T1[0] * B1[0] + T1[1] * B1[1]) + T1[2] * B1[2];
            const float cx = c2_00 + 0.3f, cy = c2_01, cz = c2_11 + 0.3f;

            // :177-182
            const float det = cx * cz - cy * cy;
            if (det == 0.0f) return false;
            const float mid = 0.5f * (cx + cz);
            const float sq = sqrtf(g_max(0.1f, mid * mid - det));
            const float e1 = mid + 1.0f * sq, e2 = mid + -1.0f * sq;
            if (e1 < 0.0f || e2 < 0.0f) return false;

            // :184-185 ndc / image_pos: computed above (same operations), before the early reject

            // :190-194
            const float radius = det_pow(splat_opacity, 0.2f) * 2.5f * sqrtf(g_max(e1, e2));
            if (!(fabsf(ipx) <= 3.0e38f) || !(fabsf(ipy) <= 3.0e38f) || !(radius <= 3.0e38f)) return false;  // gsr spec: non-finite => culled
            const float fgx = (float)gx, fgy = (float)gy;
            int32_t x0 = (int32_t)g_clamp((ipx - radius) / 16.0f, 0.0f, fgx);
            int32_t y0 = (int32_t)g_clamp((ipy - radius) / 16.0f, 0.0f, fgy);
            int32_t x1 = (int32_t)g_clamp(ceilf((ipx + radius) / 16.0f), 0.0f, fgx);
            int32_t y1 = (int32_t)g_clamp(ceilf((ipy + radius) / 16.0f), 0.0f, fgy);
            // largest tile of the un-banded rect (global Q10 bookkeeping for exact sharded runs)
            if ((uint32_t)(x1 - x0) * (uint32_t)(y1 - y0) != 0u) o.last_tile = (y1 - 1) * (int32_t)gx + (x1 - 1);
            if (y0 < a.band_y0) y0 = a.band_y0;
            if (y1 > a.band_y1) y1 = a.band_y1;
            if (y1 < y0) y1 = y0;
            // rows of [y0, y1) owned by this context: y0' = first row with row % row_mod == row_rem, then every row_mod-th
            int32_t nrows = y1 - y0;
            if (a.row_mod > 1) {
                y0 += ((a.row_rem - y0 % a.row_mod) + a.row_mod) % a.row_mod;
                nrows = y0 < y1 ? (y1 - 1 - y0) / a.row_mod + 1 : 0;
            }
            const uint32_t nt = (uint32_t)(x1 - x0) * (uint32_t)nrows;
            if (a.fast_mode) o.last_tile = nt ? (y0 + (nrows - 1) * a.row_mod) * (int32_t)gx + (x1 - 1) : -1;  // LOCAL last tile
            if (nt == 0u) return false;

            // :198-206 everything of the record except the colour
            const float d0 = sp0 - a.u.camera_pos[0], d1 = sp1 - a.u.camera_pos[1], d2 = sp2 - a.u.camera_pos[2];
            const float inv_len = 1.0f / sqrtf((d0 * d0 + d1 * d1) + d2 * d2);
            o.vx = d0 * inv_len; o.vy = d1 * inv_len; o.vz = d2 * inv_len; o.opacity = splat_opacity;
            o.r0.x = ipx; o.r0.y = ipy; o.r0.z = sp0; o.r0.w = sp1;                        // image_pos, pos_xy
            o.r1.x = cz / det; o.r1.y = -cy / det; o.r1.z = cx / det; o.r1.w = sp2;        // conic, pos_z
            // :218
            o.depth = ((uint32_t)(ndc2 * ndc2 * ndc2 * 65535.0f)) & 0xFFFFu;
            o.n = nt; o.x0 = (uint32_t)x0; o.y0 = (uint32_t)y0; o.w = (uint32_t)(x1 - x0);

    return true;
}

// One warp = 32 consecutive splats; one CTA (8 warps, 256 splats) = one link of the chained scan.  There is no CTA
// barrier after the ticket broadcast: warps meet only through shared-memory flags.  Data movement per warp:
//   phase 1: lane 0 issues three 512-byte TMA bulk copies (planes 0-2: position/time, covariance, opacity of the
//            warp's 32 splats) into the warp's shared slab and everybody waits on the warp's mbarrier;
//            cull + EWA + rect => duplicate count; the last warp of the CTA to get here publishes the CTA
//            aggregate, before phase 2, so that successor CTAs never wait on this CTA's colour work;
//   phase 2: if at least `sh_bulk_min` lanes emit keys, twelve more 512-byte bulk copies bring the SH planes
//            (6 KB in flight per warp at zero register cost); otherwise the few live lanes gather their
//            192 bytes with plain 128-bit loads (sparse view / out-of-band warps of a multi-GPU shard);
//   then records are written, the closer's look-back resolves the CTA's base offset, and every warp emits its keys.
constexpr int PROJ_WARPS = PROJ_THREADS / 32;
#ifndef GSR_PROJ_MIN_BLOCKS
#define GSR_PROJ_MIN_BLOCKS 3
#endif
constexpr size_t PROJ_SLAB_BYTES = sizeof(float4) * NUM_PLANES * 32;             // 7680 B per warp
constexpr size_t PROJ_SMEM_BYTES = PROJ_SLAB_BYTES * PROJ_WARPS;                // 61440 B per CTA

__global__ void __launch_bounds__(PROJ_THREADS, GSR_PROJ_MIN_BLOCKS) projection_kernel(const __grid_constant__ ProjectionArgs a) {
#ifndef GSR_CPU_EMU
    extern __shared__ __align__(128) unsigned char proj_smem[];
#else
    __shared__ __align__(128) unsigned char proj_smem[PROJ_SMEM_BYTES];
#endif
    __shared__ uint32_t s_bid;
    __shared__ __align__(8) uint64_t s_bar[PROJ_WARPS][2];
    __shared__ uint32_t s_wtotal[PROJ_WARPS];   // duplicate count of each warp
    __shared__ uint32_t s_count, s_ready, s_nvis;
    __shared__ int32_t s_last;
    __shared__ unsigned long long s_cta_base;
    __shared__ uint4 s_res[PROJ_THREADS];     // compaction path: (n, x0|y0<<16, w|depth<<16, last_tile) per splat slot
    __shared__ uint16_t s_list[PROJ_THREADS]; // compaction path: slots of the surviving splats
    __shared__ uint32_t s_ncomp;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    float4 *slab = reinterpret_cast<float4 *>(proj_smem + (size_t)warp * PROJ_SLAB_BYTES);  // [15][32]
    if (lane == 0) {
        mbar_init(&s_bar[warp][0], 1);
        mbar_init(&s_bar[warp][1], 1);
        fence_mbar_init();
    }
    if (tid == 0) {
        s_bid = atomicAdd(&a.frame->proj_ticket, 1u);
        s_count = 0u; s_ready = 0u; s_nvis = 0u; s_last = -1; s_ncomp = 0u;
    }
    __syncthreads();
    const uint32_t bid = s_bid;                      // position of this CTA in the chained scan
    const uint32_t vwarp = bid * PROJ_WARPS + warp;  // 32 consecutive splats
    const uint32_t id0 = vwarp * 32u;
    const uint32_t id = id0 + lane;

    // ---- phase 1: TMA the warp's slices of planes 0..2 (planes are padded to a multiple of 256 splats) ----
    if (lane == 0) {
        mbar_expect_tx(&s_bar[warp][0], 3u * 512u);
#pragma unroll
        for (int k = 0; k < 3; ++k) bulk_g2s(slab + k * 32, a.soa + (uint64_t)k * a.plane_stride + id0, 512u, &s_bar[warp][0]);
    }

    const uint32_t gx = (uint32_t)((a.u.dims[0] + TILE - 1) / TILE);

    uint32_t n = 0, x0u = 0, y0u = 0, wu = 0, depth = 0;
    int32_t last_tile = -1;
    float4 r0, r1;           // record words 0,1 (valid when n > 0)
    float splat_opacity = 0.0f, vx = 0.0f, vy = 0.0f, vz = 0.0f;

    mbar_wait(&s_bar[warp][0], 0);
    bool colour_done = false;  // compaction path: records (incl. colour) are already written
    if (!a.fast_reject) {
        if (id < a.num_splats) {
            LaneOut o;
            if (project_lane<false>(a, slab[lane], slab[32 + lane], slab[64 + lane], o) && o.n) {
                n = o.n; x0u = o.x0; y0u = o.y0; wu = o.w; depth = o.depth;
                r0 = o.r0; r1 = o.r1; splat_opacity = o.opacity; vx = o.vx; vy = o.vy; vz = o.vz;
            }
            last_tile = o.last_tile;
        }
    } else {
        // ---- fast sharded mode with CTA-level compaction.  Under SIMT a warp only saves the expensive EWA / pow / SH
        //      work if ALL its lanes are rejected, and with cyclic rows 1/G of the lanes survive in nearly every warp.
        //      So: every lane runs the cheap cull + conservative reject, the survivors of the CTA's 256 splats are
        //      compacted into s_list, and dense warps run the full math for them (results go back to the splat's own
        //      slot, so scan and emit below are unchanged and the emission order stays the splat-id order).
        bool live = false;
        LaneOut q;
        if (id < a.num_splats) live = project_lane<true>(a, slab[lane], slab[32 + lane], slab[64 + lane], q);
        s_res[tid] = make_uint4(0u, 0u, 0u, 0xFFFFFFFFu);
        const uint32_t lmask = __ballot_sync(0xffffffffu, live);
        uint32_t wbase = 0;
        if (lane == 0 && lmask) wbase = atomicAdd(&s_ncomp, (uint32_t)__popc(lmask));
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
        if (live) s_list[wbase + __popc(lmask & ((1u << lane) - 1u))] = (uint16_t)tid;
        __syncthreads();
        const uint32_t nsurv = s_ncomp;
        if (tid < nsurv) {
            const uint32_t li = s_list[tid];
            const float4 *sl = reinterpret_cast<const float4 *>(proj_smem + (size_t)(li >> 5) * PROJ_SLAB_BYTES);
            const uint32_t l2 = li & 31u;
            const uint32_t gid = bid * PROJ_THREADS + li;
            LaneOut o;
            if (project_lane<false>(a, sl[l2], sl[32 + l2], sl[64 + l2], o) && o.n) {
                float col[3];
                sh_color<false>(a.soa + 3ull * a.plane_stride + gid, a.plane_stride, o.vx, o.vy, o.vz, col);
                float4 *rec = a.records + (uint64_t)gid * 3u;
                rec[0] = o.r0; rec[1] = o.r1; rec[2] = make_float4(col[0], col[1], col[2], o.opacity);
                s_res[li] = make_uint4(o.n, o.x0 | (o.y0 << 16), o.w | (o.depth << 16), (uint32_t)o.last_tile);
            }
        }
        __syncthreads();
        const uint4 r = s_res[tid];
        n = r.x; x0u = r.y & 0xFFFFu; y0u = r.y >> 16; wu = r.z & 0xFFFFu; depth = r.z >> 16; last_tile = (int32_t)r.w;
        colour_done = true;
    }

    // ---- warp scan of the duplicate counts; the warp that finishes phase 1 LAST in its CTA (the "closer") publishes
    //      the CTA aggregate -- before anybody's colour phase -- and later resolves the CTA's base offset ----
    const uint32_t incl = warp_incl_scan_u32(n, lane);
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t emit_mask = __ballot_sync(0xffffffffu, n != 0u);
    const uint32_t nvis = __popc(emit_mask);
    const int32_t wl = __reduce_max_sync(0xffffffffu, last_tile);
    bool closer = false;
    uint32_t cta_total = 0;
    if (lane == 0) {
        s_wtotal[warp] = total;
        if (nvis) atomicAdd(&s_nvis, nvis);
        if (wl >= 0) atomicMax(&s_last, wl);
        __threadfence_block();
        closer = atomicAdd(&s_count, 1u) == PROJ_WARPS - 1;
        if (closer) {
            __threadfence_block();
#pragma unroll
            for (int w = 0; w < PROJ_WARPS; ++w) cta_total += ((volatile uint32_t *)s_wtotal)[w];
            volatile unsigned long long *st = a.lookback + bid;
            *st = (bid == 0 ? LB_PREFIX : LB_AGG) | (unsigned long long)cta_total;
        }
    }
    closer = __shfl_sync(0xffffffffu, (int)closer, 0) != 0;
    cta_total = __shfl_sync(0xffffffffu, cta_total, 0);

    // ---- phase 2: SH planes -> colour -> record.  The closer resolves the CTA's base (decoupled look-back over the
    //      CTA aggregates) while its SH bulk copies are in flight, so the other warps rarely find `s_ready` unset ----
    const bool bulk = !colour_done && nvis >= (uint32_t)a.sh_bulk_min;
    if (bulk && lane == 0) {
        mbar_expect_tx(&s_bar[warp][1], 12u * 512u);
#pragma unroll
        for (int k = 3; k < NUM_PLANES; ++k) bulk_g2s(slab + k * 32, a.soa + (uint64_t)k * a.plane_stride + id0, 512u, &s_bar[warp][1]);
    }
    if (closer) {
        const unsigned long long cta_base = lookback_exclusive(a.lookback, bid, (unsigned long long)cta_total, lane);
        if (lane == 0) {
            s_cta_base = cta_base;
            __threadfence_block();
            *(volatile uint32_t *)&s_ready = 1u;
            const uint32_t nv = *(volatile uint32_t *)&s_nvis;
            const int32_t lt = *(volatile int32_t *)&s_last;
            if (nv) atomicAdd(&a.frame->visible, nv);
            if (lt >= 0) atomicMax(&a.frame->last_tile_plus1, lt + 1);
            if (bid == gridDim.x - 1) {  // tickets are dense: this CTA closes the scan => M is known
                const unsigned long long m = cta_base + cta_total;
                a.frame->dup_total = m;
                a.frame->dup_sorted = m < (unsigned long long)a.capacity ? (uint32_t)m : a.capacity;
                a.frame->overflow = m > (unsigned long long)a.capacity ? 1u : 0u;
            }
        }
    }
    if (bulk) {
        mbar_wait(&s_bar[warp][1], 0);
        if (n) {
            float col[3];
            sh_color<true>(slab + 3 * 32 + lane, 32, vx, vy, vz, col);
            float4 *rec = a.records + (uint64_t)id * 3u;
            rec[0] = r0; rec[1] = r1; rec[2] = make_float4(col[0], col[1], col[2], splat_opacity);
        }
    } else if (n && !colour_done) {
        float col[3];
        sh_color<false>(a.soa + 3ull * a.plane_stride + id, a.plane_stride, vx, vy, vz, col);
        float4 *rec = a.records + (uint64_t)id * 3u;
        rec[0] = r0; rec[1] = r1; rec[2] = make_float4(col[0], col[1], col[2], splat_opacity);
    }

    unsigned long long base = 0;
    if (lane == 0) {
        while (*(volatile uint32_t *)&s_ready == 0u) __nanosleep(100);
        __threadfence_block();
        base = *(volatile unsigned long long *)&s_cta_base;
        for (uint32_t w = 0; w < warp; ++w) base += ((volatile uint32_t *)s_wtotal)[w];
    }
    base = __shfl_sync(0xffffffffu, base, 0);

    // ---- emit (:219-226): key slot base + off + j holds tile j (row-major) of the splat's rect.  Rects of up to
    //      EMIT_SMALL tiles (the common case: M/V ~ 1.6) are written by their own lane -- neighbouring lanes own
    //      neighbouring slots, so the stores still coalesce; larger rects are emitted by the whole warp, 32 tiles per
    //      step, which keeps one huge splat from serialising a lane for hundreds of iterations. ----
    constexpr uint32_t EMIT_SMALL = 4;
    const uint32_t my_off = incl - n;
    if (n != 0u && n <= EMIT_SMALL) {
        uint32_t x = x0u, y = y0u;
        const uint32_t x1 = x0u + wu;
#pragma unroll
        for (uint32_t j = 0; j < EMIT_SMALL; ++j) {
            if (j < n) {
                const unsigned long long g = base + my_off + j;
                if (g < (unsigned long long)a.capacity) {
                    a.keys[g] = ((y * gx + x) << 16) | depth;
                    a.values[g] = id;
                }
                if (++x == x1) { x = x0u; y += (uint32_t)a.row_mod; }
            }
        }
    }
    uint32_t big = __ballot_sync(0xffffffffu, n > EMIT_SMALL);
    while (big) {
        const int src = __ffs(big) - 1;
        big &= big - 1u;
        const uint32_t sn = __shfl_sync(0xffffffffu, n, src), soff = __shfl_sync(0xffffffffu, my_off, src);
        const uint32_t sx0 = __shfl_sync(0xffffffffu, x0u, src), sy0 = __shfl_sync(0xffffffffu, y0u, src);
        const uint32_t sw = __shfl_sync(0xffffffffu, wu, src), sdepth = __shfl_sync(0xffffffffu, depth, src);
        for (uint32_t j = lane; j < sn; j += 32u) {
            const uint32_t ry = j / sw, rx = j - ry * sw;
            const unsigned long long g = base + soff + j;
            if (g < (unsigned long long)a.capacity) {
                a.keys[g] = (((sy0 + ry * (uint32_t)a.row_mod) * gx + sx0 + rx) << 16) | sdepth;
                a.values[g] = id0 + (uint32_t)src;
            }
        }
    }
}

// ==============================================================================================================
// Sharded variant (fast sharded mode with GSR_FLAG_FAST_REJECT): compaction domain = 1024 splats per CTA.
// With cyclic tile rows only ~1/G of the splats can touch this rank, but under SIMT a warp pays for the expensive
// part (EWA, pow, SH, record) unless all 32 lanes are rejected.  So the CTA (8 warps) first runs the cheap
// cull + conservative row test for 4 x 256 consecutive splats (planes 0-2 of all of them are TMA-staged up front: 48 KB),
// compacts the survivors, and only then runs the full math on dense warps -- with ~1024/G survivors there is enough
// work to keep all 8 warps busy (a 256-splat domain left 2 of 8 busy and was slower than no reject at all).  Results go
// back to the splat's own slot, so the scan and the emit see splat-id order exactly like projection_kernel.
constexpr int SH_GROUPS = 4;
constexpr int SH_SPLATS = SH_GROUPS * PROJ_THREADS;  // 1024 splats per CTA = one link of the chained scan
constexpr size_t SH_SLAB_BYTES = sizeof(float4) * 3 * SH_SPLATS;  // planes 0..2 of the CTA's splats: [group][warp][plane][lane]

__global__ void __launch_bounds__(PROJ_THREADS, 3) projection_sharded_kernel(const __grid_constant__ ProjectionArgs a) {
#ifndef GSR_CPU_EMU
    extern __shared__ __align__(128) unsigned char proj_smem[];
#else
    __shared__ __align__(128) unsigned char proj_smem[SH_SLAB_BYTES];
#endif
    __shared__ uint4 s_res[SH_SPLATS];      // (n, x0|y0<<16, w|depth<<16, last_tile) per splat slot
    __shared__ uint16_t s_list[SH_SPLATS];  // slots of the surviving splats
    __shared__ __align__(8) uint64_t s_bar[PROJ_WARPS];
    __shared__ uint32_t s_bid, s_ncomp, s_wsum[PROJ_WARPS], s_nvis;
    __shared__ int32_t s_last;
    __shared__ unsigned long long s_base;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    float4 *slab = reinterpret_cast<float4 *>(proj_smem);
    auto slab_at = [&](uint32_t slot, int plane) -> const float4 & {  // slot = group*256 + warp*32 + lane
        return slab[((slot >> 5) * 3u + (uint32_t)plane) * 32u + (slot & 31u)];
    };
    if (lane == 0) { mbar_init(&s_bar[warp], 1); fence_mbar_init(); }
    if (tid == 0) { s_bid = atomicAdd(&a.frame->proj_ticket, 1u); s_ncomp = 0u; s_nvis = 0u; s_last = -1; }
#pragma unroll
    for (int r = 0; r < SH_GROUPS; ++r) s_res[r * PROJ_THREADS + tid] = make_uint4(0u, 0u, 0u, 0xFFFFFFFFu);
    __syncthreads();
    const uint32_t bid = s_bid;
    const uint32_t base_id = bid * SH_SPLATS;
    const uint32_t gx = (uint32_t)((a.u.dims[0] + TILE - 1) / TILE);

    // ---- TMA: planes 0..2 of the warp's four 32-splat slices (12 x 512 B onto the warp's mbarrier) ----
    if (lane == 0) {
        mbar_expect_tx(&s_bar[warp], 12u * 512u);
#pragma unroll
        for (int g = 0; g < SH_GROUPS; ++g)
#pragma unroll
            for (int k = 0; k < 3; ++k)
                bulk_g2s(slab + ((g * PROJ_WARPS + warp) * 3u + k) * 32u, a.soa + (uint64_t)k * a.plane_stride + base_id + g * PROJ_THREADS + warp * 32u,
                         512u, &s_bar[warp]);
    }
    mbar_wait(&s_bar[warp], 0);

    // ---- quick pass: cull + conservative row test, CTA-wide compaction of the survivors ----
#pragma unroll
    for (int g = 0; g < SH_GROUPS; ++g) {
        const uint32_t slot = g * PROJ_THREADS + tid;
        bool live = false;
        LaneOut q;
        if (base_id + slot < a.num_splats) live = project_lane<true>(a, slab_at(slot, 0), slab_at(slot, 1), slab_at(slot, 2), q);
        const uint32_t lmask = __ballot_sync(0xffffffffu, live);
        uint32_t wbase = 0;
        if (lane == 0 && lmask) wbase = atomicAdd(&s_ncomp, (uint32_t)__popc(lmask));
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
        if (live) s_list[wbase + __popc(lmask & ((1u << lane) - 1u))] = (uint16_t)slot;
    }
    __syncthreads();

    // ---- dense pass: full math + SH colour + record for the survivors ----
    const uint32_t nsurv = s_ncomp;
    for (uint32_t it = tid; it < nsurv; it += PROJ_THREADS) {
        const uint32_t slot = s_list[it];
        const uint32_t gid = base_id + slot;
        LaneOut o;
        const bool hit = project_lane<false>(a, slab_at(slot, 0), slab_at(slot, 1), slab_at(slot, 2), o);
        if (hit && o.n) {
            float col[3];
            sh_color<false>(a.soa + 3ull * a.plane_stride + gid, a.plane_stride, o.vx, o.vy, o.vz, col);
            float4 *rec = a.records + (uint64_t)gid * 3u;
            rec[0] = o.r0; rec[1] = o.r1; rec[2] = make_float4(col[0], col[1], col[2], o.opacity);
            s_res[slot] = make_uint4(o.n, o.x0 | (o.y0 << 16), o.w | (o.depth << 16), (uint32_t)o.last_tile);
        }
    }
    __syncthreads();

    // ---- scan: thread t owns the four consecutive slots 4t .. 4t+3 (splat-id order) ----
    uint4 r[SH_GROUPS];
    uint32_t tsum = 0, tvis = 0;
    int32_t tlast = -1;
#pragma unroll
    for (int j = 0; j < SH_GROUPS; ++j) {
        r[j] = s_res[SH_GROUPS * tid + j];
        tsum += r[j].x;
        tvis += r[j].x != 0u;
        tlast = tlast > (int32_t)r[j].w ? tlast : (int32_t)r[j].w;
    }
    const uint32_t incl = warp_incl_scan_u32(tsum, lane);
    if (lane == 31) s_wsum[warp] = incl;
    const uint32_t wvis = __reduce_add_sync(0xffffffffu, tvis);
    const int32_t wlast = __reduce_max_sync(0xffffffffu, tlast);
    if (lane == 0) {
        if (wvis) atomicAdd(&s_nvis, wvis);
        if (wlast >= 0) atomicMax(&s_last, wlast);
    }
    __syncthreads();
    uint32_t woff = 0, total = 0;
#pragma unroll
    for (uint32_t w = 0; w < PROJ_WARPS; ++w) {
        const uint32_t sw = s_wsum[w];
        if (w < warp) woff += sw;
        total += sw;
    }
    uint32_t off = woff + incl - tsum;  // exclusive offset of slot 4t inside the CTA

    // ---- chained scan across CTAs ----
    if (warp == 0) {
        if (lane == 0) {
            volatile unsigned long long *st = a.lookback + bid;
            *st = (bid == 0 ? LB_PREFIX : LB_AGG) | (unsigned long long)total;
        }
        __syncwarp();
        const unsigned long long cb = lookback_exclusive(a.lookback, bid, (unsigned long long)total, lane);
        if (lane == 0) {
            s_base = cb;
            const uint32_t nv = s_nvis;
            const int32_t lt = s_last;
            if (nv) atomicAdd(&a.frame->visible, nv);
            if (lt >= 0) atomicMax(&a.frame->last_tile_plus1, lt + 1);
            if (bid == gridDim.x - 1) {
                const unsigned long long m = cb + total;
                a.frame->dup_total = m;
                a.frame->dup_sorted = m < (unsigned long long)a.capacity ? (uint32_t)m : a.capacity;
                a.frame->overflow = m > (unsigned long long)a.capacity ? 1u : 0u;
            }
        }
    }
    __syncthreads();
    const unsigned long long base = s_base;

    // ---- emit (same rules as projection_kernel) ----
    constexpr uint32_t EMIT_SMALL = 4;
#pragma unroll
    for (int j = 0; j < SH_GROUPS; ++j) {
        const uint32_t n = r[j].x, x0u = r[j].y & 0xFFFFu, y0u = r[j].y >> 16, wu = r[j].z & 0xFFFFu, depth = r[j].z >> 16;
        const uint32_t id = base_id + SH_GROUPS * tid + j;
        if (n != 0u && n <= EMIT_SMALL) {
            uint32_t x = x0u, y = y0u;
            const uint32_t x1 = x0u + wu;
#pragma unroll
            for (uint32_t e = 0; e < EMIT_SMALL; ++e) {
                if (e < n) {
                    const unsigned long long gpos = base + off + e;
                    if (gpos < (unsigned long long)a.capacity) {
                        a.keys[gpos] = ((y * gx + x) << 16) | depth;
                        a.values[gpos] = id;
                    }
                    if (++x == x1) { x = x0u; y += (uint32_t)a.row_mod; }
                }
            }
        }
        uint32_t big = __ballot_sync(0xffffffffu, n > EMIT_SMALL);
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1u;
            const uint32_t sn = __shfl_sync(0xffffffffu, n, src), soff = __shfl_sync(0xffffffffu, off, src);
            const uint32_t sx0 = __shfl_sync(0xffffffffu, x0u, src), sy0 = __shfl_sync(0xffffffffu, y0u, src);
            const uint32_t sw = __shfl_sync(0xffffffffu, wu, src), sdepth = __shfl_sync(0xffffffffu, depth, src);
            const uint32_t sid = __shfl_sync(0xffffffffu, id, src);
            for (uint32_t e = lane; e < sn; e += 32u) {
                const uint32_t ry = e / sw, rx = e - ry * sw;
                const unsigned long long gpos = base + soff + e;
                if (gpos < (unsigned long long)a.capacity) {
                    a.keys[gpos] = (((sy0 + ry * (uint32_t)a.row_mod) * gx + sx0 + rx) << 16) | sdepth;
                    a.values[gpos] = sid;
                }
            }
        }
        off += n;
    }
}

// ==============================================================================================================
// Group mode (gsr_group_attach): the projection sharded by SPLATS.  Rank r of G runs the full-frame maths of projection_kernel for ITS
// slice of the splats only (so the cull, the EWA, pow and the SH fetch happen once per splat in the whole group, not once per rank) and
// sends every output to the rank that owns it: tile row y belongs to rank y % G, so a splat's (key, value) pairs of row y and its
// 48-byte record go into rank (y % G)'s memory as plain stores through NVLink peer pointers -- the all-to-all of SURVEY 8e fused into the
// kernel that produces the data.  Per destination the pairs must arrive in splat-id order (the stable sort keeps that order among
// equal keys, and the reference's result depends on it): every destination has its own chained scan (G links per CTA, resolved together
// by the closer warp), and source r writes into ITS receive segment of the destination, [r * seg_cap, (r + 1) * seg_cap).  The
// destination later packs the G segments in source order = splat-id order.  When all CTAs are done the last one publishes
// seq | count and seq | last tile to every destination's flag page (data first, system fence, then the flags).
__device__ __forceinline__ unsigned long long lookback_exclusive_strided(volatile unsigned long long *status, uint32_t stride, uint32_t col, uint32_t bid,
                                                                         unsigned long long total, uint32_t lane) {
    if (bid == 0) return 0ull;
    unsigned long long excl = 0ull;
    int64_t start = (int64_t)bid - 1;
    while (true) {
        const int64_t t = start - (int64_t)lane;
        unsigned long long v = (t >= 0) ? status[(uint64_t)t * stride + col] : LB_PREFIX;
        while (__any_sync(0xffffffffu, (v >> 62) == 0ull)) {
            if ((v >> 62) == 0ull) v = status[(uint64_t)t * stride + col];
        }
        const uint32_t pmask = __ballot_sync(0xffffffffu, (v >> 62) == 2ull);
        const uint32_t first = pmask ? (uint32_t)(__ffs(pmask) - 1) : 32u;
        unsigned long long c = (lane <= first) ? (v & LB_VAL) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        excl += c;
        if (pmask) break;
        start -= 32;
    }
    if (lane == 0) status[(uint64_t)bid * stride + col] = LB_PREFIX | ((excl + total) & LB_VAL);
    return excl;
}

// rows of [y0, y1) that rank d of G owns: first such row and how many
__device__ __forceinline__ void rows_of(uint32_t y0, uint32_t y1, uint32_t d, uint32_t G, uint32_t &first, uint32_t &count) {
    first = y0 + ((d + G - y0 % G) % G);
    count = first < y1 ? (y1 - 1u - first) / G + 1u : 0u;
}

__global__ void __launch_bounds__(PROJ_THREADS, GSR_PROJ_MIN_BLOCKS) projection_scatter_kernel(const __grid_constant__ ProjectionArgs a,
                                                                                               const __grid_constant__ ScatterPeers sp) {
#ifndef GSR_CPU_EMU
    extern __shared__ __align__(128) unsigned char proj_smem[];
#else
    __shared__ __align__(128) unsigned char proj_smem[PROJ_SMEM_BYTES];
#endif
    __shared__ uint32_t s_bid, s_is_last;
    __shared__ __align__(8) uint64_t s_bar[PROJ_WARPS][2];
    __shared__ uint32_t s_wtotal[PROJ_WARPS][GROUP_MAX];   // pairs of each warp for each destination
    __shared__ uint32_t s_count, s_ready, s_nvis;
    __shared__ int32_t s_last;
    __shared__ unsigned long long s_cta_base[GROUP_MAX];

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t G = (uint32_t)sp.world;
    float4 *slab = reinterpret_cast<float4 *>(proj_smem + (size_t)warp * PROJ_SLAB_BYTES);  // [15][32]
    GroupFlags *mine = sp.flags[sp.rank];
    if (lane == 0) {
        mbar_init(&s_bar[warp][0], 1);
        mbar_init(&s_bar[warp][1], 1);
        fence_mbar_init();
    }
    if (tid == 0) {
        s_bid = atomicAdd(&a.frame->proj_ticket, 1u);
        s_count = 0u; s_ready = 0u; s_nvis = 0u; s_last = -1;
    }
    __syncthreads();
    const uint32_t bid = s_bid;                      // position of this CTA in the chained scans
    const uint32_t li0 = (bid * PROJ_WARPS + warp) * 32u;   // index inside the slice
    const uint32_t id0 = sp.first + li0, id = id0 + lane;
    const bool warp_in = li0 < sp.count;             // the slice may end inside the CTA (planes are padded to 256 splats: staging stays in bounds)

    if (warp_in && lane == 0) {
        mbar_expect_tx(&s_bar[warp][0], 3u * 512u);
#pragma unroll
        for (int k = 0; k < 3; ++k) bulk_g2s(slab + k * 32, a.soa + (uint64_t)k * a.plane_stride + id0, 512u, &s_bar[warp][0]);
    }
    const uint32_t gx = (uint32_t)((a.u.dims[0] + TILE - 1) / TILE);

    uint32_t n = 0, x0u = 0, y0u = 0, y1u = 0, wu = 0, depth = 0;
    int32_t last_tile = -1;
    float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0;
    float splat_opacity = 0.0f, vx = 0.0f, vy = 0.0f, vz = 0.0f;
    if (warp_in) {
        mbar_wait(&s_bar[warp][0], 0);
        if (li0 + lane < sp.count && id < a.num_splats) {
            LaneOut o;
            if (project_lane<false>(a, slab[lane], slab[32 + lane], slab[64 + lane], o) && o.n) {
                n = o.n; x0u = o.x0; y0u = o.y0; wu = o.w; depth = o.depth; y1u = o.y0 + o.n / o.w;
                r0 = o.r0; r1 = o.r1; splat_opacity = o.opacity; vx = o.vx; vy = o.vy; vz = o.vz;
            }
            last_tile = o.last_tile;
        }
    }

    // ---- per-destination pair counts of the warp; the CTA's last warp through here (the closer) publishes the G scan links ----
    for (uint32_t d = 0; d < G; ++d) {
        uint32_t f, c;
        rows_of(y0u, y1u, d, G, f, c);
        const uint32_t tot = __reduce_add_sync(0xffffffffu, n ? wu * c : 0u);
        if (lane == 0) s_wtotal[warp][d] = tot;
    }
    const uint32_t emit_mask = __ballot_sync(0xffffffffu, n != 0u);
    const uint32_t nvis = __popc(emit_mask);
    const int32_t wl = __reduce_max_sync(0xffffffffu, last_tile);
    bool closer = false;
    if (lane == 0) {
        if (nvis) atomicAdd(&s_nvis, nvis);
        if (wl >= 0) atomicMax(&s_last, wl);
        __threadfence_block();
        closer = atomicAdd(&s_count, 1u) == PROJ_WARPS - 1;
    }
    closer = __shfl_sync(0xffffffffu, (int)closer, 0) != 0;
    uint32_t cta_total = 0;   // closer: lane d holds the CTA's pair count for destination d
    if (closer) {
        __threadfence_block();
        if (lane < G) {
#pragma unroll
            for (int w = 0; w < PROJ_WARPS; ++w) cta_total += ((volatile uint32_t *)&s_wtotal[w][0])[lane];
            volatile unsigned long long *st = sp.lookback + (uint64_t)bid * G + lane;
            *st = (bid == 0 ? LB_PREFIX : LB_AGG) | (unsigned long long)cta_total;
        }
    }

    // ---- phase 2: SH planes -> colour -> record, stored into the record table of every rank that owns one of the splat's rows ----
    const bool bulk = warp_in && nvis >= (uint32_t)a.sh_bulk_min;
    if (bulk && lane == 0) {
        mbar_expect_tx(&s_bar[warp][1], 12u * 512u);
#pragma unroll
        for (int k = 3; k < NUM_PLANES; ++k) bulk_g2s(slab + k * 32, a.soa + (uint64_t)k * a.plane_stride + id0, 512u, &s_bar[warp][1]);
    }
    if (closer) {
        for (uint32_t d = 0; d < G; ++d) {
            const uint32_t tot_d = __shfl_sync(0xffffffffu, cta_total, (int)d);
            const unsigned long long base_d = lookback_exclusive_strided(sp.lookback, G, d, bid, (unsigned long long)tot_d, lane);
            if (lane == 0) {
                s_cta_base[d] = base_d;
                if (bid == gridDim.x - 1) mine->seg_total[d] = base_d + tot_d;   // tickets are dense: this CTA closes every scan
            }
        }
        if (lane == 0) {
            __threadfence_block();
            *(volatile uint32_t *)&s_ready = 1u;
            const uint32_t nv = *(volatile uint32_t *)&s_nvis;
            const int32_t lt = *(volatile int32_t *)&s_last;
            if (nv) atomicAdd(&a.frame->visible, nv);
            if (lt >= 0) atomicMax(&mine->scat_last, lt + 1);
        }
    }
    if (bulk) mbar_wait(&s_bar[warp][1], 0);
    if (n) {
        float col[3];
        if (bulk) sh_color<true>(slab + 3 * 32 + lane, 32, vx, vy, vz, col);
        else sh_color<false>(a.soa + 3ull * a.plane_stride + id, a.plane_stride, vx, vy, vz, col);
        const float4 r2 = make_float4(col[0], col[1], col[2], splat_opacity);
        for (uint32_t d = 0; d < G; ++d) {
            uint32_t f, c;
            rows_of(y0u, y1u, d, G, f, c);
            if (c) {
                float4 *rec = sp.records[d] + (uint64_t)id * 3u;
                rec[0] = r0; rec[1] = r1; rec[2] = r2;
            }
        }
    }

    if (lane == 0) {
        while (*(volatile uint32_t *)&s_ready == 0u) __nanosleep(100);
        __threadfence_block();
    }
    __syncwarp();

    // ---- emit (:219-226), once per destination: slot base + off + j of destination d's segment holds tile j (row-major over the rows
    //      d owns) of the splat's rect.  Same hybrid as projection_kernel: small rects by their own lane, big ones by the whole warp.
    constexpr uint32_t EMIT_SMALL = 4;
    for (uint32_t d = 0; d < G; ++d) {
        uint32_t fy, cnt;
        rows_of(y0u, y1u, d, G, fy, cnt);
        const uint32_t nd = n ? wu * cnt : 0u;
        if (!__any_sync(0xffffffffu, nd != 0u)) continue;
        const uint32_t incl = warp_incl_scan_u32(nd, lane);
        unsigned long long base = 0;
        if (lane == 0) {
            base = *(volatile unsigned long long *)&s_cta_base[d];
            for (uint32_t w = 0; w < warp; ++w) base += ((volatile uint32_t *)&s_wtotal[w][0])[d];
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        uint32_t *kd = sp.keys[d], *vd = sp.values[d];
        const uint32_t my_off = incl - nd;
        if (nd != 0u && nd <= EMIT_SMALL) {
            uint32_t x = x0u, y = fy;
            const uint32_t x1 = x0u + wu;
#pragma unroll
            for (uint32_t j = 0; j < EMIT_SMALL; ++j) {
                if (j < nd) {
                    const unsigned long long g = base + my_off + j;
                    if (g < (unsigned long long)sp.seg_cap) {
                        kd[g] = ((y * gx + x) << 16) | depth;
                        vd[g] = id;
                    }
                    if (++x == x1) { x = x0u; y += G; }
                }
            }
        }
        uint32_t big = __ballot_sync(0xffffffffu, nd > EMIT_SMALL);
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1u;
            const uint32_t sn = __shfl_sync(0xffffffffu, nd, src), soff = __shfl_sync(0xffffffffu, my_off, src);
            const uint32_t sx0 = __shfl_sync(0xffffffffu, x0u, src), sy0 = __shfl_sync(0xffffffffu, fy, src);
            const uint32_t sw = __shfl_sync(0xffffffffu, wu, src), sdepth = __shfl_sync(0xffffffffu, depth, src);
            for (uint32_t j = lane; j < sn; j += 32u) {
                const uint32_t ry = j / sw, rx = j - ry * sw;
                const unsigned long long g = base + soff + j;
                if (g < (unsigned long long)sp.seg_cap) {
                    kd[g] = (((sy0 + ry * G) * gx + sx0 + rx) << 16) | sdepth;
                    vd[g] = id0 + (uint32_t)src;
                }
            }
        }
    }

    // ---- completion: when every CTA's pairs and records are on their way, tell every destination how many pairs it got from this
    //      source and the largest tile this source touched (the frame-global Q10 bookkeeping travels with the data) ----
    // The CTA barrier orders every thread's stores before thread 0's fence (cumulativity), and the ticket is a device-scope
    // synchronisation between this CTA and the one that finishes last; only that last CTA talks to other GPUs, behind ONE
    // system-scope fence.  (A system-scope fence in every CTA was measured to stretch the kernel by up to the duration of a frame
    // read-back in flight: profiles/r02_group_e2e_probe.txt.)
    __syncthreads();
#ifdef GSR_SCATTER_FENCE_PER_CTA_SYS
    if (tid == 0) __threadfence_system();
#else
    if (tid == 0) __threadfence();
#endif
    if (tid == 0) s_is_last = atomicAdd(&mine->scat_ticket, 1u) == gridDim.x - 1u ? 1u : 0u;
    __syncthreads();
    if (s_is_last && tid < 32u) {
        __threadfence_system();
        const int32_t lp1 = __shfl_sync(0xffffffffu, lane == 0 ? *(volatile int32_t *)&mine->scat_last : 0, 0);   // read once, before lane 0 resets it
        if (lane < G) {
            const unsigned long long cnt = *(volatile unsigned long long *)&mine->seg_total[lane];
            volatile unsigned long long *m = &sp.flags[lane]->seg_meta[sp.parity][sp.rank][0];
            m[1] = ((unsigned long long)sp.seq << 32) | (unsigned long long)(uint32_t)(lp1 > 0 ? lp1 : 0);
            m[0] = ((unsigned long long)sp.seq << 32) | (cnt < 0xFFFFFFFFull ? cnt : 0xFFFFFFFFull);
        }
        __syncwarp();
        if (lane == 0) { mine->scat_last = 0; mine->scat_ticket = 0u; __threadfence(); }   // ready for the next frame (stream order)
    }
}

// ==============================================================================================================
// Multiview frame (gsr_set_views): projection_kernel for K cameras at once.  Per warp, planes 0-2 arrive once (TMA) and the SH planes
// at most once (bulk when enough lanes emit in ANY view, else per-lane gathers); per view the lane runs project_lane with that
// view's constants, writes record words 0-1 into the view's table and parks its rect (n, x0|y0<<16, w|depth<<16) in shared memory
// (registers stay at the single-view kernel's level whatever K is).  One chained scan runs over the per-splat SUM of the K counts;
// a splat's pairs are emitted view-major, view v with tile ids v*T + tile -- so after the stable sort, view v's pairs are exactly
// the single-view frame's pairs in the same order.
constexpr size_t VIEW_STATE_BYTES = sizeof(uint32_t) * 3 * PROJ_THREADS;   // per view: n | x0,y0 | w,depth of every lane of the CTA

__global__ void __launch_bounds__(PROJ_THREADS, GSR_PROJ_MIN_BLOCKS) projection_views_kernel(const __grid_constant__ ViewsArgs A) {
#ifndef GSR_CPU_EMU
    extern __shared__ __align__(128) unsigned char proj_smem[];
#else
    __shared__ __align__(128) unsigned char proj_smem[PROJ_SMEM_BYTES + GSR_MAX_VIEWS * VIEW_STATE_BYTES];
#endif
    __shared__ uint32_t s_bid;
    __shared__ __align__(8) uint64_t s_bar[PROJ_WARPS][2];
    __shared__ uint32_t s_wtotal[PROJ_WARPS];
    __shared__ uint32_t s_count, s_ready, s_nvis;
    __shared__ int32_t s_last;
    __shared__ unsigned long long s_cta_base;

    const ProjectionArgs &a = A.view[0];   // the view-independent fields
    const int K = A.num_views;
    const uint32_t T = A.tiles_per_view;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    float4 *slab = reinterpret_cast<float4 *>(proj_smem + (size_t)warp * PROJ_SLAB_BYTES);  // [15][32]
    uint32_t *vstate = reinterpret_cast<uint32_t *>(proj_smem + PROJ_SMEM_BYTES);           // [view][3][PROJ_THREADS]
    if (lane == 0) {
        mbar_init(&s_bar[warp][0], 1);
        mbar_init(&s_bar[warp][1], 1);
        fence_mbar_init();
    }
    if (tid == 0) {
        s_bid = atomicAdd(&a.frame->proj_ticket, 1u);
        s_count = 0u; s_ready = 0u; s_nvis = 0u; s_last = -1;
    }
    __syncthreads();
    const uint32_t bid = s_bid;
    const uint32_t id0 = (bid * PROJ_WARPS + warp) * 32u;
    const uint32_t id = id0 + lane;

    if (lane == 0) {
        mbar_expect_tx(&s_bar[warp][0], 3u * 512u);
#pragma unroll
        for (int k = 0; k < 3; ++k) bulk_g2s(slab + k * 32, a.soa + (uint64_t)k * a.plane_stride + id0, 512u, &s_bar[warp][0]);
    }
    const uint32_t gx = (uint32_t)((a.u.dims[0] + TILE - 1) / TILE);
    mbar_wait(&s_bar[warp][0], 0);

    // ---- phase 1, per view: cull + EWA + rect; record words 0-1; the rect to shared memory ----
    uint32_t ntot = 0, any_mask = 0, nvis = 0;
    int32_t last_tile = -1;   // in the concatenated tile-id space
#pragma unroll 1
    for (int v = 0; v < K; ++v) {
        const ProjectionArgs &av = A.view[v];
        uint32_t n = 0, xy = 0, wd = 0;
        if (id < a.num_splats) {
            LaneOut o;
            if (project_lane<false>(av, slab[lane], slab[32 + lane], slab[64 + lane], o) && o.n) {
                n = o.n; xy = o.x0 | (o.y0 << 16); wd = o.w | (o.depth << 16);
                float4 *rec = av.records + (uint64_t)id * 3u;
                rec[0] = o.r0; rec[1] = o.r1;
            }
            if (o.last_tile >= 0) last_tile = (int32_t)((uint32_t)v * T) + o.last_tile;
        }
        uint32_t *st = vstate + (size_t)v * 3u * PROJ_THREADS;
        st[tid] = n; st[PROJ_THREADS + tid] = xy; st[2 * PROJ_THREADS + tid] = wd;
        ntot += n;
        const uint32_t m = __ballot_sync(0xffffffffu, n != 0u);
        any_mask |= m;
        nvis += (uint32_t)__popc(m);
    }

    // ---- scan of the per-splat totals; the closer publishes the CTA aggregate (as projection_kernel) ----
    const uint32_t incl = warp_incl_scan_u32(ntot, lane);
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    const int32_t wl = __reduce_max_sync(0xffffffffu, last_tile);
    bool closer = false;
    uint32_t cta_total = 0;
    if (lane == 0) {
        s_wtotal[warp] = total;
        if (nvis) atomicAdd(&s_nvis, nvis);
        if (wl >= 0) atomicMax(&s_last, wl);
        __threadfence_block();
        closer = atomicAdd(&s_count, 1u) == PROJ_WARPS - 1;
        if (closer) {
            __threadfence_block();
#pragma unroll
            for (int w = 0; w < PROJ_WARPS; ++w) cta_total += ((volatile uint32_t *)s_wtotal)[w];
            volatile unsigned long long *stl = a.lookback + bid;
            *stl = (bid == 0 ? LB_PREFIX : LB_AGG) | (unsigned long long)cta_total;
        }
    }
    closer = __shfl_sync(0xffffffffu, (int)closer, 0) != 0;
    cta_total = __shfl_sync(0xffffffffu, cta_total, 0);

    // ---- phase 2: the SH planes once for all views (bulk when enough lanes emit in any view), then colour + record word 2 per view ----
    const bool bulk = (uint32_t)__popc(any_mask) >= (uint32_t)a.sh_bulk_min;
    if (bulk && lane == 0) {
        mbar_expect_tx(&s_bar[warp][1], 12u * 512u);
#pragma unroll
        for (int k = 3; k < NUM_PLANES; ++k) bulk_g2s(slab + k * 32, a.soa + (uint64_t)k * a.plane_stride + id0, 512u, &s_bar[warp][1]);
    }
    if (closer) {
        const unsigned long long cta_base = lookback_exclusive(a.lookback, bid, (unsigned long long)cta_total, lane);
        if (lane == 0) {
            s_cta_base = cta_base;
            __threadfence_block();
            *(volatile uint32_t *)&s_ready = 1u;
            const uint32_t nv = *(volatile uint32_t *)&s_nvis;
            const int32_t lt = *(volatile int32_t *)&s_last;
            if (nv) atomicAdd(&a.frame->visible, nv);
            if (lt >= 0) atomicMax(&a.frame->last_tile_plus1, lt + 1);
            if (bid == gridDim.x - 1) {
                const unsigned long long m = cta_base + cta_total;
                a.frame->dup_total = m;
                a.frame->dup_sorted = m < (unsigned long long)a.capacity ? (uint32_t)m : a.capacity;
                a.frame->overflow = m > (unsigned long long)a.capacity ? 1u : 0u;
            }
        }
    }
    if (bulk) mbar_wait(&s_bar[warp][1], 0);
    if (any_mask & (1u << lane)) {
        // the view-independent part of the record (opacity) and the view direction, with the operations of project_lane
        const float4 pt = slab[lane], cb = slab[64 + lane];
        const float ms = a.u.model_scale;
        const float sp0 = pt.x * ms, sp1 = pt.y * ms, sp2 = pt.z * ms;
        const float splat_time = a.u.time - pt.w;
        const float tfl = ease_out_cubic(g_clamp(splat_time - 0.35f, 0.0f, 1.0f));
        const float splat_opacity = cb.z * tfl * tfl;
#pragma unroll 1
        for (int v = 0; v < K; ++v) {
            if (vstate[(size_t)v * 3u * PROJ_THREADS + tid] == 0u) continue;
            const ProjectionArgs &av = A.view[v];
            const float d0 = sp0 - av.u.camera_pos[0], d1 = sp1 - av.u.camera_pos[1], d2 = sp2 - av.u.camera_pos[2];
            const float inv_len = 1.0f / sqrtf((d0 * d0 + d1 * d1) + d2 * d2);
            float col[3];
            if (bulk) sh_color<true>(slab + 3 * 32 + lane, 32, d0 * inv_len, d1 * inv_len, d2 * inv_len, col);
            else sh_color<false>(a.soa + 3ull * a.plane_stride + id, a.plane_stride, d0 * inv_len, d1 * inv_len, d2 * inv_len, col);
            av.records[(uint64_t)id * 3u + 2u] = make_float4(col[0], col[1], col[2], splat_opacity);
        }
    }

    unsigned long long base = 0;
    if (lane == 0) {
        while (*(volatile uint32_t *)&s_ready == 0u) __nanosleep(100);
        __threadfence_block();
        base = *(volatile unsigned long long *)&s_cta_base;
        for (uint32_t w = 0; w < warp; ++w) base += ((volatile uint32_t *)s_wtotal)[w];
    }
    base = __shfl_sync(0xffffffffu, base, 0);

    // ---- emit, view-major per splat (same small / big rect rules as projection_kernel) ----
    constexpr uint32_t EMIT_SMALL = 4;
    uint32_t off = incl - ntot;
#pragma unroll 1
    for (int v = 0; v < K; ++v) {
        const uint32_t *st = vstate + (size_t)v * 3u * PROJ_THREADS;
        const uint32_t n = st[tid], x0u = st[PROJ_THREADS + tid] & 0xFFFFu, y0u = st[PROJ_THREADS + tid] >> 16;
        const uint32_t wu = st[2 * PROJ_THREADS + tid] & 0xFFFFu, depth = st[2 * PROJ_THREADS + tid] >> 16;
        const uint32_t tbase = (uint32_t)v * T;
        if (n != 0u && n <= EMIT_SMALL) {
            uint32_t x = x0u, y = y0u;
            const uint32_t x1 = x0u + wu;
#pragma unroll
            for (uint32_t j = 0; j < EMIT_SMALL; ++j) {
                if (j < n) {
                    const unsigned long long g = base + off + j;
                    if (g < (unsigned long long)a.capacity) {
                        a.keys[g] = ((tbase + y * gx + x) << 16) | depth;
                        a.values[g] = id;
                    }
                    if (++x == x1) { x = x0u; ++y; }
                }
            }
        }
        uint32_t big = __ballot_sync(0xffffffffu, n > EMIT_SMALL);
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1u;
            const uint32_t sn = __shfl_sync(0xffffffffu, n, src), soff = __shfl_sync(0xffffffffu, off, src);
            const uint32_t sx0 = __shfl_sync(0xffffffffu, x0u, src), sy0 = __shfl_sync(0xffffffffu, y0u, src);
            const uint32_t sw = __shfl_sync(0xffffffffu, wu, src), sdepth = __shfl_sync(0xffffffffu, depth, src);
            for (uint32_t j = lane; j < sn; j += 32u) {
                const uint32_t ry = j / sw, rx = j - ry * sw;
                const unsigned long long g = base + soff + j;
                if (g < (unsigned long long)a.capacity) {
                    a.keys[g] = ((tbase + (sy0 + ry) * gx + sx0 + rx) << 16) | sdepth;
                    a.values[g] = id0 + (uint32_t)src;
                }
            }
        }
        off += n;
    }
}

}  // namespace

uint32_t projection_num_blocks(uint32_t num_splats) { return (num_splats + PROJ_THREADS - 1) / PROJ_THREADS; }

#ifndef GSR_CPU_EMU  // host side: CUDA only
// Force-load this file's kernels (CUDA loads modules lazily; a first launch that has to load code while another context's
// kernel spins on a flag this launch would satisfy can stall the host: see gsr_group_attach).
int preload_projection_kernels() {
    cudaFuncAttributes fa;
    // dynamic shared memory opt-in is a per-device function attribute: set here, once per context creation, on the context's device
    GSR_CUDA_TRY(cudaFuncSetAttribute(projection_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PROJ_SMEM_BYTES));
    GSR_CUDA_TRY(cudaFuncSetAttribute(projection_sharded_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SH_SLAB_BYTES));
    GSR_CUDA_TRY(cudaFuncSetAttribute(projection_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PROJ_SMEM_BYTES));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, projection_kernel));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, projection_sharded_kernel));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, projection_scatter_kernel));
    GSR_CUDA_TRY(cudaFuncSetAttribute(projection_views_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(PROJ_SMEM_BYTES + GSR_MAX_VIEWS * VIEW_STATE_BYTES)));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, projection_views_kernel));
    return GSR_OK;
}

int launch_projection_views(const ViewsArgs &a, cudaStream_t stream) {
    const uint32_t blocks = projection_num_blocks(a.view[0].num_splats);
    if (blocks == 0) return GSR_OK;
    projection_views_kernel<<<blocks, PROJ_THREADS, PROJ_SMEM_BYTES + (size_t)a.num_views * VIEW_STATE_BYTES, stream>>>(a);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}
uint32_t projection_scatter_blocks(uint32_t count) { return count ? (count + PROJ_THREADS - 1) / PROJ_THREADS : 1u; }   // an empty slice still publishes its flags

int launch_projection_scatter(const ProjectionArgs &frame_args, const ScatterPeers &sp, cudaStream_t stream) {
    ProjectionArgs a = frame_args;   // the whole frame: no band, no row ownership, no reject (ownership is decided per pair, by destination)
    a.band_y0 = 0; a.band_y1 = (a.u.dims[1] + TILE - 1) / TILE;
    a.row_mod = 1; a.row_rem = 0; a.fast_reject = 0; a.fast_mode = 0; a.sh_bulk_min = 12;
    projection_scatter_kernel<<<projection_scatter_blocks(sp.count), PROJ_THREADS, PROJ_SMEM_BYTES, stream>>>(a, sp);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}

int launch_projection(const ProjectionArgs &a, cudaStream_t stream) {
    const uint32_t blocks = projection_num_blocks(a.num_splats);
    if (blocks == 0) return GSR_OK;
    if (a.fast_reject) {  // sharded variant: 1024 splats per CTA
        const uint32_t sblocks = (a.num_splats + SH_SPLATS - 1) / SH_SPLATS;
        projection_sharded_kernel<<<sblocks, PROJ_THREADS, SH_SLAB_BYTES, stream>>>(a);
        GSR_CUDA_TRY(cudaGetLastError());
        return GSR_OK;
    }
    projection_kernel<<<blocks, PROJ_THREADS, PROJ_SMEM_BYTES, stream>>>(a);
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}
#endif  // GSR_CPU_EMU

}  // namespace gsr
