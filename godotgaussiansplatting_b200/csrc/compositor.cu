// compositor.cu -- stage 4: per-tile front-to-back alpha blend.  Replaces gsplat_render.glsl:50-111.
//
// One CTA per 16x16 tile like the reference's workgroup, 256-splat chunks staged in shared memory, the same per-pixel
// arithmetic and the same tile-stop vote.  What is Blackwell-specific is how the blend is issued and scheduled:
//   * the kernel is FMA-pipe bound (113 FMA-pipe instructions per 4 splats and pixel pair; measured on B200, ubench/f32x2_latency.cu:
//     FFMA2 and scalar FFMA both retire 128 lane-FMAs/clk/SM, FFMA2 at half the issue slots, dependent-issue latency 4 cycles), so
//     every thread owns TWO horizontally adjacent pixels and the blend runs on packed fp32x2 instructions
//     (PTX add/sub/mul/fma.rn.f32x2 -> SASS FADD2/FMUL2/FFMA2).  Each lane of a packed op is an ordinary IEEE binary32 operation,
//     so results stay bit-identical to the oracle;
//   * per-splat control flow is gone: dead pixels (t <= 1/255, gsplat_render.glsl:79) keep their state by select, the warp-level
//     "all dead" test runs once per 4 splats on the transmittance of half a group earlier (off the loop-carried path), and the
//     last chunk is padded with null splats (opacity 0);
//   * the transmittance chain is two instructions per splat: alpha and 1 - alpha are formed off the critical path, the update is
//     FMUL2 + select (`t = alive ? t * (1 - alpha) : t`, bit-identical to multiplying by 1 - 0);
//   * the conic is pre-scaled at staging time (-0.5*cx, -0.5*cz, -cy: exact power-of-two/sign changes) so the `-0.5 * (...)`
//     multiply of :84 disappears from the inner loop without changing any rounding;
//   * the gather `culled_buffer[sort_buffer[...]]` (:72) for chunk i+1 is issued into registers before the blend loop of chunk i
//     (software prefetch), and the (a, b) words of splat group g+1 are read from shared memory while group g is blended;
//   * the tile-stop vote `atomicAdd(shared_t, uint(t*255))` (:97) is a warp reduction + 4 shared words;
//   * scheduling (measured, profiles/r02_compositor_*): a tile is a sequential chain of up to ~19 chunks, a frame has ~1250 such
//     chains of very different length, and the SM's warp scheduler favours its oldest warps -- so the persistent grid takes tiles
//     LONGEST-FIRST (tile_order_kernel: the previous frame's consumed chunk count of the tile, else its list length), keeps few
//     CTAs per SM and never migrates a tile (the round-1 re-queue mechanism cost a spill + restore per hand-back and made long
//     chains young again; measured slower than this order).
// Arithmetic contract: "gsr deterministic math" (common.cuh): the GLSL-legal contractions of :84 and :89 are explicit fma
// (CONTRACT = true, the default); CONTRACT = false (GSR_FLAG_UNCONTRACTED_BLEND) evaluates :84-90 with no contraction at all,
// which is bit-identical to the reference's own shader text executed by oracle/glsl_cpu.  exp() is the det_exp() polynomial,
// evaluated here two lanes at a time.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace gsr {

namespace {

constexpr int CHUNK = 256;    // gsplat_render.glsl:9 WORKGROUP_SIZE: splats per staged chunk / pixels per tile
constexpr int THREADS = 128;  // 2 pixels per thread
constexpr float MIN_ALPHA = 1.0f / 255.0f;

typedef unsigned long long u64;

#ifndef GSR_CPU_EMU
__device__ __forceinline__ u64 pk(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// a*b + c with TWO roundings per lane, for the uncontracted evaluation.  ptxas (12.9, sm_100a) contracts a mul.rn.f32x2 whose only use
// is an add.rn.f32x2 into one FFMA2 -- in spite of the .rn qualifiers and of -fmad=false (cuobjdump: 44 FFMA2 where the PTX has 24
// fma.rn.f32x2; tests/test_gpu_pipeline.py::test_uncontracted_blend_flag_... caught it on silicon).  It honours the scalar .rn pair.
__device__ __forceinline__ u64 mul_add2_unfused(u64 a, u64 b, u64 c) {
    float al, ah, bl, bh, cl, ch;
    asm volatile("mov.b64 {%0, %1}, %2;" : "=f"(al), "=f"(ah) : "l"(a));
    upk(b, bl, bh); upk(c, cl, ch);
    return pk(__fadd_rn(__fmul_rn(al, bl), cl), __fadd_rn(__fmul_rn(ah, bh), ch));
}
#else  // tests/kernel_emu: the kernels of this file compiled for the CPU (test infrastructure; libgsr never defines GSR_CPU_EMU).
       // A packed op is two independent IEEE binary32 operations -- exactly what the PTX f32x2 instructions are.
inline u64 pk(float lo, float hi) { uint32_t a, b; memcpy(&a, &lo, 4); memcpy(&b, &hi, 4); return (u64)a | ((u64)b << 32); }
inline void upk(u64 v, float &lo, float &hi) { const uint32_t a = (uint32_t)v, b = (uint32_t)(v >> 32); memcpy(&lo, &a, 4); memcpy(&hi, &b, 4); }
inline u64 fma2(u64 a, u64 b, u64 c) { float al, ah, bl, bh, cl, ch; upk(a, al, ah); upk(b, bl, bh); upk(c, cl, ch); return pk(fmaf(al, bl, cl), fmaf(ah, bh, ch)); }
inline u64 mul2(u64 a, u64 b) { float al, ah, bl, bh; upk(a, al, ah); upk(b, bl, bh); return pk(al * bl, ah * bh); }
inline u64 add2(u64 a, u64 b) { float al, ah, bl, bh; upk(a, al, ah); upk(b, bl, bh); return pk(al + bl, ah + bh); }
inline u64 sub2(u64 a, u64 b) { float al, ah, bl, bh; upk(a, al, ah); upk(b, bl, bh); return pk(al - bl, ah - bh); }
inline u64 mul_add2_unfused(u64 a, u64 b, u64 c) { return add2(mul2(a, b), c); }
#endif
__device__ __forceinline__ u64 bc(float x) { return pk(x, x); }

struct Staged {  // one gathered record, pre-scaled for the inner loop
    float4 a;    // image_pos.x, image_pos.y, -0.5*conic.x, -0.5*conic.z
    float4 b;    // -conic.y, opacity, color.r, color.g
    float c;     // color.b
};

__device__ __forceinline__ Staged null_splat() {
    Staged s;
    s.a = make_float4(0.f, 0.f, 0.f, 0.f);
    s.b = make_float4(0.f, 0.f, 0.f, 0.f);
    s.c = 0.f;
    return s;
}

__device__ __forceinline__ Staged gather(const float4 *__restrict__ records, const uint32_t *__restrict__ values, uint32_t idx) {
    const uint32_t v = __ldg(values + idx);
    const float4 *r = records + (uint64_t)v * 3u;
    const float4 r0 = __ldg(r + 0), r1 = __ldg(r + 1), r2 = __ldg(r + 2);
    Staged s;
    s.a = make_float4(r0.x, r0.y, -0.5f * r1.x, -0.5f * r1.z);
    s.b = make_float4(-r1.y, r2.w, r2.x, r2.y);
    s.c = r2.z;
    return s;
}

#ifndef GSR_COMP_GROUP
#define GSR_COMP_GROUP 4  // splats per software-pipelined group of the blend loop
#endif
constexpr int GU = GSR_COMP_GROUP;
static_assert(CHUNK % GU == 0, "a chunk is a whole number of groups");

#ifndef GSR_CPU_EMU
__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ uint32_t smid() { uint32_t r; asm volatile("mov.u32 %0, %smid;" : "=r"(r)); return r; }
#else
inline unsigned long long globaltimer_ns() { return 0ull; }
inline uint32_t smid() { return 0u; }
#endif

struct BlendK {  // broadcast constants of det_exp() for the packed lanes
    u64 L2E2, MAGIC2, ONE2, C6, C5, C4, C3, C2, C1;
};
__device__ __forceinline__ BlendK make_blend_k() {
    BlendK k;
    k.L2E2 = bc(0x1.715476p+0f); k.MAGIC2 = bc(12582912.0f); k.ONE2 = bc(1.0f);
    k.C6 = bc(0x1.446c7ep-13f); k.C5 = bc(0x1.5f48c8p-10f); k.C4 = bc(0x1.3b29d8p-7f); k.C3 = bc(0x1.c6aeccp-5f);
    k.C2 = bc(0x1.ebfbe0p-3f); k.C1 = bc(0x1.62e430p-1f);
    return k;
}

// ---- phase A: alpha = opacity * exp(power) and 1 - alpha of GU splats (their (a, b) words already in registers) for this thread's
//      two pixels, written stage by stage so that the GU dependency chains can be interleaved.  No dependence on the transmittance:
//      this part of gsplat_render.glsl:84-88 runs ahead of the sequential blend.
template <bool CONTRACT>
__device__ __forceinline__ void phase_a(const float4 A[GU], const float4 B[GU], u64 npx2, float fpy, const BlendK &K, u64 al2[GU], u64 om2[GU]) {
    float oy[GU];
    u64 ox2[GU], pw2[GU], tm2[GU], e2[GU];
#pragma unroll
    for (int u = 0; u < GU; ++u) { ox2[u] = add2(bc(A[u].x), npx2); oy[u] = A[u].y - fpy; }
    // power = -0.5*(cx*ox*ox + cz*oy*oy) - cy*ox*oy (:84) on the pre-scaled conic:
    //   CONTRACT:  fma(e, oy, fma((-0.5cz)*oy, oy, ((-0.5cx)*ox)*ox))  with e = (-cy)*ox      (q and power contractions of the gsr spec)
    //   otherwise: (((-0.5cx)*ox)*ox + ((-0.5cz)*oy)*oy) + ((-cy)*ox)*oy                       (one rounding per GLSL operator)
#pragma unroll
    for (int u = 0; u < GU; ++u) pw2[u] = mul2(bc(A[u].z), ox2[u]);
#pragma unroll
    for (int u = 0; u < GU; ++u) {
        const float czoy = A[u].w * oy[u];
        if (CONTRACT) pw2[u] = fma2(bc(czoy), bc(oy[u]), mul2(pw2[u], ox2[u]));
        else pw2[u] = mul_add2_unfused(pw2[u], ox2[u], bc(__fmul_rn(czoy, oy[u])));   // (the second product must not fuse with the sum either)
    }
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = mul2(bc(B[u].x), ox2[u]);
#pragma unroll
    for (int u = 0; u < GU; ++u) pw2[u] = CONTRACT ? fma2(e2[u], bc(oy[u]), pw2[u]) : mul_add2_unfused(e2[u], bc(oy[u]), pw2[u]);
    // exp(power): det_exp(), two lanes at a time
#pragma unroll
    for (int u = 0; u < GU; ++u) pw2[u] = mul2(pw2[u], K.L2E2);
#pragma unroll
    for (int u = 0; u < GU; ++u) {
        float tl, th;
        upk(pw2[u], tl, th);
        tl = g_min(g_max(tl, -127.0f), 128.0f);
        th = g_min(g_max(th, -127.0f), 128.0f);
        pw2[u] = pk(tl, th);
    }
#pragma unroll
    for (int u = 0; u < GU; ++u) tm2[u] = add2(pw2[u], K.MAGIC2);
#pragma unroll
    for (int u = 0; u < GU; ++u) al2[u] = sub2(tm2[u], K.MAGIC2);
#pragma unroll
    for (int u = 0; u < GU; ++u) pw2[u] = sub2(pw2[u], al2[u]);  // f
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = fma2(K.C6, pw2[u], K.C5);
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = fma2(e2[u], pw2[u], K.C4);
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = fma2(e2[u], pw2[u], K.C3);
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = fma2(e2[u], pw2[u], K.C2);
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = fma2(e2[u], pw2[u], K.C1);
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = fma2(e2[u], pw2[u], K.ONE2);
#pragma unroll
    for (int u = 0; u < GU; ++u) {
        float ml, mh;
        upk(tm2[u], ml, mh);
        tm2[u] = pk(__uint_as_float((__float_as_uint(ml) << 23) + 0x3F800000u), __uint_as_float((__float_as_uint(mh) << 23) + 0x3F800000u));
    }
#pragma unroll
    for (int u = 0; u < GU; ++u) e2[u] = mul2(e2[u], tm2[u]);
#pragma unroll
    for (int u = 0; u < GU; ++u) al2[u] = mul2(bc(B[u].y), e2[u]);
#pragma unroll
    for (int u = 0; u < GU; ++u) om2[u] = sub2(K.ONE2, al2[u]);
}

// ---- phase B: the sequential part (gsplat_render.glsl:89-90).  A dead pixel has left the reference's loop: its colour and
//      transmittance are kept by select.  `alive_mid` = "a pixel of this thread was alive after the first half of the group".
template <bool CONTRACT>
__device__ __forceinline__ void phase_b(const float4 B[GU], const float *s_c, int j, const u64 al2[GU], const u64 om2[GU], u64 &cr2, u64 &cg2, u64 &cb2,
                                        float &t0, float &t1, bool &alive_mid) {
#pragma unroll
    for (int u = 0; u < GU; ++u) {
        const float cbl = s_c[j + u];
        if (u == GU / 2) alive_mid = (t0 > MIN_ALPHA) || (t1 > MIN_ALPHA);
        const bool a0 = t0 > MIN_ALPHA, a1 = t1 > MIN_ALPHA;
        float al, ah, pl, ph;
        upk(al2[u], al, ah);
        const u64 t2 = pk(t0, t1);
        upk(mul2(t2, om2[u]), pl, ph);
        const u64 m2 = pk(a0 ? al : 0.0f, a1 ? ah : 0.0f);   // alpha = 0: an exact no-op on the colour
        if (CONTRACT) {
            cr2 = fma2(mul2(bc(B[u].z), m2), t2, cr2);
            cg2 = fma2(mul2(bc(B[u].w), m2), t2, cg2);
            cb2 = fma2(mul2(bc(cbl), m2), t2, cb2);
        } else {
            cr2 = mul_add2_unfused(mul2(bc(B[u].z), m2), t2, cr2);
            cg2 = mul_add2_unfused(mul2(bc(B[u].w), m2), t2, cg2);
            cb2 = mul_add2_unfused(mul2(bc(cbl), m2), t2, cb2);
        }
        t0 = a0 ? pl : t0;
        t1 = a1 ? ph : t1;
    }
}

#ifndef GSR_COMP_MIN_BLOCKS
#define GSR_COMP_MIN_BLOCKS 3  // resident CTAs per SM the register allocation targets (profiles/r02_compositor_sweep.txt: 2-3 is best)
#endif

// Persistent CTAs.  Ticket k of the launch renders owned tile order[k] (longest chains first) or k itself; every tile is blended
// from its first chunk to its stop by the CTA that took it.  MULTI: a multiview frame (CompositeArgs::tiles_per_view), whose tile id
// selects the view's record table and frame layer; the blend itself is the same code.
template <bool CONTRACT, bool MULTI = false>
__global__ void __launch_bounds__(THREADS, GSR_COMP_MIN_BLOCKS) composite_kernel(const __grid_constant__ CompositeArgs p) {
    __shared__ float4 s_a[CHUNK];
    __shared__ float4 s_b[CHUNK];
    __shared__ float s_c[CHUNK];
    __shared__ uint32_t s_vote[THREADS / 32];
    __shared__ uint32_t s_tile;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    {   // sparse frame: only the first `comp_cta_limit` CTAs (one per SM: the block scheduler deals a fresh grid breadth-first) work
        const uint32_t limit = p.frame->comp_cta_limit;
        if (limit && blockIdx.x >= limit) return;
    }
    const BlendK K = make_blend_k();
    uint32_t staged = 0;  // SURVEY 8 symbol C, summed over the tiles this CTA processed (uniform across the CTA)
    unsigned long long t_start = 0;  // trace only

    for (;;) {
        if (tid == 0) {
            const uint32_t ticket = atomicAdd(&p.frame->comp_head, 1u);
            s_tile = ticket < (uint32_t)p.num_tiles ? (p.order ? p.order[ticket] : ticket) : 0xFFFFFFFFu;
            if (p.trace) t_start = globaltimer_ns();
        }
        __syncthreads();
        const uint32_t local_tile = s_tile;   // index among the owned tiles
        if (local_tile == 0xFFFFFFFFu) break;
        // owned tiles: rows tile_begin/tiles_x + k*row_step, all columns (row_step == 1: one contiguous band)
        const uint32_t tile_id = (uint32_t)p.tile_begin + (local_tile / (uint32_t)p.tiles_x) * (uint32_t)(p.row_step * p.tiles_x) + local_tile % (uint32_t)p.tiles_x;
        const float4 *records = p.records;
        float4 *out = p.out;
        uint32_t view_tile = tile_id;
        if (MULTI) {
            const uint32_t view = tile_id / (uint32_t)p.tiles_per_view;
            view_tile = tile_id - view * (uint32_t)p.tiles_per_view;
            records += (uint64_t)view * p.record_stride;
            out += (uint64_t)view * p.layer_stride;
        }

        const uint32_t tx = view_tile % (uint32_t)p.tiles_x, ty = view_tile / (uint32_t)p.tiles_x;
        const int px0 = (int)(tx * TILE + 2u * (tid & 7u)), py = (int)(ty * TILE + (tid >> 3));
        const u64 npx2 = pk(-(float)px0, -(float)(px0 + 1));  // ox = image_pos.x - pixel.x  ==  image_pos.x + (-pixel.x)
        const float fpy = (float)py;

        const uint2 bounds = p.bounds[tile_id];
        const int32_t diff = (int32_t)(bounds.y - bounds.x);
        const int num_splats = diff > 0 ? diff : 0;                              // :61
        const int num_iterations = (int)ceilf((float)num_splats / (float)CHUNK);  // :62

        u64 cr2 = pk(0.f, 0.f), cg2 = cr2, cb2 = cr2;  // blended colour of the two pixels
        float t0 = 1.0f, t1 = 1.0f;                    // transmittance of the two pixels

        Staged n0 = null_splat(), n1 = null_splat();
        if (num_iterations > 0) {
            if ((int)tid < num_splats) n0 = gather(records, p.values, bounds.x + tid);
            if ((int)tid + THREADS < num_splats) n1 = gather(records, p.values, bounds.x + tid + THREADS);
        }

        int consumed = 0;  // chunks blended before the stop rule fired (next frame's scheduling hint)
        for (int i = 0; i < num_iterations; ++i) {
            const int sort_offset = CHUNK * i;
            const int chunk = (num_splats - sort_offset) < CHUNK ? (num_splats - sort_offset) : CHUNK;
            staged += (uint32_t)chunk;
            consumed = i + 1;
            s_a[tid] = n0.a; s_b[tid] = n0.b; s_c[tid] = n0.c;
            s_a[tid + THREADS] = n1.a; s_b[tid + THREADS] = n1.b; s_c[tid + THREADS] = n1.c;
            __syncthreads();
            // prefetch the next chunk's records while this one is blended (slots past the list end become null splats)
            n0 = null_splat(); n1 = null_splat();
            if (i + 1 < num_iterations) {
                const int nb = sort_offset + CHUNK;
                if (nb + (int)tid < num_splats) n0 = gather(records, p.values, bounds.x + (uint32_t)nb + tid);
                if (nb + (int)tid + THREADS < num_splats) n1 = gather(records, p.values, bounds.x + (uint32_t)nb + tid + THREADS);
            }

            // :79-91, GU splats per iteration; `chunk` rounded up to GU reads null splats (opacity 0 => exact no-op).  Software-pipelined:
            // the (a, b) words of group g+1 are loaded while group g is blended, and the warp's "anybody alive?" test uses the
            // transmittance after the first half of the group -- a dead warp may blend one more (fully masked) group before it leaves.
            const int chunkg = (chunk + GU - 1) & ~(GU - 1);
            float4 A[GU], B[GU];
#pragma unroll
            for (int u = 0; u < GU; ++u) { A[u] = s_a[u]; B[u] = s_b[u]; }
            bool go = __any_sync(0xffffffffu, (t0 > MIN_ALPHA) || (t1 > MIN_ALPHA));
            for (int j = 0; j < chunkg && go; j += GU) {
                u64 al2[GU], om2[GU];
                phase_a<CONTRACT>(A, B, npx2, fpy, K, al2, om2);
                float4 Bc[GU];
#pragma unroll
                for (int u = 0; u < GU; ++u) Bc[u] = B[u];
                const int jn = (j + GU < CHUNK) ? j + GU : j;   // the last group re-reads itself instead of running off the array
#pragma unroll
                for (int u = 0; u < GU; ++u) { A[u] = s_a[jn + u]; B[u] = s_b[jn + u]; }
                bool alive_mid = true;
                phase_b<CONTRACT>(Bc, s_c, j, al2, om2, cr2, cg2, cb2, t0, t1, alive_mid);
                go = __any_sync(0xffffffffu, alive_mid);
            }

            // :97 tile-stop vote: continue only if the sum over the tile's 256 pixels of uint(t*255) exceeds 255
            const uint32_t wsum = __reduce_add_sync(0xffffffffu, (uint32_t)(t0 * 255.0f) + (uint32_t)(t1 * 255.0f));
            if (lane == 0) s_vote[warp] = wsum;
            __syncthreads();
            uint32_t shared_t = 0;
#pragma unroll
            for (int w = 0; w < THREADS / 32; ++w) shared_t += s_vote[w];
            if (!(shared_t > 255u)) break;
        }

        // :100-101
        float r0, r1, g0, g1, b0, b1;
        upk(cr2, r0, r1); upk(cg2, g0, g1); upk(cb2, b0, b1);
        const float hx = (float)num_splats * 5e-4f;
        const float h0 = 0.0f * (1.0f - hx) + 1.0f * hx, h1 = 0.0f * (1.0f - hx) + 0.2f * hx, h2c = 1.0f * (1.0f - hx) + 0.2f * hx;
        if (py < p.height) {
            float4 *row = out + (uint64_t)py * (uint64_t)p.width;
            const float k0 = 1.0f - t0, k1 = 1.0f - t1;
            if (px0 < p.width)
                row[px0] = make_float4(r0 + h0 * k0 * p.heatmap_factor, g0 + h1 * k0 * p.heatmap_factor, b0 + h2c * k0 * p.heatmap_factor, 1.0f);
            if (px0 + 1 < p.width)
                row[px0 + 1] = make_float4(r1 + h0 * k1 * p.heatmap_factor, g1 + h1 * k1 * p.heatmap_factor, b1 + h2c * k1 * p.heatmap_factor, 1.0f);
        }
        // :105-110 pick: the elected (first) lane of each 32-wide subgroup of the reference's 16x16 workgroup is local
        // index 32*s = pixel (0, 2*s) of the tile = first pixel of thread 16*s here
        if ((tid & 15u) == 0u && tile_id == p.target_tile_id && t0 != 1.0f) {
            const uint32_t v = p.values[bounds.x + (bounds.y - bounds.x) / 10u];
            const float4 q0 = records[(uint64_t)v * 3u + 0], q1 = records[(uint64_t)v * 3u + 1];
            *p.pick = make_float4(q0.z, q0.w, q1.w, (float)num_splats);
        }
        if (tid == 0) {
            if (p.consumed) p.consumed[local_tile] = (uint32_t)consumed | 0x80000000u;   // bit 31: written this frame
            if (p.trace) {
                const uint32_t k = atomicAdd(p.trace_count, 1u);
                if (k < p.trace_cap) p.trace[k] = make_ulonglong4(((unsigned long long)tile_id << 32) | smid(), t_start, globaltimer_ns(),
                                                                  ((unsigned long long)(uint32_t)consumed << 32) | 1u | ((uint32_t)num_iterations << 1));
            }
        }
        __syncthreads();  // s_tile / staging buffers are reused by the next tile
    }
    if (tid == 0 && staged && p.count_staged) atomicAdd(&p.frame->staged, (unsigned long long)staged);
}

}  // namespace

#ifndef GSR_CPU_EMU
int preload_composite_kernels() {
    cudaFuncAttributes fa;
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, composite_kernel<true, false>));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, composite_kernel<false, false>));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, composite_kernel<true, true>));
    GSR_CUDA_TRY(cudaFuncGetAttributes(&fa, composite_kernel<false, true>));
    return GSR_OK;
}

int composite_max_ctas_per_sm(int *out) {
    int a = 0, b = 0;
    GSR_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, composite_kernel<true, false>, THREADS, 0));
    GSR_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, composite_kernel<false, false>, THREADS, 0));
    *out = a < b ? a : b;
    if (*out < 1) *out = 1;
    return GSR_OK;
}

int launch_composite(const CompositeArgs &a, cudaStream_t stream) {
    if (a.num_tiles <= 0) return GSR_OK;
    const int per_sm = a.ctas_per_sm > 0 ? a.ctas_per_sm : 1;
    const int grid = a.num_tiles < a.sm_count * per_sm ? a.num_tiles : a.sm_count * per_sm;
    if (a.tiles_per_view > 0) {
        if (a.contract) composite_kernel<true, true><<<grid, THREADS, 0, stream>>>(a);
        else composite_kernel<false, true><<<grid, THREADS, 0, stream>>>(a);
    } else {
        if (a.contract) composite_kernel<true, false><<<grid, THREADS, 0, stream>>>(a);
        else composite_kernel<false, false><<<grid, THREADS, 0, stream>>>(a);
    }
    GSR_CUDA_TRY(cudaGetLastError());
    return GSR_OK;
}
#endif  // GSR_CPU_EMU

}  // namespace gsr
