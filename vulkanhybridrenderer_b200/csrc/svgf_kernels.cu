// svgf_kernels.cu — SVGF temporal accumulation + variance, and the à-trous wavelet filter (sm_100a).
//
//   svgf_temporal_kernel      <- /root/reference/data/shaders/hybrid_render_path/svgf.comp:16-145
//   atrous_direct_kernel      <- /root/reference/data/shaders/hybrid_render_path/svgf_atrous_filter.comp:17-103
//                                (one thread per pixel, 49 direct image loads: the reference's own dataflow)
//   atrous_tiled_kernel<S>    <- same arithmetic, B200 dataflow: a 64x8 output tile whose rows are S apart, staged
//                                once in shared memory as fp32 planes, so each texel is converted once instead of 25x
//                                and every tap is two 128-bit LDS; (shadow, ao) channel pairs run on packed
//                                fp32x2 instructions (FADD2/FMUL2/FFMA2).
//
// Images: dense row-major; RGBA16F texel = uint2, RG16F texel = uint32. fp32 math, fp16 RTE stores (SURVEY Q22).
#include <cuda.h>
#include <stdlib.h>

#include <algorithm>

#include "vhr_internal.h"

namespace vhr {

// ---------------------------------------------------------------------------------------------------------------
// Temporal pass
// ---------------------------------------------------------------------------------------------------------------
struct TemporalParams {
    int W, H;
    int x_end, y_begin, y_end;     // pixel range covered by this dispatch
    float dsx, dsy;                // pfd.display_size
    const uint2 *normals;          // binding 0
    const uint2 *motion;           // binding 1
    const uint32_t *rt;            // binding 3 (RG16F)
    const uint2 *prev_normals;     // storage_images[pc.prev_frame_normals_and_object_ids]
    const uint2 *history;          // storage_images[pc.shadow_and_ao_history]
    const uint32_t *moments_in;    // storage_images[pc.shadow_and_ao_moments_history] (previous frame, Q11 snapshot)
    uint2 *integrated_out;         // storage_images[pc.integrated_shadow_and_ao[0]]
    uint32_t *moments_out;
    HaloPush push_integ, push_mom; // multi-GPU: boundary rows also go to the neighbours' copies (NVLink peer stores)
};

// svgf.comp:16-39
__device__ __forceinline__ bool is_valid_reprojection(const TemporalParams &p, int px, int py, int cur_id, float3 cur_n) {
    if (px < 0 || py < 0 || (float)px >= p.dsx || (float)py >= p.dsy) return false;
    float4 pn = unpack_rgba16f(__ldg(&p.prev_normals[(size_t)py * p.W + px]));
    if (cur_id != f2i_rz(pn.w)) return false;
    if (dot3_rn(cur_n, make_float3(pn.x, pn.y, pn.z)) < VHR_COS_PI_4) return false;
    return true;
}

__device__ __forceinline__ float mix_rn(float a, float b, float t) { return add_rn(mul_rn(a, sub_rn(1.0f, t)), mul_rn(b, t)); }

// svgf.comp:41-145 for one pixel: the integrated[0] texel (shadow, ao, var_shadow, var_ao) and the moments texel, both as stored (fp16 RTE).
// `ntexel` = the pixel's normal / object-id texel (the caller has loaded it already).
struct TemporalOut { uint2 integ; uint32_t mom; };
__device__ __forceinline__ TemporalOut temporal_pixel(const TemporalParams &p, int cx, int cy, uint2 ntexel) {
    const size_t pix = (size_t)cy * p.W + cx;

    float4 cn = unpack_rgba16f(ntexel);
    float3 cur_n = make_float3(cn.x, cn.y, cn.z);
    int cur_id = f2i_rz(cn.w);
    float2 mv = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.motion[pix])));   // .xy only
    float2 cur = unpack_rg16f(__ldg(&p.rt[pix]));

    // svgf.comp:52-55
    float pcx = add_rn(sub_rn((float)cx, mul_rn(mv.x, p.dsx)), 0.5f);
    float pcy = add_rn(sub_rn((float)cy, mul_rn(mv.y, p.dsy)), 0.5f);
    float x = sub_rn(pcx, floorf(pcx)), y = sub_rn(pcy, floorf(pcy));
    int ax = f2i_rz(pcx), ay = f2i_rz(pcy);
    float omx = sub_rn(1.0f, x), omy = sub_rn(1.0f, y);
    const float bw[4] = {mul_rn(omx, omy), mul_rn(x, omy), mul_rn(omx, y), mul_rn(x, y)};

    float prev_s = 0.0f, prev_a = 0.0f, sum = 0.0f;
    float psm0 = 0.0f, psm1 = 0.0f, pam0 = 0.0f, pam1 = 0.0f;
    // All twelve tap loads (previous normals, history, moments of the 2x2 footprint) are issued before any of them is
    // examined: the reference's order (test the normal, then fetch history) costs a second dependent memory round trip
    // per pixel, and this kernel is bound by exactly that latency (profiles/: DRAM 23 %, long-scoreboard stalls).
    uint2 tpn[4];
    uint32_t th[4], tm[4];
    bool inb[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int sx = ax + (i & 1), sy = ay + (i >> 1);
        inb[i] = !(sx < 0 || sy < 0 || (float)sx >= p.dsx || (float)sy >= p.dsy);
        const size_t sp = inb[i] ? (size_t)sy * p.W + sx : pix;
        tpn[i] = __ldg(&p.prev_normals[sp]);
        th[i] = __ldg(reinterpret_cast<const uint32_t *>(&p.history[sp]));
        tm[i] = __ldg(&p.moments_in[sp]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 pn = unpack_rgba16f(tpn[i]);
        // is_valid_reprojection (svgf.comp:16-39) on the prefetched texel
        if (inb[i] && cur_id == f2i_rz(pn.w) && !(dot3_rn(cur_n, make_float3(pn.x, pn.y, pn.z)) < VHR_COS_PI_4)) {
            float2 h = unpack_rg16f(th[i]);
            float2 m = unpack_rg16f(tm[i]);
            prev_s = add_rn(prev_s, mul_rn(bw[i], h.x));
            prev_a = add_rn(prev_a, mul_rn(bw[i], h.y));
            psm0 = add_rn(psm0, mul_rn(bw[i], m.x));
            psm1 = add_rn(psm1, mul_rn(bw[i], m.y));
            // a two-channel image reads back (r, g, 0, 1): prev AO moments accumulate (0, w) — SURVEY Q2
            pam1 = add_rn(pam1, bw[i]);
            sum = add_rn(sum, bw[i]);
        }
    }
    bool valid = sum > 1e-6f;
    if (!valid) {   // svgf.comp:81-97, accumulators not reset
        for (int yy = -1; yy <= 1; ++yy)
            for (int xx = -1; xx <= 1; ++xx) {
                int sx = ax + xx, sy = ay + yy;
                if (is_valid_reprojection(p, sx, sy, cur_id, cur_n)) {
                    size_t sp = (size_t)sy * p.W + sx;
                    float2 h = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.history[sp])));
                    float2 m = unpack_rg16f(__ldg(&p.moments_in[sp]));
                    prev_s = add_rn(prev_s, h.x);
                    prev_a = add_rn(prev_a, h.y);
                    psm0 = add_rn(psm0, m.x);
                    psm1 = add_rn(psm1, m.y);
                    pam1 = add_rn(pam1, 1.0f);
                    sum = add_rn(sum, 1.0f);
                }
            }
        valid = sum > 1e-6f;
    }

    float sm0 = cur.x, sm1 = mul_rn(cur.x, cur.x);
    float am0 = cur.y, am1 = mul_rn(cur.y, cur.y);
    float4 out;
    if (valid) {
        // one correctly rounded reciprocal and five products instead of six IEEE divisions (<= 1.5 ulp apart in fp32, far
        // below the fp16 store; the kernel is issue-bound since its tap loads were batched)
        const float rs = __frcp_rn(sum);
        prev_s = mul_rn(prev_s, rs);
        psm0 = mul_rn(psm0, rs); psm1 = mul_rn(psm1, rs);
        prev_a = mul_rn(prev_a, rs);
        pam0 = mul_rn(pam0, rs); pam1 = mul_rn(pam1, rs);
        sm0 = mix_rn(psm0, sm0, 0.2f); sm1 = mix_rn(psm1, sm1, 0.2f);
        am0 = mix_rn(pam0, am0, 0.2f); am1 = mix_rn(pam1, am1, 0.2f);
        float sv = fmaxf(0.0f, sub_rn(sm1, mul_rn(sm0, sm0)));
        float av = fmaxf(0.0f, sub_rn(am1, mul_rn(am0, am0)));
        out = make_float4(mix_rn(prev_s, cur.x, 0.2f), mix_rn(prev_a, cur.y, 0.2f), sv, av);
    } else {
        float sv = fmaxf(0.0f, sub_rn(sm1, mul_rn(sm0, sm0)));
        float av = fmaxf(0.0f, sub_rn(am1, mul_rn(am0, am0)));
        out = make_float4(cur.x, cur.y, sv, av);
    }
    TemporalOut r;
    r.integ = pack_rgba16f(out);
    r.mom = pack_rg16f(sm0, sm1);      // RG16F keeps the shadow moments only (Q2)
    return r;
}

#ifndef VHR_TEMPORAL_MIN_BLOCKS
#define VHR_TEMPORAL_MIN_BLOCKS 1      // 6 / 8 (40 / 32 registers, spills) measured 2-4 us slower than the natural 48 registers / 5 blocks
#endif
__global__ void __launch_bounds__(256, VHR_TEMPORAL_MIN_BLOCKS) svgf_temporal_kernel(const __grid_constant__ TemporalParams p) {
    const int cx = blockIdx.x * 32 + threadIdx.x;
    const int cy = p.y_begin + blockIdx.y * 8 + threadIdx.y;
    if (cx >= p.x_end || cy >= p.y_end) return;
    const size_t pix = (size_t)cy * p.W + cx;
    const TemporalOut r = temporal_pixel(p, cx, cy, __ldg(&p.normals[pix]));
    const uint2 o = r.integ;
    const uint32_t m = r.mom;
    p.integrated_out[pix] = o;
    p.moments_out[pix] = m;
    if (p.push_integ.rows | p.push_mom.rows) {    // halo exchange fused into the kernel: the next pass on the neighbour reads these rows
        if (p.push_integ.up && cy < p.y_begin + p.push_integ.rows) reinterpret_cast<uint2 *>(p.push_integ.up)[pix] = o;
        if (p.push_integ.down && cy >= p.y_end - p.push_integ.rows) reinterpret_cast<uint2 *>(p.push_integ.down)[pix] = o;
        if (p.push_mom.up && cy < p.y_begin + p.push_mom.rows) reinterpret_cast<uint32_t *>(p.push_mom.up)[pix] = m;
        if (p.push_mom.down && cy >= p.y_end - p.push_mom.rows) reinterpret_cast<uint32_t *>(p.push_mom.down)[pix] = m;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// À-trous, variant 0: the reference's dataflow (one thread per pixel, direct loads); AtrousParams: vhr_internal.h
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_out(const AtrousParams &p, int cy, size_t pix, uint2 v) {
    p.integ_out[pix] = v;
    if (p.push.rows) {
        if (p.push.up && cy < p.y_begin + p.push.rows) reinterpret_cast<uint2 *>(p.push.up)[pix] = v;
        if (p.push.down && cy >= p.y_end - p.push.rows) reinterpret_cast<uint2 *>(p.push.down)[pix] = v;
    }
}

__constant__ float c_atrous_h[5] = {1.0f / 16, 1.0f / 4, 3.0f / 8, 1.0f / 4, 1.0f / 16};

__device__ __forceinline__ bool oob(const AtrousParams &p, int sx, int sy) {
    return sx < 0 || (float)sx >= p.dsx || sy < 0 || (float)sy >= p.dsy;
}

__global__ void __launch_bounds__(256) atrous_direct_kernel(const __grid_constant__ AtrousParams p) {
    const int cx = blockIdx.x * 32 + threadIdx.x;
    const int cy = p.y_begin + blockIdx.y * 8 + threadIdx.y;
    if (cx >= p.x_end || cy >= p.y_end) return;
    const size_t pix = (size_t)cy * p.W + cx;
    float4 np4 = unpack_rgba16f(__ldg(&p.normals[pix]));
    int id_p = f2i_rz(np4.w);
    float4 ip = unpack_rgba16f(__ldg(&p.integ_in[pix]));

    // gauss_3x3_filter: weights 1/16 1/8 1/16 ..., OOB skipped, row-major accumulation order
    float var_s = 0.0f, var_a = 0.0f;
#pragma unroll
    for (int y = -1; y <= 1; ++y)
#pragma unroll
        for (int x = -1; x <= 1; ++x) {
            int sx = cx + x, sy = cy + y;
            if (oob(p, sx, sy)) continue;
            float w = (x == 0 ? 0.5f : 0.25f) * (y == 0 ? 0.5f : 0.25f);
            float4 q = unpack_rgba16f(__ldg(&p.integ_in[(size_t)sy * p.W + sx]));
            var_s = add_rn(var_s, mul_rn(w, q.z));
            var_a = add_rn(var_a, mul_rn(w, q.w));
        }
    float den_s = add_rn(mul_rn(4.0f, sqrtf(var_s)), 1e-6f);
    float den_a = add_rn(mul_rn(4.0f, sqrtf(var_a)), 1e-6f);

    float swx = 1.0f, swy = 1.0f;
    float4 sum = ip;
    for (int y = -2; y <= 2; ++y)
        for (int x = -2; x <= 2; ++x) {
            int sx = cx + x * p.step, sy = cy + y * p.step;
            if (oob(p, sx, sy) || (x == 0 && y == 0)) continue;
            size_t sp = (size_t)sy * p.W + sx;
            float4 iq = unpack_rgba16f(__ldg(&p.integ_in[sp]));
            float4 nq = unpack_rgba16f(__ldg(&p.normals[sp]));
            float kernel = c_atrous_h[y + 2] * c_atrous_h[x + 2];
            float d = add_rn(add_rn(mul_rn(np4.x, nq.x), mul_rn(np4.y, nq.y)), mul_rn(np4.z, nq.z));
            float wn = (d > 0.0f) ? fmaxf(0.0f, powf(d, 128.0f)) : 0.0f;       // SURVEY Q10
            float wid = (id_p == f2i_rz(nq.w)) ? 1.0f : 0.0f;
            float wk = mul_rn(mul_rn(kernel, wn), wid);
            float wx = mul_rn(wk, expf(-__fdiv_rn(fabsf(sub_rn(ip.x, iq.x)), den_s)));
            float wy = mul_rn(wk, expf(-__fdiv_rn(fabsf(sub_rn(ip.y, iq.y)), den_a)));
            swx = add_rn(swx, wx);
            swy = add_rn(swy, wy);
            sum.x = add_rn(sum.x, mul_rn(wx, iq.x));
            sum.y = add_rn(sum.y, mul_rn(wy, iq.y));
            sum.z = add_rn(sum.z, mul_rn(mul_rn(wx, wx), iq.z));
            sum.w = add_rn(sum.w, mul_rn(mul_rn(wy, wy), iq.w));
        }
    float4 out = make_float4(__fdiv_rn(sum.x, swx), __fdiv_rn(sum.y, swy), __fdiv_rn(sum.z, mul_rn(swx, swx)),
                             __fdiv_rn(sum.w, mul_rn(swy, swy)));
    store_out(p, cy, pix, pack_rgba16f(out));
}

// ---------------------------------------------------------------------------------------------------------------
// À-trous, variant 1: shared-memory tile with rows S apart + packed fp32x2 math
// ---------------------------------------------------------------------------------------------------------------
// Packed fp32x2 arithmetic (Blackwell FADD2 / FMUL2 / FFMA2): two IEEE fp32 operations per issue slot.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{ .reg .b64 ra, rb, rc, rd;\n\t"
        "mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; mov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\t"
        "mov.b64 {%0, %1}, rd; }"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    float2 d;
    asm("{ .reg .b64 ra, rb, rd;\n\t"
        "mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rd, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rd; }"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    float2 d;
    asm("{ .reg .b64 ra, rb, rd;\n\t"
        "mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5};\n\t"
        "add.rn.f32x2 rd, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rd; }"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

constexpr int AT_TX = 64;    // output tile width (pixels, contiguous)
constexpr int AT_TY = 8;     // output tile height (rows, S apart)

template <int S>
__global__ void __launch_bounds__(AT_TX * AT_TY, 2) atrous_tiled_kernel(const __grid_constant__ AtrousParams p) {
    constexpr int COLS = AT_TX + 4 * S;
    constexpr int ROWS = AT_TY + 4;
    extern __shared__ float4 smem[];
    float4 *s_n = smem;                    // [ROWS][COLS] normal.xyz, object id (as float)
    float4 *s_i = smem + ROWS * COLS;      // [ROWS][COLS] shadow, ao, var_shadow, var_ao

    const int tx = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * AT_TX + tx;
    const int x0 = blockIdx.x * AT_TX;
    // blockIdx.y enumerates (super-tile k, residue r): rows y = y_begin + k*S*TY + r + S*j
    const int k = blockIdx.y / S, r = blockIdx.y % S;
    const int yb = p.y_begin + k * (S * AT_TY) + r;

    // ---- stage the tile: each texel is loaded and converted to fp32 once -----------------------------------
    for (int idx = tid; idx < ROWS * COLS; idx += AT_TX * AT_TY) {
        int row = idx / COLS, col = idx - row * COLS;
        int gx = x0 - 2 * S + col;
        int gy = yb + (row - 2) * S;
        float4 n = make_float4(0.0f, 0.0f, 0.0f, -1.0f);   // out of bounds: zero normal => weight 0 ("skipped")
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (gx >= 0 && gx < p.W && gy >= 0 && gy < p.H) {
            size_t sp = (size_t)gy * p.W + gx;
            n = unpack_rgba16f(__ldg(&p.normals[sp]));
            v = unpack_rgba16f(__ldg(&p.integ_in[sp]));
            n.w = (float)f2i_rz(n.w);
        }
        s_n[idx] = n;
        s_i[idx] = v;
    }
    __syncthreads();

    const int cx = x0 + tx;
    const int cy = yb + ty * S;
    if (cx >= p.x_end || cy >= p.y_end) return;

    const int crow = ty + 2, ccol = tx + 2 * S;
    const float4 np4 = s_n[crow * COLS + ccol];
    const float4 ip = s_i[crow * COLS + ccol];

    // ---- 3x3 gaussian of the variance (same accumulation order as the reference) ----------------------------
    float2 var = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int y = -1; y <= 1; ++y)
#pragma unroll
        for (int x = -1; x <= 1; ++x) {
            const float w = (x == 0 ? 0.5f : 0.25f) * (y == 0 ? 0.5f : 0.25f);
            float2 q;
            if (S == 1) {
                float4 t = s_i[(crow + y) * COLS + ccol + x];   // OOB texels staged as 0 => contribute 0
                q = make_float2(t.z, t.w);
            } else if (y == 0) {
                float4 t = s_i[crow * COLS + ccol + x];
                q = make_float2(t.z, t.w);
            } else {
                int sx = cx + x, sy = cy + y;
                q = make_float2(0.0f, 0.0f);
                if (sx >= 0 && sx < p.W && sy >= 0 && sy < p.H)
                    q = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.integ_in[(size_t)sy * p.W + sx]) + 1));
            }
            var.x = add_rn(var.x, mul_rn(w, q.x));
            var.y = add_rn(var.y, mul_rn(w, q.y));
        }
    // exp(-|dl| / (4 sqrt(var) + 1e-6)) = exp2(|dl| * nk), nk = -log2(e) / (4 sqrt(var) + 1e-6)
    const float LOG2E = 1.4426950408889634f;
    float2 nk = make_float2(__fdiv_rn(-LOG2E, add_rn(mul_rn(4.0f, sqrtf(var.x)), 1e-6f)),
                            __fdiv_rn(-LOG2E, add_rn(mul_rn(4.0f, sqrtf(var.y)), 1e-6f)));
    const float2 lp = make_float2(ip.x, ip.y);
    const float2 neg_lp = make_float2(-ip.x, -ip.y);

    float2 sw = make_float2(1.0f, 1.0f);
    float2 sc = make_float2(ip.x, ip.y);     // colour sums
    float2 sv = make_float2(ip.z, ip.w);     // variance sums
    (void)lp;
#pragma unroll
    for (int y = -2; y <= 2; ++y) {
#pragma unroll
        for (int x = -2; x <= 2; ++x) {
            if (x == 0 && y == 0) continue;
            const int o = (crow + y) * COLS + ccol + x * S;
            const float4 nq = s_n[o];
            const float4 iq = s_i[o];
            const float kernel = ((y == 0) ? 0.375f : ((y == 1 || y == -1) ? 0.25f : 0.0625f)) *
                                 ((x == 0) ? 0.375f : ((x == 1 || x == -1) ? 0.25f : 0.0625f));
            float d = np4.x * nq.x + np4.y * nq.y + np4.z * nq.z;
            float d2 = d * d, d4 = d2 * d2, d8 = d4 * d4, d16 = d8 * d8, d32 = d16 * d16, d64 = d32 * d32;
            float wn = d64 * d64;                                                   // d^128
            float wk = (d > 0.0f && nq.w == np4.w) ? kernel * wn : 0.0f;            // Q10 + object-id edge stop
            float2 dl = add2(make_float2(iq.x, iq.y), neg_lp);                      // l_q - l_p
            float2 e = mul2(make_float2(fabsf(dl.x), fabsf(dl.y)), nk);
            float2 w = mul2(make_float2(wk, wk), make_float2(ex2_approx(e.x), ex2_approx(e.y)));
            sw = add2(sw, w);
            sc = fma2(w, make_float2(iq.x, iq.y), sc);
            sv = fma2(mul2(w, w), make_float2(iq.z, iq.w), sv);
        }
    }
    float4 out = make_float4(__fdiv_rn(sc.x, sw.x), __fdiv_rn(sc.y, sw.y), __fdiv_rn(sv.x, mul_rn(sw.x, sw.x)),
                             __fdiv_rn(sv.y, mul_rn(sw.y, sw.y)));
    store_out(p, cy, (size_t)cy * p.W + cx, pack_rgba16f(out));
}

template <int S>
static int launch_tiled(vhr_context *ctx, const AtrousParams &p, int x_pixels, int y_pixels) {
    constexpr int COLS = AT_TX + 4 * S, ROWS = AT_TY + 4;
    constexpr size_t smem = (size_t)2 * ROWS * COLS * sizeof(float4);
    static_assert(smem <= 48 * 1024, "tile must fit the default dynamic shared memory limit");
    dim3 block(AT_TX, AT_TY);
    dim3 grid((x_pixels + AT_TX - 1) / AT_TX, ((y_pixels + S * AT_TY - 1) / (S * AT_TY)) * S);
    atrous_tiled_kernel<S><<<grid, block, smem, ctx->stream>>>(p);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// À-trous, variant 2 (default): pixel pairs on packed fp32x2 + register-level tap reuse
// ---------------------------------------------------------------------------------------------------------------
// The first profile of variant 1 (profiles/r01_ncu_full_summary.md) shows the filter bound by instruction issue (70 %)
// and shared-memory bandwidth (2 x LDS.128 per tap and pixel = 63 % of the LSU's wavefront rate), not by HBM (5 %).
// This variant attacks both:
//   * a thread owns a PAIR of pixels PD columns apart and every shared-memory plane stores the two pixels' values side
//     by side, so one LDS.128 delivers two aligned register pairs and the WHOLE tap pipeline — normal dot product, id
//     edge stop, the seven squarings of d^128, luminance weights, all accumulations — runs on FMUL2/FFMA2/FADD2
//     (two pixels per issue slot instead of two channels of one pixel);
//   * a thread owns RY lattice-adjacent rows of that pair, so a loaded tap is used by up to RY outputs
//     ((RY+4)*5 loads for RY*25 taps) — shared-memory traffic per tap drops by 5*RY/(RY+4);
//   * FFMA2 halves the issue slots but not the FP32 lane-cycles (measured: the first packed version, 28.75 FP32 ops per
//     tap and pixel, ran no faster than variant 1), so the arithmetic itself is cut: kernel weight, d^128 (a cubic in
//     d - 1 for 128 log2 d) and both luminance stops fold into the argument of ONE ex2 per channel, the id stop is an
//     integer compare + select on the ALU pipe. 18 FP32 ops + 2 MUFU.EX2 + 2 ALU ops per tap and pixel.
// Degree of the polynomial for 128 log2(1 + e) in the tap weight (see pair_compute). 2: the cubic term is dropped — it only matters where
// the weight is already small: the absolute weight error 2^(184.7 e) * ln 2 * 61.6 |e|^3 peaks at 2.7e-5 (e = -0.023) before the kernel
// factor h <= 3/32, i.e. < 3e-6 per tap against a weight sum >= 1. One FFMA2 per tap and pixel pair less.
#ifndef VHR_ATROUS_POLY_DEGREE
#define VHR_ATROUS_POLY_DEGREE 2
#endif
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void upk_u32(u64 v, uint32_t &lo, uint32_t &hi) { asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v)); }
__device__ __forceinline__ u64 pmul(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 padd(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 pfma(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 pclamp0(u64 v) { float a, b; upk(v, a, b); return pk(fmaxf(a, 0.0f), fmaxf(b, 0.0f)); }
__device__ __forceinline__ u64 pex2_negabs(u64 v) { float a, b; upk(v, a, b); return pk(ex2_approx(-fabsf(a)), ex2_approx(-fabsf(b))); }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sqrt_approx(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

template <int S, int PD, int RY, int TR>
struct PairCfg {
    static constexpr int PC = PD + 4 * S;        // staged pair-columns per row
    static constexpr int LR = TR * RY;           // lattice rows (S apart) per CTA
    static constexpr int SR = LR + 4;            // staged rows
    static constexpr int THREADS = PD * TR;
    static constexpr size_t PLANES = (size_t)4 * SR * PC * sizeof(ulonglong2);
    // S > 1: the 3x3 variance gaussian reads rows y - 1 and y + 1 of every output row, which are not lattice rows of the tile; their
    // (var_shadow, var_ao) half pairs are staged raw, 2 LR rows of XW = 2 PD + 2 pixels (columns x0 - 1 .. x0 + 2 PD)
    static constexpr int XW = 2 * PD + 2;
    static constexpr size_t VXROWS = (S > 1) ? (size_t)2 * LR * XW * sizeof(uint32_t) : 0;
    static constexpr size_t SMEM = PLANES + VXROWS;
};

// Taps + normalisation + store for one staged tile (shared by the direct-staging and the TMA-staged kernels): thread
// (tx, ty) owns pixel columns x0 + tx and x0 + tx + PD on the RY lattice rows ty*RY.. of the tile whose first row is yb.
template <int S, int PD, int RY, int TR, bool VX = false>
__device__ __forceinline__ void pair_compute(const AtrousParams &p, const ulonglong2 *__restrict__ sN0, const ulonglong2 *__restrict__ sN1,
                                             const ulonglong2 *__restrict__ sL, const ulonglong2 *__restrict__ sV, int x0, int yb, int tx, int ty,
                                             const uint32_t *__restrict__ sVx = nullptr) {
    typedef PairCfg<S, PD, RY, TR> C;
    constexpr int PC = C::PC;
    const int ca = x0 + tx, cb = ca + PD;
    const int lr0 = ty * RY;
    if (ca >= p.x_end || yb + lr0 * S >= p.y_end) return;
    const int jc = tx + 2 * S;

    // ---- per-output set-up ----------------------------------------------------------------------------------------
    u64 pnx[RY], pny[RY], pnz[RY], nls[RY], nla[RY];
    uint32_t ida[RY], idb[RY];
    float ksa[RY], ksb[RY], kaa[RY], kab[RY];
    u64 sws[RY], swa[RY], scs[RY], sca[RY], svs[RY], sva[RY];
    const u64 ONE = pk(1.0f, 1.0f);
#pragma unroll
    for (int i = 0; i < RY; ++i) {
        const int oc = (lr0 + i + 2) * PC + jc;
        const ulonglong2 n0 = sN0[oc], n1 = sN1[oc], l = sL[oc], v = sV[oc];
        pnx[i] = n0.x; pny[i] = n0.y; pnz[i] = n1.x;
        upk_u32(n1.y, ida[i], idb[i]);
        float a, b;
        upk(l.x, a, b); nls[i] = pk(-a, -b);
        upk(l.y, a, b); nla[i] = pk(-a, -b);
        sws[i] = ONE; swa[i] = ONE; scs[i] = l.x; sca[i] = l.y; svs[i] = v.x; sva[i] = v.y;

        // 3x3 gaussian of the variance, reference accumulation order; weights are powers of two, so the fused
        // multiply-adds round exactly like the reference's separate multiply and add
        u64 gs = pk(0.0f, 0.0f), ga = gs;
        const int cy = yb + (lr0 + i) * S;
#pragma unroll
        for (int y = -1; y <= 1; ++y)
#pragma unroll
            for (int x = -1; x <= 1; ++x) {
                const float w = (x == 0 ? 0.5f : 0.25f) * (y == 0 ? 0.5f : 0.25f);
                u64 qs, qa;
                if (S == 1 || y == 0) {
                    const ulonglong2 t = sV[oc + y * PC + x];          // OOB texels staged as 0
                    qs = t.x; qa = t.y;
                } else if (VX) {
                    // rows y - 1 / y + 1 staged by the kernel (out-of-image texels as 0)
                    const uint32_t *rowp = sVx + ((lr0 + i) * 2 + (y > 0 ? 1 : 0)) * C::XW + tx + x + 1;
                    const float2 ta = unpack_rg16f(rowp[0]), tb = unpack_rg16f(rowp[PD]);
                    qs = pk(ta.x, tb.x); qa = pk(ta.y, tb.y);
                } else {
                    const int sy = cy + y;
                    float2 ta = make_float2(0.0f, 0.0f), tb = ta;
                    if (sy >= 0 && sy < p.H) {
                        const uint32_t *rowp = reinterpret_cast<const uint32_t *>(p.integ_in + (size_t)sy * p.W);
                        const int xa = ca + x, xb = cb + x;
                        if (xa >= 0 && xa < p.W) ta = unpack_rg16f(__ldg(rowp + 2 * xa + 1));
                        if (xb >= 0 && xb < p.W) tb = unpack_rg16f(__ldg(rowp + 2 * xb + 1));
                    }
                    qs = pk(ta.x, tb.x); qa = pk(ta.y, tb.y);
                }
                gs = pfma(pk(w, w), qs, gs);
                ga = pfma(pk(w, w), qa, ga);
            }
        // exp(-|dl| / (4 sqrt(var) + 1e-6)) = exp2(-|dl| * k), k = log2(e) / (4 sqrt(var) + 1e-6)
        const float LOG2E = 1.4426950408889634f;
        float gsa, gsb, gaa, gab;
        upk(gs, gsa, gsb); upk(ga, gaa, gab);
        ksa[i] = LOG2E * rcp_approx(fmaf(4.0f, sqrt_approx(gsa), 1e-6f));
        ksb[i] = LOG2E * rcp_approx(fmaf(4.0f, sqrt_approx(gsb), 1e-6f));
        kaa[i] = LOG2E * rcp_approx(fmaf(4.0f, sqrt_approx(gaa), 1e-6f));
        kab[i] = LOG2E * rcp_approx(fmaf(4.0f, sqrt_approx(gab), 1e-6f));
    }

    // ---- taps: each staged texel pair is loaded once and used by every output row it is a tap of ------------------
    // All three edge stops and the kernel weight go through ONE exponential per channel:
    //     w = h * max(d,0)^128 * [id_q == id_p] * exp(-|dl|/sigma) = exp2(g - |dl| * k)
    //     g = log2(h) + 128 log2(d),  128 log2(1+e) ~ C1 e + C2 e^2 + C3 e^3   (e = d - 1, from the dot product started at -1)
    // The cubic's error in g is 46 e^4: below 1e-6 in the weight for every d (where |e| is large the weight itself is
    // < 1e-5), i.e. less than the rounding of the seven fp32 squarings it replaces; d <= 0 gives g <= -338 => w = 0
    // (pow()'s negative-base rule, SURVEY Q10); a different object id replaces g by -1e30 => w = 0.
    const u64 M1 = pk(-1.0f, -1.0f);
    const u64 C1 = pk(184.66496523378731f, 184.66496523378731f);
    const u64 C2 = pk(-92.33248261689366f, -92.33248261689366f);
#if VHR_ATROUS_POLY_DEGREE >= 3
    const u64 C3 = pk(61.55498841126244f, 61.55498841126244f);
#endif
#pragma unroll
    for (int tr = 0; tr < RY + 4; ++tr) {
#pragma unroll
        for (int x = -2; x <= 2; ++x) {
            const int o = (lr0 + tr) * PC + jc + x * S;
            const ulonglong2 n0 = sN0[o], n1 = sN1[o], l = sL[o], v = sV[o];
            uint32_t qa, qb;
            upk_u32(n1.y, qa, qb);      // (a plain shift makes ptxas compare 64-bit values: three ISETP per pair instead of two)
#pragma unroll
            for (int i = 0; i < RY; ++i) {
                const int y = tr - 2 - i;                       // this texel is tap (x, y) of output row i
                if (y < -2 || y > 2 || (x == 0 && y == 0)) continue;
                // log2 of the kernel weight h(y) h(x), h = (1/16, 1/4, 3/8, 1/4, 1/16)
                const float lgh = ((y == 0) ? -1.4150374992788437f : ((y == 1 || y == -1) ? -2.0f : -4.0f)) +
                                  ((x == 0) ? -1.4150374992788437f : ((x == 1 || x == -1) ? -2.0f : -4.0f));
                u64 e = pfma(pnx[i], n0.x, M1);
                e = pfma(pny[i], n0.y, e);
                e = pfma(pnz[i], n1.x, e);
#if VHR_ATROUS_POLY_DEGREE >= 3
                u64 u = pfma(C3, e, C2);
                u = pfma(u, e, C1);
#else
                const u64 u = pfma(C2, e, C1);
#endif
                const u64 g = pfma(u, e, pk(lgh, lgh));
                float ga, gb, da, db;
                upk(g, ga, gb);
                ga = (qa == ida[i]) ? ga : -1.0e30f;
                gb = (qb == idb[i]) ? gb : -1.0e30f;
                upk(padd(l.x, nls[i]), da, db);
                const u64 wsh = pk(ex2_approx(fmaf(-fabsf(da), ksa[i], ga)), ex2_approx(fmaf(-fabsf(db), ksb[i], gb)));
                upk(padd(l.y, nla[i]), da, db);
                const u64 wao = pk(ex2_approx(fmaf(-fabsf(da), kaa[i], ga)), ex2_approx(fmaf(-fabsf(db), kab[i], gb)));
                sws[i] = padd(sws[i], wsh);
                swa[i] = padd(swa[i], wao);
                scs[i] = pfma(wsh, l.x, scs[i]);
                sca[i] = pfma(wao, l.y, sca[i]);
                svs[i] = pfma(pmul(wsh, wsh), v.x, svs[i]);
                sva[i] = pfma(pmul(wao, wao), v.y, sva[i]);
            }
        }
    }

    // ---- normalise, fp16 RTE store -----------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < RY; ++i) {
        const int cy = yb + (lr0 + i) * S;
        if (cy >= p.y_end) break;
        float wsa, wsb, waa, wab, csa, csb, caa, cab, vsa, vsb, vaa, vab;
        upk(sws[i], wsa, wsb); upk(swa[i], waa, wab);
        upk(scs[i], csa, csb); upk(sca[i], caa, cab);
        upk(svs[i], vsa, vsb); upk(sva[i], vaa, vab);
        const float rsa = rcp_approx(wsa), rsb = rcp_approx(wsb), raa = rcp_approx(waa), rab = rcp_approx(wab);
        const size_t orow = (size_t)cy * p.W;
        store_out(p, cy, orow + ca, pack_rgba16f(make_float4(csa * rsa, caa * raa, vsa * (rsa * rsa), vaa * (raa * raa))));
        if (cb < p.x_end) store_out(p, cy, orow + cb, pack_rgba16f(make_float4(csb * rsb, cab * rab, vsb * (rsb * rsb), vab * (rab * rab))));
    }
}

template <int S, int PD, int RY, int TR>
__global__ void __launch_bounds__(PD * TR, (PD * TR <= 128) ? 4 : 2) atrous_pair_kernel(const __grid_constant__ AtrousParams p) {
    typedef PairCfg<S, PD, RY, TR> C;
    constexpr int PC = C::PC, SR = C::SR, LR = C::LR;
    extern __shared__ ulonglong2 psm[];
    ulonglong2 *sN0 = psm;                 // (nx_a, nx_b), (ny_a, ny_b)
    ulonglong2 *sN1 = psm + SR * PC;       // (nz_a, nz_b), (id_a, id_b)
    ulonglong2 *sL = psm + 2 * SR * PC;    // (shadow_a, shadow_b), (ao_a, ao_b)
    ulonglong2 *sV = psm + 3 * SR * PC;    // (var_shadow_a, var_shadow_b), (var_ao_a, var_ao_b)
    uint32_t *sVx = reinterpret_cast<uint32_t *>(psm + 4 * SR * PC);   // S > 1: raw (var_shadow, var_ao) of the rows above / below every lattice row

    const int tx = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * PD + tx;
    const int x0 = blockIdx.x * (2 * PD);
    const int k = blockIdx.y / S, r = blockIdx.y % S;       // (super-tile, residue): rows y = yb + S*j
    const int yb = p.y_begin + k * (S * LR) + r;
    constexpr int NVX = (S > 1) ? (2 * LR * C::XW + C::THREADS - 1) / C::THREADS : 0;
    uint32_t rvx[NVX > 0 ? NVX : 1];
    if (S > 1) {
#pragma unroll
        for (int it = 0; it < NVX; ++it) {
            const int idx = tid + it * C::THREADS;
            const int e = idx / C::XW, c = idx - e * C::XW;
            const int gy = yb + (e >> 1) * S + ((e & 1) ? 1 : -1), gx = x0 - 1 + c;
            rvx[it] = 0u;
            if (idx < 2 * LR * C::XW && gy >= 0 && gy < p.H && gx >= 0 && gx < p.W) rvx[it] = __ldg(reinterpret_cast<const uint32_t *>(p.integ_in + (size_t)gy * p.W + gx) + 1);
        }
    }

    // ---- stage: every texel converted to fp32 once, pixel a = column j, pixel b = column j + PD ------------------
    // Two sweeps (all loads, then convert + store) so that every global load of the tile is in flight at once: the
    // first profile of this kernel had its warps parked on long-scoreboard stalls, one round trip per loop iteration.
    constexpr int NIT = (SR * PC + C::THREADS - 1) / C::THREADS;
    uint2 rna[NIT], rnb[NIT], rva[NIT], rvb[NIT];
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
        const int idx = tid + it * C::THREADS;
        const int row = idx / PC, j = idx - row * PC;
        const int gy = yb + (row - 2) * S;
        const int gxa = x0 - 2 * S + j, gxb = gxa + PD;
        rna[it] = rnb[it] = rva[it] = rvb[it] = make_uint2(0u, 0u);     // out of bounds: zero normal => weight 0 ("skipped")
        if (idx < SR * PC && gy >= 0 && gy < p.H) {
            const size_t rowp = (size_t)gy * p.W;
            if (gxa >= 0 && gxa < p.W) { rna[it] = __ldg(&p.normals[rowp + gxa]); rva[it] = __ldg(&p.integ_in[rowp + gxa]); }
            if (gxb >= 0 && gxb < p.W) { rnb[it] = __ldg(&p.normals[rowp + gxb]); rvb[it] = __ldg(&p.integ_in[rowp + gxb]); }
        }
    }
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
        const int idx = tid + it * C::THREADS;
        if (idx < SR * PC) {
            const float4 na = unpack_rgba16f(rna[it]), nb = unpack_rgba16f(rnb[it]);
            const float4 va = unpack_rgba16f(rva[it]), vb = unpack_rgba16f(rvb[it]);
            const int ia = f2i_rz(na.w), ib = f2i_rz(nb.w);
            sN0[idx] = make_ulonglong2(pk(na.x, nb.x), pk(na.y, nb.y));
            sN1[idx] = make_ulonglong2(pk(na.z, nb.z), (u64)(uint32_t)ia | ((u64)(uint32_t)ib << 32));
            sL[idx] = make_ulonglong2(pk(va.x, vb.x), pk(va.y, vb.y));
            sV[idx] = make_ulonglong2(pk(va.z, vb.z), pk(va.w, vb.w));
        }
    }
    if (S > 1) {
#pragma unroll
        for (int it = 0; it < NVX; ++it) {
            const int idx = tid + it * C::THREADS;
            if (idx < 2 * LR * C::XW) sVx[idx] = rvx[it];
        }
    }
    __syncthreads();

    pair_compute<S, PD, RY, TR, (S > 1)>(p, sN0, sN1, sL, sV, x0, yb, tx, ty, sVx);
}

// ---------------------------------------------------------------------------------------------------------------
// svgf.comp + the first a-trous iteration in ONE kernel (VHR_OPT_SVGF_FUSED, north_star "fused reprojection + variance + first
// a-trous step"; reference sequence hybrid_render_path.cpp:299-307)
// ---------------------------------------------------------------------------------------------------------------
// The pair kernel's staging sweep does not LOAD the integrated[0] texels of its tile + 2-pixel halo, it COMPUTES them: every staged
// pixel runs temporal_pixel() (the whole of svgf.comp), the result is rounded to fp16 exactly as the image store would and goes
// straight into the shared-memory planes; pixels inside the tile also write integrated[0] and the moments image, so every image
// ends up bit-identical to the two-kernel sequence. Halo pixels are recomputed by the neighbouring CTAs ((PD + 4) (LR + 4) 2 evaluations
// per 2 PD LR outputs = 1.59x for the 128 x 8 tile). What it saves: one launch, the re-read of integrated[0] and of the normals.
template <int PD, int RY, int TR>
__global__ void __launch_bounds__(PD * TR, 2) svgf_fused_kernel(const __grid_constant__ TemporalParams t, const __grid_constant__ AtrousParams p) {
    typedef PairCfg<1, PD, RY, TR> C;
    constexpr int PC = C::PC, SR = C::SR, LR = C::LR;
    extern __shared__ ulonglong2 psm[];
    ulonglong2 *sN0 = psm, *sN1 = psm + SR * PC, *sL = psm + 2 * SR * PC, *sV = psm + 3 * SR * PC;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * PD + tx;
    const int x0 = blockIdx.x * (2 * PD);
    const int yb = p.y_begin + blockIdx.y * LR;
    for (int idx = tid; idx < SR * PC; idx += C::THREADS) {
        const int row = idx / PC, j = idx - row * PC;
        const int gy = yb + row - 2;
        // one staged pixel: the tile's own pixels also leave the kernel (side a owns columns [x0, x0 + PD), side b [x0 + PD, x0 + 2 PD))
        auto stage = [&](int gx, int c0, float4 &n, float4 &v) {
            n = make_float4(0.0f, 0.0f, 0.0f, 0.0f);        // out of bounds: zero normal => weight 0 ("skipped")
            v = n;
            if (gy >= 0 && gy < p.H && gx >= 0 && gx < p.W) {
                const size_t pix = (size_t)gy * p.W + gx;
                const uint2 nt = __ldg(&p.normals[pix]);
                const TemporalOut r = temporal_pixel(t, gx, gy, nt);
                if (row >= 2 && row < 2 + LR && gy < t.y_end && gx >= c0 && gx < c0 + PD && gx < t.x_end) {
                    t.integrated_out[pix] = r.integ;
                    t.moments_out[pix] = r.mom;
                }
                n = unpack_rgba16f(nt);
                v = unpack_rgba16f(r.integ);
            }
        };
        float4 na, va, nb, vb;
        stage(x0 - 2 + j, x0, na, va);
        stage(x0 - 2 + j + PD, x0 + PD, nb, vb);
        const int ia = f2i_rz(na.w), ib = f2i_rz(nb.w);
        sN0[idx] = make_ulonglong2(pk(na.x, nb.x), pk(na.y, nb.y));
        sN1[idx] = make_ulonglong2(pk(na.z, nb.z), (u64)(uint32_t)ia | ((u64)(uint32_t)ib << 32));
        sL[idx] = make_ulonglong2(pk(va.x, vb.x), pk(va.y, vb.y));
        sV[idx] = make_ulonglong2(pk(va.z, vb.z), pk(va.w, vb.w));
    }
    __syncthreads();
    pair_compute<1, PD, RY, TR>(p, sN0, sN1, sL, sV, x0, yb, tx, ty);
}

// ---------------------------------------------------------------------------------------------------------------
// À-trous, variant 3 (default for steps 1..8): variant 2's arithmetic in a persistent CTA with TMA-staged tiles
// ---------------------------------------------------------------------------------------------------------------
// The profile of variant 2 (profiles/r01_ncu_atrous_pair.md) attributes a third of its warp-time to staging: address
// arithmetic, bounds predicates, and above all the global-load round trip in front of every tile, with only two CTAs per
// SM to hide it. Here one elected thread hands the whole tile + halo to the TMA unit:
//   * the images are described to TMA as 3-D tensors (x, row mod S, row div S) of 8-byte texels, so one
//     cp.async.bulk.tensor box {2 PD + 4 S texels, 1, LR + 4} fetches rows S apart; out-of-image coordinates arrive as
//     zeros (= taps the reference skips), no bounds code anywhere;
//   * the CTA is persistent over tiles: the raw fp16 box of tile t+1 lands in shared memory (mbarrier complete_tx)
//     while the taps of tile t run; a short convert sweep (LDS raw -> fp32 pair planes) replaces the staging loop.
struct AtrousTmaParams {
    AtrousParams a;
    int n_tx, n_tiles;         // tiles per row of tiles, total (n_tx * tile rows * S)
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, int c0, int c1, int c2, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(smem_u32(dst)),
                 "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
                 : "memory");
}

template <int S, int PD, int RY, int TR>
struct TmaCfg {
    typedef PairCfg<S, PD, RY, TR> C;
    static constexpr int PCT = 2 * PD + 4 * S;                                 // staged texels per row (the TMA box width)
    static constexpr size_t PLANES = (size_t)4 * C::SR * C::PC * sizeof(ulonglong2);
    static constexpr size_t RAW = (size_t)C::SR * PCT * sizeof(uint2);         // one raw image box
    static constexpr size_t SMEM = PLANES + 2 * RAW + 16;
};

template <int S, int PD, int RY, int TR>
__global__ void __launch_bounds__(PD * TR, 2) atrous_tma_kernel(const __grid_constant__ AtrousTmaParams q, const __grid_constant__ CUtensorMap map_normals,
                                                                const __grid_constant__ CUtensorMap map_integ) {
    typedef PairCfg<S, PD, RY, TR> C;
    typedef TmaCfg<S, PD, RY, TR> T;
    constexpr int PC = C::PC, SR = C::SR, LR = C::LR, PCT = T::PCT;
    const AtrousParams &p = q.a;
    extern __shared__ __align__(128) unsigned char tsm[];
    ulonglong2 *sN0 = reinterpret_cast<ulonglong2 *>(tsm);
    ulonglong2 *sN1 = sN0 + SR * PC, *sL = sN0 + 2 * SR * PC, *sV = sN0 + 3 * SR * PC;
    uint2 *raw_n = reinterpret_cast<uint2 *>(tsm + T::PLANES);
    uint2 *raw_i = reinterpret_cast<uint2 *>(tsm + T::PLANES + T::RAW);
    uint64_t *bar = reinterpret_cast<uint64_t *>(tsm + T::PLANES + 2 * T::RAW);

    const int tx = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * PD + tx;

    // tile -> (x0, first row yb); the TMA box starts 2 S texels left of / 2 lattice rows above it
    auto tile_origin = [&](int tile, int &x0, int &yb) {
        const int bx = tile % q.n_tx, by = tile / q.n_tx;
        x0 = bx * (2 * PD);
        yb = p.y_begin + (by / S) * (S * LR) + (by % S);
    };
    auto issue = [&](int tile) {
        int x0, yb;
        tile_origin(tile, x0, yb);
        const int base = yb - 2 * S;                       // first staged row (may be negative)
        const int qrow = (base >= 0) ? base / S : -((-base + S - 1) / S);
        const int rrow = base - qrow * S;                  // 0 <= rrow < S: rows base + j S = (rrow, qrow + j)
        mbar_expect_tx(bar, (uint32_t)(2 * T::RAW));
        tma_load_3d(raw_n, &map_normals, x0 - 2 * S, rrow, qrow, bar);
        tma_load_3d(raw_i, &map_integ, x0 - 2 * S, rrow, qrow, bar);
    };

    if (tid == 0) {
        mbar_init(bar, 1);
        if ((int)blockIdx.x < q.n_tiles) issue(blockIdx.x);
    }
    __syncthreads();

    uint32_t parity = 0;
    for (int tile = blockIdx.x; tile < q.n_tiles; tile += gridDim.x) {
        mbar_wait(bar, parity);
        parity ^= 1u;
        // ---- convert the raw fp16 boxes into the fp32 pair planes (pixel a = texel j, pixel b = texel j + PD) ------
        for (int idx = tid; idx < SR * PC; idx += C::THREADS) {
            const int row = idx / PC, j = idx - row * PC;
            const uint2 *rn = raw_n + row * PCT + j, *ri = raw_i + row * PCT + j;
            const float4 na = unpack_rgba16f(rn[0]), nb = unpack_rgba16f(rn[PD]);
            const float4 va = unpack_rgba16f(ri[0]), vb = unpack_rgba16f(ri[PD]);
            const int ia = f2i_rz(na.w), ib = f2i_rz(nb.w);
            sN0[idx] = make_ulonglong2(pk(na.x, nb.x), pk(na.y, nb.y));
            sN1[idx] = make_ulonglong2(pk(na.z, nb.z), (u64)(uint32_t)ia | ((u64)(uint32_t)ib << 32));
            sL[idx] = make_ulonglong2(pk(va.x, vb.x), pk(va.y, vb.y));
            sV[idx] = make_ulonglong2(pk(va.z, vb.z), pk(va.w, vb.w));
        }
        __syncthreads();                                   // planes complete, raw boxes free
        if (tid == 0 && tile + (int)gridDim.x < q.n_tiles) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy reads of raw before the async-proxy overwrite
            issue(tile + gridDim.x);
        }
        int x0, yb;
        tile_origin(tile, x0, yb);
        pair_compute<S, PD, RY, TR>(p, sN0, sN1, sL, sV, x0, yb, tx, ty);
        __syncthreads();                                   // every tap read done before the next convert overwrites the planes
    }
}

template <int S, int PD, int RY, int TR>
static int launch_pair(vhr_context *ctx, const AtrousParams &p, int x_pixels, int y_pixels) {
    typedef PairCfg<S, PD, RY, TR> C;
    static_assert(C::SMEM <= 110 * 1024, "two CTAs per SM must fit in shared memory");
    static uint64_t configured = 0;     // bit d: done on device d (function attributes live in the device's context, not in the process)
    if (!(configured >> (ctx->device & 63) & 1ull)) {
        VHR_CUDA_CHECK(cudaFuncSetAttribute(atrous_pair_kernel<S, PD, RY, TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
        configured |= 1ull << (ctx->device & 63);
    }
    dim3 block(PD, TR);
    dim3 grid((x_pixels + 2 * PD - 1) / (2 * PD), ((y_pixels + S * C::LR - 1) / (S * C::LR)) * S);
    atrous_pair_kernel<S, PD, RY, TR><<<grid, block, C::SMEM, ctx->stream>>>(p);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode_tiled = nullptr;

// (x, row mod S, row div S) view of a dense RGBA16F image, box = {box_w texels, 1, box_rows}. The image allocation is
// padded by 16 rows of zeros (alloc_image), which is what the last partial slab (rows H .. ceil(H/S) S) reads.
static int make_tensor_map(CUtensorMap *map, const void *ptr, int width, int height, int S, int box_w, int box_rows) {
    if (!g_encode_tiled) {
        cudaDriverEntryPointQueryResult qres;
        void *fn = nullptr;
        VHR_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) return fail(VHR_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
        g_encode_tiled = (EncodeTiledFn)fn;
    }
    const cuuint64_t W = (cuuint64_t)width, H = (cuuint64_t)height;
    const cuuint64_t dims[3] = {W, (cuuint64_t)S, (H + S - 1) / S};
    const cuuint64_t strides[2] = {W * 8, W * 8 * (cuuint64_t)S};     // bytes, dims 1 and 2
    const cuuint32_t box[3] = {(cuuint32_t)box_w, 1u, (cuuint32_t)box_rows};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64 /* 8-byte elements: one texel */, 3, const_cast<void *>(ptr), dims, strides, box,
                                estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(VHR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a %dx%d image, step %d", (int)r, width, height, S);
    return VHR_OK;
}

template <int S, int PD, int RY, int TR>
static int launch_tma(vhr_context *ctx, const AtrousParams &p, int x_pixels, int y_pixels) {
    typedef PairCfg<S, PD, RY, TR> C;
    typedef TmaCfg<S, PD, RY, TR> T;
    static_assert(T::SMEM <= 112 * 1024, "two CTAs per SM must fit in shared memory");
    static uint64_t configured = 0;     // bit d: done on device d
    static int sms_of[64] = {};
    if (!(configured >> (ctx->device & 63) & 1ull)) {
        VHR_CUDA_CHECK(cudaFuncSetAttribute(atrous_tma_kernel<S, PD, RY, TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM));
        VHR_CUDA_CHECK(cudaDeviceGetAttribute(&sms_of[ctx->device & 63], cudaDevAttrMultiProcessorCount, ctx->device));
        configured |= 1ull << (ctx->device & 63);
    }
    const int sms = sms_of[ctx->device & 63];
    CUtensorMap map_n, map_i;
    if (int rc = make_tensor_map(&map_n, p.normals, p.W, p.H, S, T::PCT, C::SR)) return rc;
    if (int rc = make_tensor_map(&map_i, p.integ_in, p.W, p.H, S, T::PCT, C::SR)) return rc;
    AtrousTmaParams q;
    q.a = p;
    q.n_tx = (x_pixels + 2 * PD - 1) / (2 * PD);
    q.n_tiles = q.n_tx * ((y_pixels + S * C::LR - 1) / (S * C::LR)) * S;
    const int grid = std::min(q.n_tiles, 2 * sms);          // persistent: two resident CTAs per SM, tiles dealt round-robin
    atrous_tma_kernel<S, PD, RY, TR><<<grid, dim3(PD, TR), T::SMEM, ctx->stream>>>(q, map_n, map_i);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Launchers
// ---------------------------------------------------------------------------------------------------------------
static bool dispatch_range(vhr_context *ctx, const Image *ref, uint32_t xg, uint32_t yg, int &x_end, int &y0, int &y1) {
    x_end = (int)std::min<uint64_t>(ref->width, (uint64_t)xg * 8);
    int y_cov = (int)std::min<uint64_t>(ref->height, (uint64_t)yg * 8);
    y0 = std::max(0, ctx->opt.row_begin);
    y1 = ctx->opt.row_end < 0 ? y_cov : std::min(y_cov, ctx->opt.row_end);
    return x_end > 0 && y1 > y0;
}

static int check_image(const Image *im, int fmt, const Image *ref, const char *what) {
    if (!im || !im->ptr) return fail(VHR_ERR_INVALID, "%s: image not bound / unknown storage slot", what);
    if (im->format != fmt) return fail(VHR_ERR_INVALID, "%s: format %d, expected %d", what, im->format, fmt);
    if (ref && (im->width != ref->width || im->height != ref->height))
        return fail(VHR_ERR_INVALID, "%s: size %ux%u differs from %ux%u", what, im->width, im->height, ref->width, ref->height);
    return VHR_OK;
}

int launch_svgf_temporal(vhr_context *ctx, uint32_t xg, uint32_t yg, const SVGFPushConstants &pc) {
    // descriptor set 3 of the "SVGF Denoise Pass" (hybrid_render_path.cpp:264-272): 0 normals, 1 motion, 2 depth, 3 rt, 4 denoised
    if (ctx->n_bound < 4) return fail(VHR_ERR_STATE, "svgf.comp: pass images not bound (need bindings 0..3)");
    Image *normals = ctx->bound[0], *motion = ctx->bound[1], *rt = ctx->bound[3];
    Image *integ0 = storage_slot(ctx, pc.integrated_shadow_and_ao[0]);
    Image *prevn = storage_slot(ctx, pc.prev_frame_normals_and_object_ids);
    Image *hist = storage_slot(ctx, pc.shadow_and_ao_history);
    Image *mom = storage_slot(ctx, pc.shadow_and_ao_moments_history);
    int rc;
    if ((rc = check_image(normals, VHR_FORMAT_R16G16B16A16_SFLOAT, nullptr, "svgf.comp normals"))) return rc;
    if ((rc = check_image(motion, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "svgf.comp motion"))) return rc;
    if ((rc = check_image(rt, VHR_FORMAT_R16G16_SFLOAT, normals, "svgf.comp raytraced shadow/ao"))) return rc;
    if ((rc = check_image(integ0, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "svgf.comp integrated[0]"))) return rc;
    if ((rc = check_image(prevn, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "svgf.comp prev normals"))) return rc;
    if ((rc = check_image(hist, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "svgf.comp history"))) return rc;
    if ((rc = check_image(mom, VHR_FORMAT_R16G16_SFLOAT, normals, "svgf.comp moments"))) return rc;
    if (!mom->twin) {   // second moments buffer for the snapshot semantics (SURVEY Q11)
        VHR_CUDA_CHECK(cudaMalloc(&mom->twin, mom->bytes));
        VHR_CUDA_CHECK(cudaMemsetAsync(mom->twin, 0, mom->bytes, ctx->stream));
    }
    for (const Image *im : {prevn, hist, mom})
        if ((rc = resolve_read(ctx, im))) return rc;
    if ((rc = make_writable(ctx, integ0, covers_image(ctx, integ0, (uint64_t)xg * 8, (uint64_t)yg * 8)))) return rc;
    TemporalParams p;
    p.W = (int)normals->width; p.H = (int)normals->height;
    if (!dispatch_range(ctx, normals, xg, yg, p.x_end, p.y_begin, p.y_end)) return VHR_OK;
    p.dsx = ctx->pfd.display_size[0]; p.dsy = ctx->pfd.display_size[1];
    p.normals = (const uint2 *)normals->ptr; p.motion = (const uint2 *)motion->ptr; p.rt = (const uint32_t *)rt->ptr;
    p.prev_normals = (const uint2 *)prevn->ptr; p.history = (const uint2 *)hist->ptr;
    p.moments_in = (const uint32_t *)mom->ptr; p.integrated_out = (uint2 *)integ0->ptr; p.moments_out = (uint32_t *)mom->twin;
    // multi-GPU: iteration 0 on the neighbours reads 2 rows of this output beyond their band, their next temporal pass
    // reads `motion_halo` rows of these moments
    // Without the interleaved ray pass (ray_block_rows = 0) nothing orders this kernel's halo stores into the neighbours' integrated[0]
    // after THEIR last a-trous iteration of the previous frame, which still reads that image and exchanges nothing (SURVEY Q1): one
    // flag round trip first. With ray_block_rows = 8 the ray pass's all-ranks exchange already sits in between.
    if (ctx->part.enabled && ctx->part.world > 1 && ctx->part.ray_block_rows == 0)
        if ((rc = peer_sync_neighbours(ctx))) return rc;
    p.push_integ = halo_push_for(ctx, integ0, false, 2);
    p.push_mom = halo_push_for(ctx, mom, true, ctx->part.motion_halo);
    ctx->fused_it0.valid = false;
    Image *integ1 = storage_slot(ctx, pc.integrated_shadow_and_ao[1]);
    const bool full = covers_image(ctx, integ0, (uint64_t)xg * 8, (uint64_t)yg * 8);
    if (ctx->opt.svgf_fused && full && ctx->opt.atrous_variant >= 2 && integ1 && integ1 != integ0 && p.dsx == (float)p.W && p.dsy == (float)p.H &&
        !check_image(integ1, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "svgf.comp integrated[1]")) {
        // fused temporal + a-trous iteration 0 (step 1): the reference's next call, Dispatch(svgf_atrous_filter.comp) with atrous_step 1 on
        // the same slots, is then answered without a launch (launch_svgf_atrous)
        typedef PairCfg<1, 64, 2, 4> C;
        if ((rc = make_writable(ctx, integ1, true))) return rc;
        static uint64_t configured = 0;
        if (!(configured >> (ctx->device & 63) & 1ull)) {
            VHR_CUDA_CHECK(cudaFuncSetAttribute(svgf_fused_kernel<64, 2, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
            configured |= 1ull << (ctx->device & 63);
        }
        AtrousParams a;
        a.W = p.W; a.H = p.H; a.x_end = p.x_end; a.y_begin = p.y_begin; a.y_end = p.y_end; a.step = 1; a.dsx = p.dsx; a.dsy = p.dsy;
        a.normals = p.normals; a.integ_in = (const uint2 *)integ0->ptr; a.integ_out = (uint2 *)integ1->ptr;
        dim3 block(64, 4), grid((p.x_end + 127) / 128, (p.y_end - p.y_begin + C::LR - 1) / C::LR);
        svgf_fused_kernel<64, 2, 4><<<grid, block, C::SMEM, ctx->stream>>>(p, a);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->fused_it0.valid = true;
        ctx->fused_it0.in_slot = pc.integrated_shadow_and_ao[0];
        ctx->fused_it0.out_slot = pc.integrated_shadow_and_ao[1];
        ctx->fused_it0.epoch = ctx->epoch;
    } else {
        dim3 block(32, 8), grid((p.x_end + 31) / 32, (p.y_end - p.y_begin + 7) / 8);
        svgf_temporal_kernel<<<grid, block, 0, ctx->stream>>>(p);
        VHR_CUDA_CHECK(cudaGetLastError());
    }
    ctx->launches++;
    std::swap(mom->ptr, mom->twin);   // this frame's moments become "the" moments image
    for (int r = 0; r < VHR_MAX_RANKS; ++r) std::swap(mom->peer[r], mom->peer_twin[r]);
    return peer_sync_neighbours(ctx);
}

static int launch_direct(vhr_context *ctx, const AtrousParams &p, int x_pixels, int y_pixels) {
    dim3 block(32, 8), grid((x_pixels + 31) / 32, (y_pixels + 7) / 8);
    atrous_direct_kernel<<<grid, block, 0, ctx->stream>>>(p);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

// The kernel instance of a dispatch: variant, step, and whether the UBO's display size matches the images
static AtrousLauncher pick_launcher(const vhr_context *ctx, const AtrousParams &p) {
    // The tiled kernel bounds-checks against the image size; the reference checks against pfd.display_size. They are
    // the same thing whenever the UBO matches the images, which the tiled path requires.
    bool tiled_ok = ctx->opt.atrous_variant >= 1 && p.dsx == (float)p.W && p.dsy == (float)p.H;
    static const int dev_tr = getenv("VHR_ATROUS_TR") ? atoi(getenv("VHR_ATROUS_TR")) : 4;     // development A/B switch
    if (tiled_ok && ctx->opt.atrous_variant >= 2 && dev_tr == 3) {      // three rows per thread, 192-thread CTAs (168 registers): 22 % fewer shared-memory loads per tap
        switch (p.step) {
            case 1: return launch_pair<1, 64, 3, 3>;
            case 2: return launch_pair<2, 64, 3, 3>;
            case 4: return launch_pair<4, 64, 3, 3>;
            case 8: return launch_pair<8, 64, 3, 3>;
            default: break;
        }
    }
    if (tiled_ok && ctx->opt.atrous_variant >= 2 && dev_tr == 2) {
        switch (p.step) {
            case 1: return launch_pair<1, 64, 2, 2>;
            case 2: return launch_pair<2, 64, 2, 2>;
            case 4: return launch_pair<4, 64, 2, 2>;
            case 8: return launch_pair<8, 64, 2, 2>;
            case 16: return launch_pair<16, 64, 2, 2>;
            default: break;
        }
    }
    if (tiled_ok && ctx->opt.atrous_variant == 3 && (p.W % 2) == 0) {        // TMA needs 16-byte row strides
        switch (p.step) {
            case 1: return launch_tma<1, 64, 2, 4>;
            case 2: return launch_tma<2, 64, 2, 4>;
            case 4: return launch_tma<4, 64, 2, 4>;
            case 8: return launch_tma<8, 64, 2, 4>;
            default: break;   // step 16: the raw boxes no longer fit beside the planes twice per SM -> variant 2
        }
    }
    if (tiled_ok && ctx->opt.atrous_variant >= 2) {
        switch (p.step) {
            case 1: return launch_pair<1, 64, 2, 4>;
            case 2: return launch_pair<2, 64, 2, 4>;
            case 4: return launch_pair<4, 64, 2, 4>;
            case 8: return launch_pair<8, 64, 2, 4>;
            case 16: return launch_pair<16, 64, 2, 4>;
            default: break;   // other steps: direct kernel
        }
    } else if (tiled_ok) {
        switch (p.step) {
            case 1: return launch_tiled<1>;
            case 2: return launch_tiled<2>;
            case 4: return launch_tiled<4>;
            case 8: return launch_tiled<8>;
            case 16: return launch_tiled<16>;
            default: break;   // other steps: direct kernel
        }
    }
    return launch_direct;
}

static int atrous_launch_only(vhr_context *ctx, uint32_t xg, uint32_t yg, const SVGFPushConstants &pc, bool &pushed) {
    if (ctx->n_bound < 1) return fail(VHR_ERR_STATE, "svgf_atrous_filter.comp: pass images not bound");
    Image *normals = ctx->bound[0];
    Image *in = storage_slot(ctx, pc.integrated_shadow_and_ao[0]);
    Image *out = storage_slot(ctx, pc.integrated_shadow_and_ao[1]);
    int rc;
    if ((rc = check_image(normals, VHR_FORMAT_R16G16B16A16_SFLOAT, nullptr, "atrous normals"))) return rc;
    if ((rc = check_image(in, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "atrous integrated[0]"))) return rc;
    if ((rc = check_image(out, VHR_FORMAT_R16G16B16A16_SFLOAT, normals, "atrous integrated[1]"))) return rc;
    if (in == out) return fail(VHR_ERR_INVALID, "atrous: integrated[0] and [1] are the same image");
    if (pc.atrous_step < 1) return fail(VHR_ERR_INVALID, "atrous: step %d < 1", pc.atrous_step);
    if ((rc = resolve_read(ctx, in))) return rc;
    if ((rc = make_writable(ctx, out, covers_image(ctx, out, (uint64_t)xg * 8, (uint64_t)yg * 8)))) return rc;
    // one deferred dispatch at a time: an earlier one that this dispatch did not read or overwrite whole goes first
    if ((rc = launch_pending_atrous(ctx))) return rc;
    AtrousParams p;
    p.W = (int)normals->width; p.H = (int)normals->height;
    if (!dispatch_range(ctx, normals, xg, yg, p.x_end, p.y_begin, p.y_end)) return VHR_OK;
    p.step = pc.atrous_step;
    p.dsx = ctx->pfd.display_size[0]; p.dsy = ctx->pfd.display_size[1];
    p.normals = (const uint2 *)normals->ptr; p.integ_in = (const uint2 *)in->ptr; p.integ_out = (uint2 *)out->ptr;
    // multi-GPU: the next iteration (step 2s) reads 4s rows beyond a band; iteration 0's output is also next frame's
    // history (motion halo); the reference never reads the last iteration's output (SURVEY Q1), so it is not exchanged
    if (ctx->part.enabled && p.step != ctx->part.no_exchange_step)
        p.push = halo_push_for(ctx, out, false, p.step == 1 ? std::max(4, ctx->part.motion_halo) : 4 * p.step);
    pushed = p.push.rows > 0;
    const AtrousLauncher fn = pick_launcher(ctx, p);
    const int xp = p.x_end, yp = p.y_end - p.y_begin;
    // Deferred (PendingAtrous): the reference's last iteration writes an image that the next frame's iteration 0 overwrites unread
    // (SURVEY Q1), so that launch is dropped; every other iteration is launched by the one after it, which reads its output.
    if (ctx->part.enabled || ctx->opt.svgf_fused || ctx->queue[1]) return fn(ctx, p, xp, yp);
    PendingAtrous &d = ctx->atrous_pending;
    d.p = p; d.launch = fn; d.x_pixels = xp; d.y_pixels = yp; d.stream = ctx->stream;
    d.valid = true;
    return VHR_OK;
}

int launch_pending_atrous(vhr_context *ctx) {
    PendingAtrous &d = ctx->atrous_pending;
    if (!d.valid) return VHR_OK;
    d.valid = false;
    VHR_CUDA_CHECK(cudaSetDevice(ctx->device));       // resolved from entry points that do not select the device themselves
    cudaStream_t cur = ctx->stream;
    ctx->stream = d.stream;
    const int rc = d.launch(ctx, d.p, d.x_pixels, d.y_pixels);
    ctx->stream = cur;
    return rc;
}

int resolve_read(vhr_context *ctx, const Image *im) {
    const PendingAtrous &d = ctx->atrous_pending;
    return d.valid && im && im->ptr == d.p.integ_out ? launch_pending_atrous(ctx) : VHR_OK;
}

static bool recorded(const PendingAtrous &d, const void *buf) {
    return buf && (buf == d.p.integ_out || buf == d.p.integ_in || buf == d.p.normals);
}

int resolve_touch(vhr_context *ctx, const Image *im) {
    const PendingAtrous &d = ctx->atrous_pending;
    return d.valid && im && recorded(d, im->ptr) ? launch_pending_atrous(ctx) : VHR_OK;
}

int resolve_free(vhr_context *ctx, const Image *im) {
    PendingAtrous &d = ctx->atrous_pending;
    if (d.valid && im && im->ptr == d.p.integ_out) {
        d.valid = false;
        return VHR_OK;
    }
    return resolve_touch(ctx, im);
}

int resolve_write(vhr_context *ctx, const void *buf, bool whole) {
    PendingAtrous &d = ctx->atrous_pending;
    if (!d.valid || !recorded(d, buf)) return VHR_OK;
    if (whole && buf == d.p.integ_out) {
        d.valid = false;
        return VHR_OK;
    }
    return launch_pending_atrous(ctx);
}

int launch_svgf_atrous(vhr_context *ctx, uint32_t xg, uint32_t yg, const SVGFPushConstants &pc) {
    if (ctx->fused_it0.valid) {       // iteration 0 came out of the fused svgf.comp kernel one call ago: nothing left to launch
        const bool same = ctx->fused_it0.epoch + 1 == ctx->epoch && pc.atrous_step == 1 && pc.integrated_shadow_and_ao[0] == ctx->fused_it0.in_slot &&
                          pc.integrated_shadow_and_ao[1] == ctx->fused_it0.out_slot;
        ctx->fused_it0.valid = false;
        if (same) return VHR_OK;
    }
    bool pushed = false;
    if (int rc = atrous_launch_only(ctx, xg, yg, pc, pushed)) return rc;
    return pushed ? peer_sync_neighbours(ctx) : VHR_OK;
}

}  // namespace vhr
