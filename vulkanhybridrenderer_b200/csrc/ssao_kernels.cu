// ssao_kernels.cu — Alchemy screen-space ambient occlusion and its 13x13 box blur (sm_100a).
//
//   ssao_kernel       <- /root/reference/data/shaders/hybrid_render_path/ssao.comp:14-53
//   ssao_blur_kernel  <- /root/reference/data/shaders/hybrid_render_path/ssao_blur.comp:11-26
//
// `texture()` through the reference's default sampler (resource_manager.cpp:58-69: LINEAR, REPEAT) is evaluated in
// software with the Vulkan spec's float weights — CUDA texture units filter with 8-bit fixed-point weights, which
// would not match the CPU oracle (SURVEY Q16).
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "vhr_internal.h"

namespace vhr {

struct SsaoParams {
    int W, H;
    int x_end, y_begin, y_end;
    float radius;
    float Wf, Hf;             // (float)W, (float)H
    const float4 *quads;      // (d[y][x], d[y][x+1], d[y+1][x], d[y+1][x+1]) per texel, REPEAT-wrapped (depth_quads_kernel); or nullptr
    const uint2 *normals;     // binding 0 (RGBA16F, sampled)
    const float *depth;       // binding 1 (D32F, sampled)
    uint2 *out;               // binding 2 (RGBA16F)
    HaloPush push;            // multi-GPU: the blur on the neighbours reads 6 rows of this output beyond their band
};

__device__ __forceinline__ void ssao_store(const SsaoParams &p, int gy, size_t pix, uint2 v) {
    p.out[pix] = v;
    if (p.push.rows) {
        if (p.push.up && gy < p.y_begin + p.push.rows) reinterpret_cast<uint2 *>(p.push.up)[pix] = v;
        if (p.push.down && gy >= p.y_end - p.push.rows) reinterpret_cast<uint2 *>(p.push.down)[pix] = v;
    }
}

__device__ __forceinline__ float sample_depth(const SsaoParams &p, float u, float v) {
    int x0, x1, y0, y1;
    float a, b;
    bilinear_setup(u, p.W, x0, x1, a);
    bilinear_setup(v, p.H, y0, y1, b);
    float t00 = __ldg(&p.depth[(size_t)y0 * p.W + x0]), t10 = __ldg(&p.depth[(size_t)y0 * p.W + x1]);
    float t01 = __ldg(&p.depth[(size_t)y1 * p.W + x0]), t11 = __ldg(&p.depth[(size_t)y1 * p.W + x1]);
    return bilerp_rn(a, b, t00, t10, t01, t11);
}

// get_view_space_position (glsl_common.h:111-116) for the 16 SAMPLES of a pixel. With PERSPECTIVE (the inverse projection has the
// sparsity of an inverse perspective matrix: only m00, m11, m23, m32, m33 non-zero — checked on the host) the products of the
// matrix-vector product that multiply exact zeros are not issued: glm's pairwise sum (c0 x + c1 y) + (c2 z + c3 w) with zero terms IS the
// remaining term, so the values are the oracle's. FAST (study switch): one MUFU reciprocal and three products instead of the three IEEE
// divisions by w.
template <bool PERSPECTIVE, bool FAST>
__device__ __forceinline__ float3 unproject_sample(const float *inv, float depth, float u, float v) {
    const float x = fmaf(u, 2.0f, -1.0f), y = fmaf(v, 2.0f, -1.0f);      // = fl(fl(2 u) - 1): the doubling is exact
    float4 q;
    if (PERSPECTIVE) {
        q = make_float4(mul_rn(inv[0], x), mul_rn(inv[5], y), inv[14], add_rn(mul_rn(inv[11], depth), inv[15]));
    } else {
        q = mul44_rn(inv, make_float4(x, y, depth, 1.0f));
    }
    if (FAST) {
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(q.w));
        return make_float3(q.x * r, q.y * r, q.z * r);
    }
    const ExactDivisor dw = exact_divisor(q.w);       // the three IEEE quotients (vhr_common.cuh)
    return make_float3(div_exact(q.x, dw), div_exact(q.y, dw), div_exact(q.z, dw));
}
__device__ __noinline__ float occlusion_term_library(float4 q, float3 P, float3 N) {
    const float3 Q = make_float3(__fdiv_rn(q.x, q.w), __fdiv_rn(q.y, q.w), __fdiv_rn(q.z, q.w));
    const float3 V = make_float3(sub_rn(Q.x, P.x), sub_rn(Q.y, P.y), sub_rn(Q.z, P.z));
    return __fdiv_rn(fmaxf(sub_rn(dot3_rn(V, N), 1e-4f), 0.0f), add_rn(dot3_rn(V, V), 1e-4f));
}
// One sample's occlusion term max(dot(V, N) - beta, 0) / (dot(V, V) + 1e-4), V = view-space sample - P (ssao.comp:42-44), in the oracle's
// operations. The four IEEE divisions share two refined reciprocals and ONE fall-back branch (div_exact_flag). BOUNDED (PERSPECTIVE only):
// the caller vouches for the three dividends of the unprojection — the host has checked |m00|, |m11| in [2^-14, 2^8] and |m23| in
// [2^-38, 2^38], and the sample went through the fixed-point tap path (|u n| < 2^14), so x = 2u - 1 is zero or in [2^-24, 2^15] — and
// their range tests are not issued.
template <bool PERSPECTIVE, bool BOUNDED>
__device__ __forceinline__ float occlusion_term(const float *inv, float depth, float u, float v, float3 P, float3 N) {
    const float x = fmaf(u, 2.0f, -1.0f), y = fmaf(v, 2.0f, -1.0f);      // = fl(fl(2 u) - 1): the doubling is exact
    float4 q;
    if (PERSPECTIVE) q = make_float4(mul_rn(inv[0], x), mul_rn(inv[5], y), inv[14], add_rn(mul_rn(inv[11], depth), inv[15]));
    else q = mul44_rn(inv, make_float4(x, y, depth, 1.0f));
    bool rare = false;
    const ExactDivisor dw = exact_divisor(q.w);
    const float3 Q = (PERSPECTIVE && BOUNDED)
                         ? make_float3(div_exact_flag_bounded(q.x, dw, rare), div_exact_flag_bounded(q.y, dw, rare), div_exact_flag_bounded(q.z, dw, rare))
                         : make_float3(div_exact_flag(q.x, dw, rare), div_exact_flag(q.y, dw, rare), div_exact_flag(q.z, dw, rare));
    const float3 V = make_float3(sub_rn(Q.x, P.x), sub_rn(Q.y, P.y), sub_rn(Q.z, P.z));
    // fmaxf returns the non-NaN operand, like the GLSL max() on NVIDIA hardware the oracle restates
    const float num = fmaxf(sub_rn(dot3_rn(V, N), 1e-4f), 0.0f);
    const float den = add_rn(dot3_rn(V, V), 1e-4f);
    float term = div_exact_flag(num, exact_divisor(den), rare);
    if (rare) term = occlusion_term_library(q, P, N);       // a finite operand outside 2^+-40
    return term;
}
struct SsaoParams;
__device__ __noinline__ float occlusion_term_general_tap(const SsaoParams &p, const float *inv, float u, float v, float3 P, float3 N);

// texture(depth, (u, v)).x of a SAMPLE, in two halves so that the loads of several samples are in flight together.
// tap_setup: the tap selection and the two filter weights, exactly the oracle's (bilinear_setup): with t = fl(fl(u n) - 0.5) the snapped
// coordinate floor(t 256 + 0.5) / 256 is the integer k = floor(fma(t, 256, 0.5)) (the product by 256 is exact and for |t| < 2^14 so is
// the sum), texel = k >> 8, weight = (k & 255) / 256 — one F2I instead of two FRND + F2I + the float fraction. Returns the texel index
// y0 W + x0, or -1 for anything unusual (texel outside the image, |t| >= 2^14, NaN): those samples take the general path.
// The four taps then come as ONE 16-byte load from the quad image (QUADS) — a gather at 32 unrelated places costs the L1 about two
// cycles per 128-byte line and load instruction (tools/probes/probe_tld4.cu: 33 M footprints in 114 us as quads, 238 us as four 4-byte
// loads, 121 us as texture gathers), and it is this, not the arithmetic, that bounds the kernel once the instructions are cut.
struct Tap { int idx; float a, b; };
template <bool QUADS>
__device__ __forceinline__ Tap tap_setup(const SsaoParams &p, float u, float v) {
    Tap t;
    t.idx = -1; t.a = 0.0f; t.b = 0.0f;
    const float tu = sub_rn(mul_rn(u, p.Wf), 0.5f), tv = sub_rn(mul_rn(v, p.Hf), 0.5f);
    if (fabsf(tu) < 16384.0f && fabsf(tv) < 16384.0f) {
        const int ku = __float2int_rd(fmaf(tu, 256.0f, 0.5f)), kv = __float2int_rd(fmaf(tv, 256.0f, 0.5f));
        int x0 = ku >> 8, y0 = kv >> 8;
        // the quad image has the REPEAT wrap of the right / bottom neighbour built in; without it both taps must be inside.
        // One period of REPEAT is applied here (QUADS): the samples of a pixel within a radius of the image border fall outside by the
        // dozen, and the general path for one lane is paid by the whole warp (ncu: 197 executed instructions per sample against
        // ~125 in the listing before this was added)
        if (QUADS) {
            x0 += x0 < 0 ? p.W : 0; x0 -= x0 >= p.W ? p.W : 0;
            y0 += y0 < 0 ? p.H : 0; y0 -= y0 >= p.H ? p.H : 0;
        }
        if ((unsigned)x0 < (unsigned)(p.W - (QUADS ? 0 : 1)) && (unsigned)y0 < (unsigned)(p.H - (QUADS ? 0 : 1))) {
            // (2^23 + m) / 256 - 2^15 = m / 256 exactly: the weight without an integer-to-float conversion
            t.a = fmaf(__uint_as_float(0x4B000000u | (uint32_t)(ku & 255)), 0.00390625f, -32768.0f);
            t.b = fmaf(__uint_as_float(0x4B000000u | (uint32_t)(kv & 255)), 0.00390625f, -32768.0f);
            t.idx = y0 * p.W + x0;
        }
    }
    return t;
}
template <bool QUADS>
__device__ __forceinline__ float4 tap_load(const SsaoParams &p, const Tap &t) {
    const int i = t.idx < 0 ? 0 : t.idx;       // a sample on the general path loads texel 0 and ignores it
    if (QUADS) return __ldg(p.quads + i);
    const float *r0 = p.depth + i;
    return make_float4(__ldg(r0), __ldg(r0 + 1), __ldg(r0 + p.W), __ldg(r0 + p.W + 1));
}
// (kept out of line: taken by the few taps on the REPEAT seam; inlined copies would triple the unrolled sample loop)
__device__ __noinline__ float sample_depth_general(const SsaoParams &p, float u, float v) { return sample_depth(p, u, v); }
// a sample off the fixed-point tap path (|u n| >= 2^14, NaN): general tap, general matrix product (same values as the sparse form), every
// range test
__device__ __noinline__ float occlusion_term_general_tap(const SsaoParams &p, const float *inv, float u, float v, float3 P, float3 N) {
    return occlusion_term<false, false>(inv, sample_depth(p, u, v), u, v, P, N);
}

// Pre-pass of the SSAO dispatch: the bilinear footprint of every depth texel as one float4 (8 MB read, 33 MB written at 1080p)
__global__ void __launch_bounds__(256) depth_quads_kernel(const float *__restrict__ depth, float4 *__restrict__ quads, int W, int H) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= W || y >= H) return;
    const int x1 = x + 1 == W ? 0 : x + 1, y1 = y + 1 == H ? 0 : y + 1;
    const float *r0 = depth + (size_t)y * W, *r1 = depth + (size_t)y1 * W;
    quads[(size_t)y * W + x] = make_float4(__ldg(r0 + x), __ldg(r0 + x1), __ldg(r1 + x), __ldg(r1 + x1));
}

// sin and cos of an angle in [0, 2 pi] (ssao.comp:38: random01 * 2 * PI): quadrant by the 1.5 * 2^23 rounding constant, two-term
// Cody-Waite reduction to |f| <= pi / 4, degree-7 / degree-8 minimax polynomials (the single-precision cephes coefficients). Within one
// ulp of the correctly rounded value on all 2^23 angles the RNG can produce (tests/test_oracle_cpu.py restates it in numpy), at a third
// of sincosf's instructions — and NOT the default (study switch VHR_SSAO_VARIANT bit 2): it differs from the C library's correctly
// rounded value on 12-17 % of the angles where sincosf almost never does, which moves 1e-5 of the samples across a 1/256 filter step:
// 0.05-0.13 % of the pixels of the small test images beyond the 1e-3 bar (measured), against 0.002 % with sincosf.
__device__ __forceinline__ void sincos_turn(float x, float &s, float &c) {
    const float m = fmaf(x, 0.636619772f, 12582912.0f);
    const uint32_t q = __float_as_uint(m);
    const float qf = m - 12582912.0f;
    float f = fmaf(qf, -1.57079637f, x);
    f = fmaf(qf, 4.37113883e-8f, f);
    const float f2 = f * f;
    float sp = fmaf(f2, -1.9515295891e-4f, 8.3321608736e-3f);
    sp = fmaf(sp, f2, -1.6666654611e-1f);
    const float sn = fmaf(f * f2, sp, f);
    float cp = fmaf(f2, 2.443315711809948e-5f, -1.388731625493765e-3f);
    cp = fmaf(cp, f2, 4.166664568298827e-2f);
    cp = fmaf(cp, f2, -0.5f);
    const float cs = fmaf(cp, f2, 1.0f);
    const bool odd = (q & 1u) != 0u;
    s = __uint_as_float(__float_as_uint(odd ? cs : sn) ^ ((q << 30) & 0x80000000u));
    c = __uint_as_float(__float_as_uint(odd ? sn : cs) ^ (((q + 1u) << 30) & 0x80000000u));
}

// VARIANT (study switch VHR_SSAO_VARIANT): 0 = default: fixed-point filter coordinate, the four taps of a sample as one load from the
// quad image, four samples' loads in flight, everything else in the oracle's operations and order (same bits as the loop of rounds 1-2,
// 255 -> ~160 instructions per sample); bit 0 = that older loop; bit 1 = four 4-byte tap loads instead of the quad image; bit 2 =
// sincos_turn instead of sincosf; bit 3 = the continuous part (interpolation, division by w, occlusion term) on fused / approximate
// operations — ~110 instructions per sample, but Q - P cancels eight digits for a sample next to the pixel, so one ulp of Q moves
// that sample's term by up to 1e-2: 0.05-0.13 % of the pixels of the small test images beyond the 1e-3 bar (PSNR 80 dB; measured).
template <bool PERSPECTIVE, int VARIANT>
__global__ void __launch_bounds__(256) ssao_kernel(const __grid_constant__ SsaoParams p, const __grid_constant__ PerFrameData pfd) {
    const int gx = blockIdx.x * 32 + threadIdx.x;
    const int gy = p.y_begin + blockIdx.y * 8 + threadIdx.y;
    if (gx >= p.x_end || gy >= p.y_end) return;
    const size_t pix = (size_t)gy * p.W + gx;
    const float cu = mul_rn((float)gx, pfd.display_size_inverse[0]);
    const float cv = mul_rn((float)gy, pfd.display_size_inverse[1]);
    float current_depth = sample_depth(p, cu, cv);
    if (current_depth == 0.0f) {
        ssao_store(p, gy, pix, make_uint2(0u, 0u));
        return;
    }
    float3 P = unproject_rn(pfd.camera_proj_inverse, current_depth, cu, cv);
    float3 nw;
    {
        int x0, x1, y0, y1;
        float a, b;
        bilinear_setup(cu, p.W, x0, x1, a);
        bilinear_setup(cv, p.H, y0, y1, b);
        float4 t00 = unpack_rgba16f(__ldg(&p.normals[(size_t)y0 * p.W + x0]));
        float4 t10 = unpack_rgba16f(__ldg(&p.normals[(size_t)y0 * p.W + x1]));
        float4 t01 = unpack_rgba16f(__ldg(&p.normals[(size_t)y1 * p.W + x0]));
        float4 t11 = unpack_rgba16f(__ldg(&p.normals[(size_t)y1 * p.W + x1]));
        nw = make_float3(bilerp_rn(a, b, t00.x, t10.x, t01.x, t11.x), bilerp_rn(a, b, t00.y, t10.y, t01.y, t11.y),
                         bilerp_rn(a, b, t00.z, t10.z, t01.z, t11.z));
    }
    float3 N = mul33_of44_rn(pfd.camera_view, nw);
    float perspective_radius = __fdiv_rn(p.radius, P.z);
    uint32_t rng = seed_thread(((uint32_t)gy * (uint32_t)pfd.display_size[1] + (uint32_t)gx) * pfd.frame_index);
    float sum = 0.0f;
    if (VARIANT & 1) {
        for (int i = 0; i < 16; ++i) {
            float ang = mul_rn(mul_rn(random01(rng), 2.0f), VHR_PI);
            float dist = mul_rn(random01(rng), perspective_radius);
            float s, c;
            sincosf(ang, &s, &c);
            float su = add_rn(cu, mul_rn(c, dist)), sv = add_rn(cv, mul_rn(s, dist));
            float3 Q = unproject_sample<PERSPECTIVE, false>(pfd.camera_proj_inverse, sample_depth(p, su, sv), su, sv);
            float3 V = make_float3(sub_rn(Q.x, P.x), sub_rn(Q.y, P.y), sub_rn(Q.z, P.z));
            // fmaxf returns the non-NaN operand, like the GLSL max() on NVIDIA hardware the oracle restates
            float num = fmaxf(sub_rn(dot3_rn(V, N), 1e-4f), 0.0f);
            sum = add_rn(sum, __fdiv_rn(num, add_rn(dot3_rn(V, V), 1e-4f)));
        }
    } else {
        constexpr bool QUADS = !(VARIANT & 2), FAST = (VARIANT & 8) != 0;
        constexpr int G = (VARIANT & 16) ? 4 : 1;  // samples whose taps are loaded together (bit 4: four; the kernel is issue-bound, it does not pay)
#pragma unroll(G == 1 ? 4 : 1)
        for (int i = 0; i < 16; i += G) {
            float su[G], sv[G];
            Tap tap[G];
            float4 q[G];
#pragma unroll
            for (int j = 0; j < G; ++j) {
                // fl(fl(r * 2) * PI) = fl(r * (2 PI)): the doubling is exact
                const float ang = mul_rn(random01(rng), 2.0f * VHR_PI);
                const float dist = mul_rn(random01(rng), perspective_radius);
                float s, c;
                if (VARIANT & 4) sincos_turn(ang, s, c);
                else sincosf(ang, &s, &c);
                su[j] = add_rn(cu, mul_rn(c, dist)); sv[j] = add_rn(cv, mul_rn(s, dist));
                tap[j] = tap_setup<QUADS>(p, su[j], sv[j]);
                q[j] = tap_load<QUADS>(p, tap[j]);
            }
#pragma unroll
            for (int j = 0; j < G; ++j) {
                if (FAST) {
                    float d;
                    if (tap[j].idx < 0) d = sample_depth_general(p, su[j], sv[j]);
                    else {
                        const float top = fmaf(tap[j].a, q[j].y - q[j].x, q[j].x), bot = fmaf(tap[j].a, q[j].w - q[j].z, q[j].z);
                        d = fmaf(tap[j].b, bot - top, top);
                    }
                    const float3 Q = unproject_sample<PERSPECTIVE, true>(pfd.camera_proj_inverse, d, su[j], sv[j]);
                    const float3 V = make_float3(Q.x - P.x, Q.y - P.y, Q.z - P.z);
                    const float num = fmaxf(fmaf(V.x, N.x, fmaf(V.y, N.y, fmaf(V.z, N.z, -1e-4f))), 0.0f);
                    float r;
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaf(V.x, V.x, fmaf(V.y, V.y, fmaf(V.z, V.z, 1e-4f)))));
                    sum = fmaf(num, r, sum);
                } else if (tap[j].idx < 0) {
                    sum = add_rn(sum, occlusion_term_general_tap(p, pfd.camera_proj_inverse, su[j], sv[j], P, N));
                } else {
                    const float d = bilerp_rn(tap[j].a, tap[j].b, q[j].x, q[j].y, q[j].z, q[j].w);
                    sum = add_rn(sum, occlusion_term<PERSPECTIVE, true>(pfd.camera_proj_inverse, d, su[j], sv[j], P, N));
                }
            }
        }
    }
    float ao = fmaxf(sub_rn(1.0f, mul_rn(0.125f, sum)), 0.0f);
    ssao_store(p, gy, pix, pack_rgba16f(make_float4(ao, ao, ao, ao)));
}

// 13x13 box sum of .x, OOB skipped, always divided by 169 (ssao_blur.comp:11-26): horizontal 13-sums, then vertical 13-sums, each summed
// left to right / top to bottom.
struct BlurParams {
    int W, H;
    int x_end, y_begin, y_end;
    const uint2 *in;
    uint2 *out;
};

// Default: a 64 x 32-pixel tile per 256-thread block (a 6-texel apron costs 1.63x the tile instead of the 3.4x of the first kernel's 32 x 8
// tile), register blocking in both passes: a thread forms four adjacent horizontal sums from sixteen values fetched as four 16-byte
// shared-memory loads, and eight vertically adjacent outputs from twenty horizontal sums. Every sum adds its thirteen terms in the same
// order as the first kernel (VHR_SSAO_BLUR_VARIANT=1), so the images are bit-identical to it.
__global__ void __launch_bounds__(256) ssao_blur_tile_kernel(const __grid_constant__ BlurParams p) {
    constexpr int TX = 64, TY = 32, R = 6, RW = TX + 2 * R, RH = TY + 2 * R;      // raw tile 76 x 44
    __shared__ __align__(16) float raw[RH][RW];
    __shared__ __align__(16) float hsum[RH][TX];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * TX, y0 = p.y_begin + blockIdx.y * TY;
    for (int idx = tid; idx < RH * RW; idx += 256) {
        const int row = idx / RW, col = idx - row * RW;
        const int gx = x0 - R + col, gy = y0 - R + row;
        float v = 0.0f;
        if (gx >= 0 && gx < p.W && gy >= 0 && gy < p.H)
            v = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.in[(size_t)gy * p.W + gx]))).x;
        raw[row][col] = v;
    }
    __syncthreads();
    for (int gi = tid; gi < RH * (TX / 4); gi += 256) {
        const int row = gi >> 4, c0 = (gi & 15) * 4;
        float v[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 t = *reinterpret_cast<const float4 *>(&raw[row][c0 + 4 * q]);
            v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
        }
        float h[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float sum = 0.0f;
#pragma unroll
            for (int k = 0; k < 2 * R + 1; ++k) sum += v[j + k];
            h[j] = sum;
        }
        *reinterpret_cast<float4 *>(&hsum[row][c0]) = make_float4(h[0], h[1], h[2], h[3]);
    }
    __syncthreads();
    const int c = tid & 63, r0 = (tid >> 6) * 8;
    const int cx = x0 + c;
    float hv[8 + 2 * R];
#pragma unroll
    for (int k = 0; k < 8 + 2 * R; ++k) hv[k] = hsum[r0 + k][c];
    if (cx >= p.x_end) return;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int cy = y0 + r0 + i;
        if (cy >= p.y_end) break;
        float sum = 0.0f;
#pragma unroll
        for (int k = 0; k < 2 * R + 1; ++k) sum += hv[i + k];
        const float o = __fdiv_rn(sum, 169.0f);
        p.out[(size_t)cy * p.W + cx] = pack_rgba16f(make_float4(o, o, o, o));
    }
}

// The first kernel (VHR_SSAO_BLUR_VARIANT=1): 32 x 8 outputs per block, one output per thread.
__global__ void __launch_bounds__(256) ssao_blur_kernel(const __grid_constant__ BlurParams p) {
    constexpr int TX = 32, TY = 8, R = 6;
    __shared__ float raw[TY + 2 * R][TX + 2 * R + 1];
    __shared__ float hsum[TY + 2 * R][TX];
    const int tid = threadIdx.y * TX + threadIdx.x;
    const int x0 = blockIdx.x * TX, y0 = p.y_begin + blockIdx.y * TY;
    for (int idx = tid; idx < (TY + 2 * R) * (TX + 2 * R); idx += TX * TY) {
        int row = idx / (TX + 2 * R), col = idx - row * (TX + 2 * R);
        int gx = x0 - R + col, gy = y0 - R + row;
        float v = 0.0f;
        if (gx >= 0 && gx < p.W && gy >= 0 && gy < p.H)
            v = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.in[(size_t)gy * p.W + gx]))).x;
        raw[row][col] = v;
    }
    __syncthreads();
    for (int idx = tid; idx < (TY + 2 * R) * TX; idx += TX * TY) {
        int row = idx / TX, col = idx - row * TX;
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < 2 * R + 1; ++k) s += raw[row][col + k];
        hsum[row][col] = s;
    }
    __syncthreads();
    const int cx = x0 + threadIdx.x, cy = y0 + threadIdx.y;
    if (cx >= p.x_end || cy >= p.y_end) return;
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < 2 * R + 1; ++k) s += hsum[threadIdx.y + k][threadIdx.x];
    float o = __fdiv_rn(s, 169.0f);
    p.out[(size_t)cy * p.W + cx] = pack_rgba16f(make_float4(o, o, o, o));
}

static bool dispatch_range(vhr_context *ctx, const Image *ref, uint32_t xg, uint32_t yg, int &x_end, int &y0, int &y1) {
    x_end = (int)std::min<uint64_t>(ref->width, (uint64_t)xg * 8);
    int y_cov = (int)std::min<uint64_t>(ref->height, (uint64_t)yg * 8);
    y0 = std::max(0, ctx->opt.row_begin);
    y1 = ctx->opt.row_end < 0 ? y_cov : std::min(y_cov, ctx->opt.row_end);
    return x_end > 0 && y1 > y0;
}

// The quad image of a depth image (screen-space passes: ssao.comp, ssr.comp), rebuilt by every dispatch that gathers from it.
int build_depth_quads(vhr_context *ctx, const float *depth, int W, int H, const float4 **quads) {
    const int q = ctx->stream == ctx->queue[1] && ctx->queue[1] != nullptr ? 1 : 0;       // the selected queue's own buffer
    const size_t texels = (size_t)W * H;
    if (ctx->depth_quads_texels[q] < texels) {
        if (ctx->d_depth_quads[q]) { VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->d_depth_quads[q]); ctx->d_depth_quads[q] = nullptr; }
        VHR_CUDA_CHECK(cudaMalloc(&ctx->d_depth_quads[q], texels * sizeof(float4)));
        ctx->depth_quads_texels[q] = texels;
    }
    depth_quads_kernel<<<dim3((W + 31) / 32, (H + 7) / 8), dim3(32, 8), 0, ctx->stream>>>(depth, ctx->d_depth_quads[q], W, H);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    *quads = ctx->d_depth_quads[q];
    return VHR_OK;
}

int launch_ssao(vhr_context *ctx, uint32_t xg, uint32_t yg, float radius) {
    // descriptor set 3 of the "SSAO Pass" (hybrid_render_path.cpp:143-150): 0 normals, 1 depth, 2 raw output
    if (ctx->n_bound < 3) return fail(VHR_ERR_STATE, "ssao.comp: pass images not bound (need bindings 0..2)");
    Image *normals = ctx->bound[0], *depth = ctx->bound[1], *out = ctx->bound[2];
    if (!normals || !depth || !out) return fail(VHR_ERR_STATE, "ssao.comp: unbound image");
    if (normals->format != VHR_FORMAT_R16G16B16A16_SFLOAT || depth->format != VHR_FORMAT_D32_SFLOAT ||
        out->format != VHR_FORMAT_R16G16B16A16_SFLOAT)
        return fail(VHR_ERR_INVALID, "ssao.comp: unexpected image formats");
    if (depth->width != normals->width || depth->height != normals->height || out->width != normals->width ||
        out->height != normals->height)
        return fail(VHR_ERR_INVALID, "ssao.comp: image sizes differ");
    if (int rc = make_writable(ctx, out, covers_image(ctx, out, (uint64_t)xg * 8, (uint64_t)yg * 8))) return rc;
    SsaoParams p;
    p.W = (int)normals->width; p.H = (int)normals->height;
    if (!dispatch_range(ctx, normals, xg, yg, p.x_end, p.y_begin, p.y_end)) return VHR_OK;
    p.radius = radius;
    p.Wf = (float)p.W; p.Hf = (float)p.H;
    p.normals = (const uint2 *)normals->ptr; p.depth = (const float *)depth->ptr; p.out = (uint2 *)out->ptr;
    // multi-GPU (row bands; every rank holds the full depth / normal G-buffer the samples reach into): the 13x13 blur on the
    // neighbours reads 6 rows of this output beyond their band -> pushed by this kernel, then the flag-word round trip
    p.push = halo_push_for(ctx, out, false, 6);
    if (p.push.rows && ((p.push.up == nullptr && ctx->part.rank > 0) || (p.push.down == nullptr && ctx->part.rank + 1 < ctx->part.world)))
        return fail(VHR_ERR_STATE, "ssao.comp: the neighbours' '%s' image is not attached (vhr_image_attach_peer)", "Screen Space Ambient Occlusion Raw");
    dim3 block(32, 8), grid((p.x_end + 31) / 32, (p.y_end - p.y_begin + 7) / 8);
    // inverse perspective sparsity (column-major m[c * 4 + r]): everything but m00, m11, m23 (index 11), m32 (index 14), m33 (index 15) is zero
    bool perspective = true;
    for (int i = 0; i < 16; ++i)
        if (i != 0 && i != 5 && i != 11 && i != 14 && i != 15 && ctx->pfd.camera_proj_inverse[i] != 0.0f) perspective = false;
    // ... and its coefficients in the range occlusion_term<.., BOUNDED> relies on (any real camera: m00, m11 = tan(fov / 2) terms, m23 = -1);
    // m00 and m11 positive, so that a zero dividend m00 x or m11 y is +0 (div_exact_flag_bounded's precondition: x = fl(2 u - 1) is never -0)
    {
        const float *m = ctx->pfd.camera_proj_inverse;
        const float a0 = m[0], a5 = m[5], a14 = std::fabs(m[14]);
        if (!(a0 >= 6.1035156e-5f && a0 <= 256.0f && a5 >= 6.1035156e-5f && a5 <= 256.0f && a14 >= 3.6379788e-12f && a14 <= 2.7487791e11f)) perspective = false;
    }
    static const int variant = [] { const char *e = getenv("VHR_SSAO_VARIANT"); return e ? atoi(e) : 0; }();
    p.quads = nullptr;
    if (!(variant & 1) && !(variant & 2)) {
        // the samples of a row band reach any row of the depth image: the whole quad image on every rank
        if (int rc = build_depth_quads(ctx, p.depth, p.W, p.H, &p.quads)) return rc;
    }
#define VHR_SSAO_CASE(V) case V: if (perspective) ssao_kernel<true, V><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); \
                                 else ssao_kernel<false, V><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;
    switch (variant) {
        VHR_SSAO_CASE(0) VHR_SSAO_CASE(1) VHR_SSAO_CASE(2) VHR_SSAO_CASE(4) VHR_SSAO_CASE(8) VHR_SSAO_CASE(12) VHR_SSAO_CASE(16) VHR_SSAO_CASE(24)
        default: return fail(VHR_ERR_INVALID, "VHR_SSAO_VARIANT = %d (0, 1, 2, 4, 8, 12, 16 or 24)", variant);
    }
#undef VHR_SSAO_CASE
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return p.push.rows ? peer_sync_neighbours(ctx) : VHR_OK;
}

int launch_ssao_blur(vhr_context *ctx, uint32_t xg, uint32_t yg) {
    // "SSAO Blur Pass" (hybrid_render_path.cpp:170-177): 0 raw, 1 blurred
    if (ctx->n_bound < 2) return fail(VHR_ERR_STATE, "ssao_blur.comp: pass images not bound (need bindings 0..1)");
    Image *in = ctx->bound[0], *out = ctx->bound[1];
    if (!in || !out) return fail(VHR_ERR_STATE, "ssao_blur.comp: unbound image");
    if (in->format != VHR_FORMAT_R16G16B16A16_SFLOAT || out->format != VHR_FORMAT_R16G16B16A16_SFLOAT)
        return fail(VHR_ERR_INVALID, "ssao_blur.comp: unexpected image formats");
    if (in->width != out->width || in->height != out->height) return fail(VHR_ERR_INVALID, "ssao_blur.comp: image sizes differ");
    if (ctx->pfd.display_size[0] != (float)in->width || ctx->pfd.display_size[1] != (float)in->height)
        return fail(VHR_ERR_INVALID, "ssao_blur.comp: PerFrameData.display_size does not match the images");
    if (int rc = make_writable(ctx, out, covers_image(ctx, out, (uint64_t)xg * 8, (uint64_t)yg * 8))) return rc;
    BlurParams p;
    p.W = (int)in->width; p.H = (int)in->height;
    if (!dispatch_range(ctx, in, xg, yg, p.x_end, p.y_begin, p.y_end)) return VHR_OK;
    p.in = (const uint2 *)in->ptr; p.out = (uint2 *)out->ptr;
    static const int variant = [] { const char *e = getenv("VHR_SSAO_BLUR_VARIANT"); return e ? atoi(e) : 0; }();
    if (variant == 1) {
        dim3 block(32, 8), grid((p.x_end + 31) / 32, (p.y_end - p.y_begin + 7) / 8);
        ssao_blur_kernel<<<grid, block, 0, ctx->stream>>>(p);
    } else {
        ssao_blur_tile_kernel<<<dim3((p.x_end + 63) / 64, (p.y_end - p.y_begin + 31) / 32), 256, 0, ctx->stream>>>(p);
    }
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

}  // namespace vhr
