// composition_kernels.cu — the hybrid path's composition pass as a CUDA kernel (sm_100a).
//
//   composition_kernel <- /root/reference/data/shaders/hybrid_render_path/composition.frag:60-161 drawn as the
//                         full-screen triangle of composition.vert ("Composition Pass",
//                         /root/reference/src/render_paths/hybrid_render_path.cpp:333-379)
//
// Consumer of the ray-traced / denoised images: per pixel it rebuilds the world position, evaluates the Cook-Torrance
// terms of common.glsl:116-150 with the shadow, AO and reflection images selected by the three specialisation
// constants and writes RENDER_OUTPUT. One thread per pixel, every input texel read exactly once (texture() at a pixel
// centre through a LINEAR sampler returns the texel itself, SURVEY Q17) — a pure streaming kernel, HBM-bound.
// Output formats: B8G8R8A8_SRGB (the reference's swapchain, vulkan_context.cpp:331: linear -> sRGB encode on store),
// B8G8R8A8_UNORM (no encode) or R16G16B16A16_SFLOAT (linear HDR, what the parity tests compare). NaN stores as 0, like
// the float -> UNORM conversion of the reference's attachment write (sky pixels: the unprojection divides by w = 0).
//
// Gathered output (VHR_OPT_OUTPUT_RANK under a partition): the <GATHER = true> instances store every texel of the rank's band a second
// time, with the same bits, into the output rank's RENDER_OUTPUT over NVLink, so that rank ends with the whole frame. The <false>
// instances are the single-GPU kernels; the output rank itself runs them too.
#include <algorithm>
#include <type_traits>

#include "vhr_internal.h"

namespace vhr {

struct CompositionParams {
    int W, H;
    int y_begin, y_end;
    int shadow_mode, ao_mode, reflection_mode;     // common.glsl:12-25
    int out_format;
    int rt_is_rg16;                                // binding 7: 1 = raw RG16F image, 0 = denoised RGBA16F image
    int shadow_w, shadow_h;
    const uint32_t *albedo;        // binding 0  BGRA8
    const uint2 *normals;          // binding 1
    const uint2 *motion;           // binding 2 (.zw = metallic, roughness)
    const float *depth;            // binding 3
    const float *shadow_map;       // binding 4
    const uint2 *ssao;             // binding 5
    const uint2 *ssr;              // binding 6
    const void *rt;                // binding 7
    const uint2 *refl;             // binding 8
    void *out;                     // attachment 0
};
struct CompositionGatherParams : CompositionParams {
    void *out_gather;              // the output rank's render output
};

// Divisions, square roots and the sRGB power run on the MUFU unit (rcp / rsq / lg2 / ex2, <= 2 ulp) instead of the IEEE
// sequences: the first version of this kernel spent ~85 us at 1080p on ~25 exact divisions and three powf() per pixel
// (14 % of the HBM rate it is bound by). The results stay inside the parity bar (1e-3 on linear radiance, one code on
// the 8-bit outputs); products and sums keep the oracle's evaluation order.
__device__ __forceinline__ float fdiv(float a, float b) { return __fdividef(a, b); }
__device__ __forceinline__ float3 normalize_fast(float3 a) {
    const float r = rsqrtf(dot3_rn(a, a));
    return make_float3(mul_rn(a.x, r), mul_rn(a.y, r), mul_rn(a.z, r));
}
__device__ __forceinline__ float srgb_encode(float c) {
    // NaN -> 0, clamp to [0, 1] (Vulkan float -> UNORM conversion), then the sRGB OETF
    c = (c == c) ? fminf(fmaxf(c, 0.0f), 1.0f) : 0.0f;
    return c <= 0.0031308f ? 12.92f * c : fmaf(1.055f, exp2f(__log2f(c) * (1.0f / 2.4f)), -0.055f);
}
__device__ __forceinline__ uint32_t unorm8_rn(float c) {
    c = (c == c) ? fminf(fmaxf(c, 0.0f), 1.0f) : 0.0f;
    return (uint32_t)__float2int_rn(c * 255.0f);
}
__device__ __forceinline__ float mixc_rn(float a, float b, float t) { return add_rn(mul_rn(a, sub_rn(1.0f, t)), mul_rn(b, t)); }

__device__ __forceinline__ float sample_shadow_map(const CompositionParams &p, float u, float v) {
    int x0, x1, y0, y1;
    float a, b;
    bilinear_setup(u, p.shadow_w, x0, x1, a);
    bilinear_setup(v, p.shadow_h, y0, y1, b);
    const float *d = p.shadow_map;
    const size_t W = (size_t)p.shadow_w;
    return bilerp_rn(a, b, __ldg(&d[y0 * W + x0]), __ldg(&d[y0 * W + x1]), __ldg(&d[y1 * W + x0]), __ldg(&d[y1 * W + x1]));
}

// The three modes are template parameters, the CUDA counterpart of the reference's specialisation constants
// (composition.frag:6-8, hybrid_render_path.cpp:361-369): each of the 27 pipelines carries only the loads and the
// arithmetic of its own mode.
template <int SHADOW_MODE, int AO_MODE, int REFLECTION_MODE, bool GATHER>
__global__ void __launch_bounds__(256) composition_kernel(const __grid_constant__ std::conditional_t<GATHER, CompositionGatherParams, CompositionParams> p,
                                                          const __grid_constant__ PerFrameData pfd) {
    const int x = blockIdx.x * 64 + threadIdx.x;        // blockDim = (64, 4): 512-byte rows of 8-byte texels per warp pair
    const int y = p.y_begin + blockIdx.y * 4 + threadIdx.y;
    if (x >= p.W || y >= p.y_end) return;
    const size_t pix = (size_t)y * p.W + x;
    // in_uv of the full-screen triangle at the pixel centre
    const float u = fdiv(add_rn((float)x, 0.5f), (float)p.W), v = fdiv(add_rn((float)y, 0.5f), (float)p.H);

    const uint32_t a8 = __ldg(&p.albedo[pix]);          // B8G8R8A8: byte 0 = B
    const float3 albedo = make_float3(fdiv((float)((a8 >> 16) & 0xffu), 255.0f), fdiv((float)((a8 >> 8) & 0xffu), 255.0f),
                                      fdiv((float)(a8 & 0xffu), 255.0f));
    const float depth = __ldg(&p.depth[pix]);
    float3 P;
    {
        const float4 q = mul44_rn(pfd.camera_viewproj_inverse, make_float4(sub_rn(mul_rn(u, 2.0f), 1.0f), sub_rn(mul_rn(v, 2.0f), 1.0f), depth, 1.0f));
        const float rw = fdiv(1.0f, q.w);
        P = make_float3(mul_rn(q.x, rw), mul_rn(q.y, rw), mul_rn(q.z, rw));
    }
    const float4 n4 = unpack_rgba16f(__ldg(&p.normals[pix]));
    const float3 N = make_float3(n4.x, n4.y, n4.z);
    const float2 mr = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.motion[pix]) + 1));   // .zw

    float2 rt = make_float2(1.0f, 1.0f);
    if (SHADOW_MODE == 0 || AO_MODE == 0)
        rt = p.rt_is_rg16 ? unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(p.rt) + pix))
                          : unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(reinterpret_cast<const uint2 *>(p.rt) + pix)));

    const float3 cam = make_float3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
    const float3 V = normalize_fast(make_float3(sub_rn(cam.x, P.x), sub_rn(cam.y, P.y), sub_rn(cam.z, P.z)));
    const float3 L = make_float3(-pfd.directional_light.direction[0], -pfd.directional_light.direction[1], -pfd.directional_light.direction[2]);
    const float3 H = normalize_fast(make_float3(add_rn(L.x, V.x), add_rn(L.y, V.y), add_rn(L.z, V.z)));

    float shadow = 1.0f;
    if (SHADOW_MODE == 0) {
        shadow = rt.x;
    } else if (SHADOW_MODE == 1) {
        // composition.frag:81-104: SHADOW_BIAS_MATRIX * projview * P, 4x4 PCF on the 4096^2 shadow map
        const float4 lp = mul44_rn(pfd.directional_light.projview, make_float4(P.x, P.y, P.z, 1.0f));
        const float4 ls = make_float4(add_rn(mul_rn(0.5f, lp.x), mul_rn(0.5f, lp.w)), add_rn(mul_rn(0.5f, lp.y), mul_rn(0.5f, lp.w)), lp.z, lp.w);
        const float sx = fdiv(ls.x, ls.w), sy = fdiv(ls.y, ls.w), sz = fdiv(ls.z, ls.w);
        const float scale = 1.0f / 4096.0f;
        float acc = 0.0f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const float ox = -1.5f + (float)(i >> 2), oy = -1.5f + (float)(i & 3);
            const float ds = sample_shadow_map(p, add_rn(sx, mul_rn(ox, scale)), add_rn(sy, mul_rn(oy, scale)));
            acc = add_rn(acc, (sz < sub_rn(ds, 1e-4f)) ? 0.0f : 1.0f);
        }
        shadow = fdiv(acc, 16.0f);
    }
    float ao = 1.0f;
    if (AO_MODE == 0) ao = rt.y;
    else if (AO_MODE == 1) ao = unpack_rg16f(__ldg(reinterpret_cast<const uint32_t *>(&p.ssao[pix]))).x;

    const float metallic = fminf(fmaxf(mr.x, 0.0f), 1.0f);
    const float roughness = fminf(fmaxf(mr.y, 0.04f), 1.0f);
    const float *li = pfd.directional_light.intensity, *lc = pfd.directional_light.color;

    const float3 f0 = make_float3(mixc_rn(0.04f, albedo.x, metallic), mixc_rn(0.04f, albedo.y, metallic), mixc_rn(0.04f, albedo.z, metallic));
    // fresnel_schlick (common.glsl:116-119), left to right
    const float hv = fmaxf(dot3_rn(H, V), 0.0f);
    const float o = sub_rn(1.0f, hv);
    auto fres = [&](float f) { return add_rn(f, mul_rn(mul_rn(mul_rn(mul_rn(mul_rn(sub_rn(1.0f, f), o), o), o), o), o)); };
    const float3 F = make_float3(fres(f0.x), fres(f0.y), fres(f0.z));
    const float ndl = fmaxf(dot3_rn(N, L), 0.0f);

    // diffuse_brdf (common.glsl:146-150)
    const float sdm = sub_rn(1.0f, metallic);
    const float3 dbrdf = make_float3(fdiv(mul_rn(mul_rn(sub_rn(1.0f, F.x), sdm), albedo.x), VHR_PI),
                                     fdiv(mul_rn(mul_rn(sub_rn(1.0f, F.y), sdm), albedo.y), VHR_PI),
                                     fdiv(mul_rn(mul_rn(sub_rn(1.0f, F.z), sdm), albedo.z), VHR_PI));
    // specular_brdf (common.glsl:121-144)
    const float a2 = mul_rn(roughness, roughness);
    const float nh = fmaxf(dot3_rn(N, H), 0.0f);
    const float ff = add_rn(mul_rn(mul_rn(nh, nh), sub_rn(a2, 1.0f)), 1.0f);
    const float D = fdiv(a2, mul_rn(mul_rn(VHR_PI, ff), ff));
    const float kk = mul_rn(mul_rn(add_rn(roughness, 1.0f), add_rn(roughness, 1.0f)), 0.125f);
    const float nv = fmaxf(dot3_rn(N, V), 0.0f);
    const float g_nvk = fdiv(nv, add_rn(mul_rn(nv, sub_rn(1.0f, kk)), kk));
    const float g_nlk = fdiv(ndl, add_rn(mul_rn(ndl, sub_rn(1.0f, kk)), kk));
    const float dg = mul_rn(D, mul_rn(g_nvk, g_nlk));
    const float denom = fmaxf(mul_rn(mul_rn(4.0f, nv), ndl), 1e-6f);
    const float3 sbrdf = make_float3(fdiv(mul_rn(dg, F.x), denom), fdiv(mul_rn(dg, F.y), denom), fdiv(mul_rn(dg, F.z), denom));

    // brdf * N_dot_L * light_intensity * light_color * shadow, left to right (composition.frag:136-137)
    auto lit = [&](float brdf, int c) { return mul_rn(mul_rn(mul_rn(mul_rn(brdf, ndl), li[c]), lc[c]), shadow); };
    const float3 ambient = make_float3(mul_rn(mul_rn(ao, albedo.x), VHR_PI_INVERSE), mul_rn(mul_rn(ao, albedo.y), VHR_PI_INVERSE),
                                       mul_rn(mul_rn(ao, albedo.z), VHR_PI_INVERSE));
    const float3 diffuse = make_float3(lit(dbrdf.x, 0), lit(dbrdf.y, 1), lit(dbrdf.z, 2));
    float3 specular = make_float3(lit(sbrdf.x, 0), lit(sbrdf.y, 1), lit(sbrdf.z, 2));

    if (REFLECTION_MODE == 0 || REFLECTION_MODE == 1) {     // composition.frag:139-156 (ray traced / SSR: same blend)
        const float4 r4 = unpack_rgba16f(__ldg(REFLECTION_MODE == 0 ? &p.refl[pix] : &p.ssr[pix]));
        const float3 refl = make_float3(mul_rn(r4.x, shadow), mul_rn(r4.y, shadow), mul_rn(r4.z, shadow));
        if (metallic == 1.0f) specular = refl;
        else specular = make_float3(mixc_rn(specular.x, refl.x, roughness), mixc_rn(specular.y, refl.y, roughness), mixc_rn(specular.z, refl.z, roughness));
    }
    float3 lighting = make_float3(add_rn(add_rn(ambient.x, diffuse.x), specular.x), add_rn(add_rn(ambient.y, diffuse.y), specular.y),
                                  add_rn(add_rn(ambient.z, diffuse.z), specular.z));

    if (p.out_format == VHR_FORMAT_R16G16B16A16_SFLOAT) {
        lighting.x = (lighting.x == lighting.x) ? lighting.x : 0.0f;
        lighting.y = (lighting.y == lighting.y) ? lighting.y : 0.0f;
        lighting.z = (lighting.z == lighting.z) ? lighting.z : 0.0f;
        const uint2 c = pack_rgba16f(make_float4(lighting.x, lighting.y, lighting.z, 1.0f));
        reinterpret_cast<uint2 *>(p.out)[pix] = c;
        if constexpr (GATHER) reinterpret_cast<uint2 *>(p.out_gather)[pix] = c;
    } else {
        float r = lighting.x, g = lighting.y, b = lighting.z;
        if (p.out_format == VHR_FORMAT_B8G8R8A8_SRGB) { r = srgb_encode(r); g = srgb_encode(g); b = srgb_encode(b); }
        const uint32_t c = unorm8_rn(b) | (unorm8_rn(g) << 8) | (unorm8_rn(r) << 16) | 0xff000000u;
        reinterpret_cast<uint32_t *>(p.out)[pix] = c;
        if constexpr (GATHER) reinterpret_cast<uint32_t *>(p.out_gather)[pix] = c;
    }
}

// raytraced_render_path/composition.frag:11-13 drawn as the full-screen triangle of composition.vert: out_color = texture(raytraced_output,
// in_uv) at the pixel centre = the texel, stored to RENDER_OUTPUT (sRGB-encoded when the attachment is B8G8R8A8_SRGB; alpha stays linear).
struct PresentParams {
    int W, H, y_begin, y_end, out_format;
    const uint32_t *in;      // binding 0: RaytracedOutput, B8G8R8A8_UNORM
    void *out;
};
struct PresentGatherParams : PresentParams {
    void *out_gather;        // the output rank's render output
};
template <bool GATHER>
__global__ void __launch_bounds__(256) present_kernel(const __grid_constant__ std::conditional_t<GATHER, PresentGatherParams, PresentParams> p) {
    const int x = blockIdx.x * 64 + threadIdx.x, y = p.y_begin + blockIdx.y * 4 + threadIdx.y;
    if (x >= p.W || y >= p.y_end) return;
    const size_t pix = (size_t)y * p.W + x;
    const uint32_t c = __ldg(&p.in[pix]);
    if (p.out_format == VHR_FORMAT_B8G8R8A8_UNORM) {
        reinterpret_cast<uint32_t *>(p.out)[pix] = c;
        if constexpr (GATHER) reinterpret_cast<uint32_t *>(p.out_gather)[pix] = c;
        return;
    }
    const float b = fdiv((float)(c & 0xffu), 255.0f), g = fdiv((float)((c >> 8) & 0xffu), 255.0f), r = fdiv((float)((c >> 16) & 0xffu), 255.0f);
    if (p.out_format == VHR_FORMAT_R16G16B16A16_SFLOAT) {
        const uint2 h = pack_rgba16f(make_float4(r, g, b, fdiv((float)(c >> 24), 255.0f)));
        reinterpret_cast<uint2 *>(p.out)[pix] = h;
        if constexpr (GATHER) reinterpret_cast<uint2 *>(p.out_gather)[pix] = h;
        return;
    }
    const uint32_t e = unorm8_rn(srgb_encode(b)) | (unorm8_rn(srgb_encode(g)) << 8) | (unorm8_rn(srgb_encode(r)) << 16) | (c & 0xff000000u);
    reinterpret_cast<uint32_t *>(p.out)[pix] = e;
    if constexpr (GATHER) reinterpret_cast<uint32_t *>(p.out_gather)[pix] = e;
}

// VHR_OPT_OUTPUT_RANK (include/vhr_b200.h): `gather` = this draw gathers the frame on the output rank; `peer_out` = where this rank's
// texels go a second time (nullptr on the output rank itself, which only receives). Every failure comes before anything is enqueued,
// so a rank that fails leaves no flag written and no stream waiting.
static int gather_target(vhr_context *ctx, Image *out, const char *what, bool &gather, void *&peer_out) {
    const Partition &pt = ctx->part;
    const int p = ctx->opt.output_rank;
    gather = pt.enabled && pt.world > 1 && p >= 0;
    peer_out = nullptr;
    if (!gather) return VHR_OK;
    if (p >= pt.world) return fail(VHR_ERR_INVALID, "%s: VHR_OPT_OUTPUT_RANK %d is not a rank of the partition (world %d)", what, p, pt.world);
    if (p == pt.rank) return VHR_OK;
    peer_out = out->peer[p];
    if (!peer_out)
        return fail(VHR_ERR_STATE, "%s: the render output (%s) has no image of rank %d attached (vhr_image_attach_peer)", what,
                    image_label(ctx, out).c_str(), p);
    return VHR_OK;
}

// Load both instances a gathering draw may launch before its leading flag wait is enqueued: with lazy module loading a first launch
// would otherwise wait for this stream, which then waits for the other ranks — a deadlock when they are contexts driven by this same
// thread and have not issued their signals yet. `slot` tells the 27 mode combinations and present_kernel (27) apart.
template <typename K0, typename K1>
static int load_pair(vhr_context *ctx, int slot, K0 k0, K1 k1) {
    static uint64_t loaded[28] = {};
    if (loaded[slot] >> (ctx->device & 63) & 1ull) return VHR_OK;
    cudaFuncAttributes attr;
    VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, k0));
    VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, k1));
    loaded[slot] |= 1ull << (ctx->device & 63);
    return VHR_OK;
}

int launch_present(vhr_context *ctx) {
    // "Composition Pass" of the ray-traced path (raytraced_render_path.cpp:49-76): 0 RaytracedOutput (sampled), colour attachment 0 at index 1
    if (ctx->n_bound < 2 || !ctx->bound[0] || !ctx->bound[1]) return fail(VHR_ERR_STATE, "raytraced composition: images not bound (RaytracedOutput + the render output)");
    Image *in = ctx->bound[0], *out = ctx->bound[1];
    if (in->format != VHR_FORMAT_B8G8R8A8_UNORM) return fail(VHR_ERR_INVALID, "raytraced composition: binding 0 has format %d", in->format);
    if (out->format != VHR_FORMAT_B8G8R8A8_SRGB && out->format != VHR_FORMAT_B8G8R8A8_UNORM && out->format != VHR_FORMAT_R16G16B16A16_SFLOAT)
        return fail(VHR_ERR_INVALID, "raytraced composition: render output format %d", out->format);
    if (in->width != out->width || in->height != out->height) return fail(VHR_ERR_INVALID, "raytraced composition: image sizes differ");
    bool gather;
    void *peer_out;
    if (int rc = gather_target(ctx, out, "raytraced composition", gather, peer_out)) return rc;
    if (gather)
        if (int rc = load_pair(ctx, 27, present_kernel<false>, present_kernel<true>)) return rc;
    if (int rc = make_writable(ctx, out, covers_image(ctx, out, out->width, out->height))) return rc;
    PresentGatherParams p;      // its PresentParams part is all the <false> instance takes
    p.W = (int)out->width; p.H = (int)out->height;
    p.y_begin = std::max(0, ctx->opt.row_begin);
    p.y_end = ctx->opt.row_end < 0 ? p.H : std::min(p.H, ctx->opt.row_end);
    if (p.y_end <= p.y_begin && !gather) return VHR_OK;
    p.out_format = out->format; p.in = (const uint32_t *)in->ptr; p.out = out->ptr; p.out_gather = peer_out;
    // gathering: the output rank may still read the previous frame's output (nothing else orders that on this path)
    if (gather)
        if (int rc = peer_sync_all(ctx)) return rc;
    if (p.y_end > p.y_begin) {
        dim3 block(64, 4), grid((p.W + 63) / 64, (p.y_end - p.y_begin + 3) / 4);
        if (peer_out) present_kernel<true><<<grid, block, 0, ctx->stream>>>(p);
        else present_kernel<false><<<grid, block, 0, ctx->stream>>>(p);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
    }
    return gather ? peer_sync_all(ctx) : VHR_OK;      // every rank's rows have landed before anything on the output rank reads them
}

int launch_composition(vhr_context *ctx, int shadow_mode, int ao_mode, int reflection_mode) {
    // descriptor set 3 of the "Composition Pass" (hybrid_render_path.cpp:335-349): 0 albedo, 1 normals, 2 motion, 3 depth,
    // 4 shadow map, 5 SSAO, 6 SSR, 7 (denoised) shadow+AO, 8 reflections; colour attachment 0 follows at index 9
    if (ctx->n_bound < 10) return fail(VHR_ERR_STATE, "composition: pass images not bound (9 sampled images + the render output)");
    Image **b = ctx->bound;
    const int want[9] = {VHR_FORMAT_B8G8R8A8_UNORM, VHR_FORMAT_R16G16B16A16_SFLOAT, VHR_FORMAT_R16G16B16A16_SFLOAT, VHR_FORMAT_D32_SFLOAT,
                         VHR_FORMAT_D32_SFLOAT, VHR_FORMAT_R16G16B16A16_SFLOAT, VHR_FORMAT_R16G16B16A16_SFLOAT, 0, VHR_FORMAT_R16G16B16A16_SFLOAT};
    Image *out = b[9];
    for (int i = 0; i < 9; ++i) {
        if (i == 7) {
            if (b[7]->format != VHR_FORMAT_R16G16B16A16_SFLOAT && b[7]->format != VHR_FORMAT_R16G16_SFLOAT)
                return fail(VHR_ERR_INVALID, "composition: binding 7 has format %d", b[7]->format);
        } else if (b[i]->format != want[i]) {
            return fail(VHR_ERR_INVALID, "composition: binding %d has format %d, expected %d", i, b[i]->format, want[i]);
        }
        if (i != 4 && (b[i]->width != out->width || b[i]->height != out->height))
            return fail(VHR_ERR_INVALID, "composition: binding %d is %ux%u, render output is %ux%u", i, b[i]->width, b[i]->height, out->width, out->height);
    }
    if (out->format != VHR_FORMAT_B8G8R8A8_SRGB && out->format != VHR_FORMAT_B8G8R8A8_UNORM && out->format != VHR_FORMAT_R16G16B16A16_SFLOAT)
        return fail(VHR_ERR_INVALID, "composition: render output format %d", out->format);
    if (shadow_mode < 0 || shadow_mode > 2 || ao_mode < 0 || ao_mode > 2 || reflection_mode < 0 || reflection_mode > 2)
        return fail(VHR_ERR_INVALID, "composition: specialisation constants (%d, %d, %d)", shadow_mode, ao_mode, reflection_mode);
    bool gather;
    void *peer_out;
    if (int rc = gather_target(ctx, out, "composition", gather, peer_out)) return rc;
    typedef void (*Kernel)(const CompositionParams, const PerFrameData);
    typedef void (*GatherKernel)(const CompositionGatherParams, const PerFrameData);
#define VHR_COMP_ROW(S, A, G) {composition_kernel<S, A, 0, G>, composition_kernel<S, A, 1, G>, composition_kernel<S, A, 2, G>}
#define VHR_COMP_TABLE(G) {{VHR_COMP_ROW(0, 0, G), VHR_COMP_ROW(0, 1, G), VHR_COMP_ROW(0, 2, G)}, \
                           {VHR_COMP_ROW(1, 0, G), VHR_COMP_ROW(1, 1, G), VHR_COMP_ROW(1, 2, G)}, \
                           {VHR_COMP_ROW(2, 0, G), VHR_COMP_ROW(2, 1, G), VHR_COMP_ROW(2, 2, G)}}
    static const Kernel table[3][3][3] = VHR_COMP_TABLE(false);
    static const GatherKernel gather_table[3][3][3] = VHR_COMP_TABLE(true);
#undef VHR_COMP_TABLE
#undef VHR_COMP_ROW
    const Kernel single = table[shadow_mode][ao_mode][reflection_mode];
    const GatherKernel both = gather_table[shadow_mode][ao_mode][reflection_mode];
    if (gather)
        if (int rc = load_pair(ctx, (shadow_mode * 3 + ao_mode) * 3 + reflection_mode, single, both)) return rc;
    if (int rc = make_writable(ctx, out, covers_image(ctx, out, out->width, out->height))) return rc;
    CompositionGatherParams p;      // its CompositionParams part is all the <false> instances take
    p.W = (int)out->width; p.H = (int)out->height;
    p.y_begin = std::max(0, ctx->opt.row_begin);
    p.y_end = ctx->opt.row_end < 0 ? p.H : std::min(p.H, ctx->opt.row_end);
    if (p.y_end <= p.y_begin && !gather) return VHR_OK;
    p.shadow_mode = shadow_mode; p.ao_mode = ao_mode; p.reflection_mode = reflection_mode;
    p.out_format = out->format;
    p.rt_is_rg16 = b[7]->format == VHR_FORMAT_R16G16_SFLOAT;
    p.shadow_w = (int)b[4]->width; p.shadow_h = (int)b[4]->height;
    p.albedo = (const uint32_t *)b[0]->ptr; p.normals = (const uint2 *)b[1]->ptr; p.motion = (const uint2 *)b[2]->ptr;
    p.depth = (const float *)b[3]->ptr; p.shadow_map = (const float *)b[4]->ptr; p.ssao = (const uint2 *)b[5]->ptr;
    p.ssr = (const uint2 *)b[6]->ptr; p.rt = b[7]->ptr; p.refl = (const uint2 *)b[8]->ptr; p.out = out->ptr;
    p.out_gather = peer_out;
    // gathering: the output rank may still read the previous frame's output, and no earlier pass of this frame need have waited for it
    if (gather)
        if (int rc = peer_sync_all(ctx)) return rc;
    if (p.y_end > p.y_begin) {
        dim3 block(64, 4), grid((p.W + 63) / 64, (p.y_end - p.y_begin + 3) / 4);
        if (peer_out) both<<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
        else single<<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
    }
    return gather ? peer_sync_all(ctx) : VHR_OK;      // every rank's rows have landed before anything on the output rank reads them
}

}  // namespace vhr
