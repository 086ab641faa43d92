// oracle/oracle_rt.cpp — TEST INFRASTRUCTURE ONLY. CPU restatement of the ray-traced passes.
// Parity unpinned (see oracle_common.h). Citations relative to /root/reference.
//
//   vo_scene_create   <- src/rendering_backend/resource_manager.cpp:291-360,593-718 (UpdateGeometry / UpdateBLAS /
//                        UpdateTLAS: one world-space, opaque, two-sided triangle soup; geometry index = flat
//                        primitive index; indices relative to vertex_offset; per-geometry 3x4 transform)
//   vo_raygen         <- data/shaders/hybrid_render_path/raygen.rgen:14-66 (+ miss.rmiss:6-8,
//                        reflection_miss.rmiss:6-8, reflection_hit.rchit:10-72)
//   vo_gbuffer        <- data/shaders/hybrid_render_path/gbuf.vert:19-28, gbuf.frag:17-59 and the clear values
//                        of hybrid_render_path.cpp:16-19 (scaffolding: primary rays stand in for the rasteriser)
//   vo_shade_hits     <- the per-hit code of the passes above and of vo_raytraced on hits the caller gives (tests)
//
// The reference's BVH build, traversal and ray/triangle test live inside the Vulkan driver
// (vkCmdBuildAccelerationStructuresKHR / traceRayEXT — third-party, unversioned; SURVEY §8c). They are
// restated here from the Vulkan ray-tracing semantics: any triangle of the soup with tMin < t < tMax counts,
// no culling, shared edges watertight. The stand-in is a binned-SAH BVH2 with a double-precision watertight
// (Woop/Benthin/Wald 2013) ray/triangle test, i.e. effectively exact for float inputs.
#include "oracle_common.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <climits>
#include <cstring>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

using namespace vo;

namespace {

struct Node {            // 32 B
    float bmin[3];
    uint32_t left_first; // inner: index of left child (right = left+1); leaf: first triangle
    float bmax[3];
    uint32_t count;      // 0 = inner
};

struct Scene {
    std::vector<Vertex> vertices;
    std::vector<uint32_t> indices;
    std::vector<Primitive> primitives;
    std::vector<float> tri;          // 9 floats per triangle, world space, BVH leaf order
    std::vector<uint32_t> tri_geom;  // flat primitive index (gl_GeometryIndexEXT)
    std::vector<uint32_t> tri_prim;  // triangle index inside the primitive (gl_PrimitiveID)
    std::vector<Node> nodes;
    uint32_t n_tris = 0;
    // textures[] (glsl_common.h:104): ResourceManager::UploadTextureFromData (resource_manager.cpp:152-193) with the
    // glTF sampler (GetSampler :880-910); index = slot the materials name (glsl_common.h:82-91)
    struct Texture {
        uint32_t w = 0, h = 0;
        std::vector<uint8_t> rgba;
        bool srgb = false;            // VK_FORMAT_R8G8B8A8_SRGB (base colour, scene_loader.cpp:249-252)
        int mag = 1, min = 1;         // VkFilter: 0 NEAREST, 1 LINEAR
        int wrap_u = 0, wrap_v = 0;   // VkSamplerAddressMode: 0 REPEAT, 1 MIRRORED_REPEAT, 2 CLAMP_TO_EDGE, 3 CLAMP_TO_BORDER
    };
    std::vector<Texture> textures;
};

// ---- texture(textures[i], uv) -------------------------------------------------------------------------------------
// Vulkan spec, "Texel Coordinate Systems": ray-tracing stages have no implicit derivatives and the images have one mip
// level, so the lookup is LOD 0 with the mag filter; unnormalised coordinate u * size, LINEAR taps floor(u - 0.5) and
// +1 with weight fract(u - 0.5), NEAREST tap floor(u); wrapping per address mode; border = opaque black
// (resource_manager.cpp:67,902). sRGB texels are decoded to linear BEFORE filtering (Khronos Data Format spec 13.3.1).
inline int wrap_texel(int i, int n, int mode) {
    auto mod = [](int a, int b) { int m = a % b; return m < 0 ? m + b : m; };
    switch (mode) {
        case 0: return mod(i, n);
        case 1: { int m = mod(i, 2 * n) - n; m = m >= 0 ? m : -(1 + m); return (n - 1) - m; }
        case 2: return std::min(std::max(i, 0), n - 1);
        default: return (i < 0 || i >= n) ? -1 : i;
    }
}
inline float srgb_to_linear(uint8_t c) {
    double e = (double)c / 255.0;
    return (float)(e <= 0.04045 ? e / 12.92 : std::pow((e + 0.055) / 1.055, 2.4));
}
inline vec4 fetch_texel(const Scene::Texture &t, int x, int y) {
    if (x < 0 || y < 0) return vec4{0.0f, 0.0f, 0.0f, 1.0f};
    const uint8_t *c = &t.rgba[((size_t)y * t.w + x) * 4];
    if (t.srgb) return vec4{srgb_to_linear(c[0]), srgb_to_linear(c[1]), srgb_to_linear(c[2]), (float)c[3] / 255.0f};
    return vec4{(float)c[0] / 255.0f, (float)c[1] / 255.0f, (float)c[2] / 255.0f, (float)c[3] / 255.0f};
}
inline int texel_index(float f) { return (f == f && std::fabs(f) < 1e9f) ? (int)f : 0; }   // non-finite coordinate: texel 0
inline vec4 sample_texture(const Scene &s, int idx, vec2 uv) {
    const Scene::Texture &t = s.textures[(size_t)idx];
    int W = (int)t.w, H = (int)t.h;
    if (t.mag == 0) {
        int i = texel_index(std::floor(uv.x * (float)W)), j = texel_index(std::floor(uv.y * (float)H));
        return fetch_texel(t, wrap_texel(i, W, t.wrap_u), wrap_texel(j, H, t.wrap_v));
    }
    // 8 fractional bits of sub-texel precision, rounded to nearest (see oracle_svgf.cpp bilinear_setup)
    float uu = std::floor((uv.x * (float)W - 0.5f) * 256.0f + 0.5f) * 0.00390625f, vv = std::floor((uv.y * (float)H - 0.5f) * 256.0f + 0.5f) * 0.00390625f;
    float fu = std::floor(uu), fv = std::floor(vv);
    float a = uu - fu, b = vv - fv;
    int i = texel_index(fu), j = texel_index(fv);
    int x0 = wrap_texel(i, W, t.wrap_u), x1 = wrap_texel(i + 1, W, t.wrap_u), y0 = wrap_texel(j, H, t.wrap_v), y1 = wrap_texel(j + 1, H, t.wrap_v);
    vec4 t00 = fetch_texel(t, x0, y0), t10 = fetch_texel(t, x1, y0), t01 = fetch_texel(t, x0, y1), t11 = fetch_texel(t, x1, y1);
    auto lerp = [&](float c00, float c10, float c01, float c11) {
        return (1 - a) * (1 - b) * c00 + a * (1 - b) * c10 + (1 - a) * b * c01 + a * b * c11;
    };
    return vec4{lerp(t00.x, t10.x, t01.x, t11.x), lerp(t00.y, t10.y, t01.y, t11.y), lerp(t00.z, t10.z, t01.z, t11.z), lerp(t00.w, t10.w, t01.w, t11.w)};
}
inline bool has_texture(const Scene &s, int idx) { return idx >= 0 && (size_t)idx < s.textures.size() && s.textures[(size_t)idx].w != 0; }

struct Hit { double t, u, v; uint32_t tri; };   // u,v = barycentrics of vertex 1 and 2 (hitAttributeEXT)

// Row-major 3x4 application of Primitive.transform (resource_manager.cpp:608-617): x' = m00 x + m01 y + m02 z + m03,
// accumulated left to right in fp32 without contraction. The CUDA builder uses the same order, so both sides
// trace bit-identical world-space vertices.
inline void xform_point(const float *m, const float *p, float *o) {
    for (int r = 0; r < 3; ++r) o[r] = ((m[0 * 4 + r] * p[0] + m[1 * 4 + r] * p[1]) + m[2 * 4 + r] * p[2]) + m[3 * 4 + r];
}

struct BuildCtx {
    const float *tri;
    std::vector<float> cmin;   // per-tri bounds
    std::vector<float> cmax;
    std::vector<float> cen;
    std::vector<uint32_t> idx;
    std::vector<Node> nodes;
    std::atomic<uint32_t> next{0};
};

inline float half_area(const float *mn, const float *mx) {
    float dx = mx[0] - mn[0], dy = mx[1] - mn[1], dz = mx[2] - mn[2];
    return dx * dy + dy * dz + dz * dx;
}

void build_rec(BuildCtx &c, uint32_t node_idx, uint32_t first, uint32_t count, int depth) {
    Node &n = c.nodes[node_idx];
    float bmin[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, bmax[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    float cbmin[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, cbmax[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (uint32_t i = first; i < first + count; ++i) {
        uint32_t t = c.idx[i];
        for (int a = 0; a < 3; ++a) {
            bmin[a] = std::min(bmin[a], c.cmin[3 * t + a]);
            bmax[a] = std::max(bmax[a], c.cmax[3 * t + a]);
            cbmin[a] = std::min(cbmin[a], c.cen[3 * t + a]);
            cbmax[a] = std::max(cbmax[a], c.cen[3 * t + a]);
        }
    }
    for (int a = 0; a < 3; ++a) { n.bmin[a] = bmin[a]; n.bmax[a] = bmax[a]; }
    const uint32_t kLeaf = 4;
    if (count <= 2) { n.left_first = first; n.count = count; return; }

    const int NB = 16;
    int best_axis = -1, best_split = 0;
    float best_cost = FLT_MAX;
    for (int a = 0; a < 3; ++a) {
        float ext = cbmax[a] - cbmin[a];
        if (!(ext > 0.0f)) continue;
        float scale = (float)NB / ext;
        uint32_t bc[NB] = {0};
        float bmn[NB][3], bmx[NB][3];
        for (int b = 0; b < NB; ++b) for (int k = 0; k < 3; ++k) { bmn[b][k] = FLT_MAX; bmx[b][k] = -FLT_MAX; }
        for (uint32_t i = first; i < first + count; ++i) {
            uint32_t t = c.idx[i];
            int b = std::min(NB - 1, (int)((c.cen[3 * t + a] - cbmin[a]) * scale));
            bc[b]++;
            for (int k = 0; k < 3; ++k) {
                bmn[b][k] = std::min(bmn[b][k], c.cmin[3 * t + k]);
                bmx[b][k] = std::max(bmx[b][k], c.cmax[3 * t + k]);
            }
        }
        float la[NB - 1], ra[NB - 1];
        uint32_t lc[NB - 1], rc[NB - 1];
        float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        uint32_t cnt = 0;
        for (int b = 0; b < NB - 1; ++b) {
            cnt += bc[b];
            for (int k = 0; k < 3; ++k) { mn[k] = std::min(mn[k], bmn[b][k]); mx[k] = std::max(mx[k], bmx[b][k]); }
            lc[b] = cnt; la[b] = cnt ? half_area(mn, mx) : 0.0f;
        }
        for (int k = 0; k < 3; ++k) { mn[k] = FLT_MAX; mx[k] = -FLT_MAX; }
        cnt = 0;
        for (int b = NB - 1; b > 0; --b) {
            cnt += bc[b];
            for (int k = 0; k < 3; ++k) { mn[k] = std::min(mn[k], bmn[b][k]); mx[k] = std::max(mx[k], bmx[b][k]); }
            rc[b - 1] = cnt; ra[b - 1] = cnt ? half_area(mn, mx) : 0.0f;
        }
        for (int b = 0; b < NB - 1; ++b) {
            if (lc[b] == 0 || rc[b] == 0) continue;
            float cost = la[b] * lc[b] + ra[b] * rc[b];
            if (cost < best_cost) { best_cost = cost; best_axis = a; best_split = b; }
        }
    }
    // SAH termination: small ranges become leaves when splitting does not pay (traversal cost 1, test cost 1)
    float leaf_cost = half_area(bmin, bmax) * (float)count;
    if (best_axis < 0 && count <= 8) { n.left_first = first; n.count = count; return; }
    if (best_axis >= 0 && count <= kLeaf && best_cost + half_area(bmin, bmax) >= leaf_cost) {
        n.left_first = first; n.count = count; return;
    }
    uint32_t mid;
    if (best_axis < 0) {
        mid = first + count / 2;   // degenerate: all centroids equal -> median split
    } else {
        float ext = cbmax[best_axis] - cbmin[best_axis];
        float scale = (float)NB / ext;
        uint32_t *b = c.idx.data() + first, *e = b + count;
        uint32_t *m = std::partition(b, e, [&](uint32_t t) {
            int bin = std::min(NB - 1, (int)((c.cen[3 * t + best_axis] - cbmin[best_axis]) * scale));
            return bin <= best_split;
        });
        mid = (uint32_t)(m - c.idx.data());
        if (mid == first || mid == first + count) mid = first + count / 2;
    }
    uint32_t left = c.next.fetch_add(2);
    n.left_first = left;
    n.count = 0;
    uint32_t lcount = mid - first, rcount = count - lcount;
    if (count > 20000 && depth < 12) {
#pragma omp task shared(c)
        build_rec(c, left, first, lcount, depth + 1);
#pragma omp task shared(c)
        build_rec(c, left + 1, mid, rcount, depth + 1);
#pragma omp taskwait
    } else {
        build_rec(c, left, first, lcount, depth + 1);
        build_rec(c, left + 1, mid, rcount, depth + 1);
    }
}

// Double-precision watertight ray/triangle test (Woop, Benthin, Wald 2013), two-sided, tMin < t < tMax.
struct RayD {
    double o[3], d[3];
    int kx, ky, kz;
    double Sx, Sy, Sz;
    double tmin, tmax;
    double inv[3];
};
inline void ray_setup(RayD &r, vec3 o, vec3 d, float tmin, float tmax) {
    r.o[0] = o.x; r.o[1] = o.y; r.o[2] = o.z;
    r.d[0] = d.x; r.d[1] = d.y; r.d[2] = d.z;
    r.tmin = tmin; r.tmax = tmax;
    double ax = std::fabs(r.d[0]), ay = std::fabs(r.d[1]), az = std::fabs(r.d[2]);
    r.kz = (ax > ay) ? ((ax > az) ? 0 : 2) : ((ay > az) ? 1 : 2);
    r.kx = (r.kz + 1) % 3; r.ky = (r.kx + 1) % 3;
    if (r.d[r.kz] < 0.0) std::swap(r.kx, r.ky);
    r.Sx = r.d[r.kx] / r.d[r.kz];
    r.Sy = r.d[r.ky] / r.d[r.kz];
    r.Sz = 1.0 / r.d[r.kz];
    for (int a = 0; a < 3; ++a) r.inv[a] = 1.0 / r.d[a];
}
inline bool tri_hit(const RayD &r, const float *tv, double &t, double &u, double &v) {
    double A[3], B[3], C[3];
    for (int a = 0; a < 3; ++a) { A[a] = (double)tv[a] - r.o[a]; B[a] = (double)tv[3 + a] - r.o[a]; C[a] = (double)tv[6 + a] - r.o[a]; }
    double Ax = A[r.kx] - r.Sx * A[r.kz], Ay = A[r.ky] - r.Sy * A[r.kz];
    double Bx = B[r.kx] - r.Sx * B[r.kz], By = B[r.ky] - r.Sy * B[r.kz];
    double Cx = C[r.kx] - r.Sx * C[r.kz], Cy = C[r.ky] - r.Sy * C[r.kz];
    double U = Cx * By - Cy * Bx;
    double V = Ax * Cy - Ay * Cx;
    double W = Bx * Ay - By * Ax;
    if ((U < 0.0 || V < 0.0 || W < 0.0) && (U > 0.0 || V > 0.0 || W > 0.0)) return false;
    double det = U + V + W;
    if (det == 0.0) return false;
    double Az = r.Sz * A[r.kz], Bz = r.Sz * B[r.kz], Cz = r.Sz * C[r.kz];
    double T = U * Az + V * Bz + W * Cz;
    double tt = T / det;
    if (!(tt > r.tmin && tt < r.tmax)) return false;
    t = tt; u = V / det; v = W / det;
    return true;
}
inline bool box_hit(const RayD &r, const Node &n, double tmax, double &tnear) {
    double t0 = r.tmin, t1 = tmax;
    for (int a = 0; a < 3; ++a) {
        double lo = ((double)n.bmin[a] - r.o[a]) * r.inv[a];
        double hi = ((double)n.bmax[a] - r.o[a]) * r.inv[a];
        if (lo > hi) std::swap(lo, hi);
        // NaN (0 * inf) lanes must not cull: comparisons below keep t0/t1 when lo/hi are NaN
        if (lo > t0) t0 = lo;
        if (hi < t1) t1 = hi;
    }
    tnear = t0;
    return t0 <= t1 * (1.0 + 1e-12) + 1e-300;
}

bool trace_any(const Scene &s, vec3 o, vec3 d, float tmin, float tmax) {
    if (s.nodes.empty()) return false;
    RayD r; ray_setup(r, o, d, tmin, tmax);
    uint32_t stack[128]; int sp = 0;
    stack[sp++] = 0;
    while (sp) {
        const Node &n = s.nodes[stack[--sp]];
        double tn;
        if (!box_hit(r, n, r.tmax, tn)) continue;
        if (n.count) {
            for (uint32_t i = 0; i < n.count; ++i) {
                double t, u, v;
                if (tri_hit(r, &s.tri[(size_t)(n.left_first + i) * 9], t, u, v)) return true;
            }
        } else {
            stack[sp++] = n.left_first;
            stack[sp++] = n.left_first + 1;
        }
    }
    return false;
}

// `accept` = the any-hit stage (NULL: opaque geometry, every candidate counts): a rejected candidate is ignored and the
// traversal goes on — the G-buffer producer's alpha test (gbuf.frag:27-32).
template <class Accept>
bool trace_closest_filtered(const Scene &s, vec3 o, vec3 d, float tmin, float tmax, Hit &hit, const Accept &accept) {
    if (s.nodes.empty()) return false;
    RayD r; ray_setup(r, o, d, tmin, tmax);
    bool found = false;
    uint32_t stack[128]; int sp = 0;
    stack[sp++] = 0;
    while (sp) {
        const Node &n = s.nodes[stack[--sp]];
        double tn;
        if (!box_hit(r, n, r.tmax, tn)) continue;
        if (n.count) {
            for (uint32_t i = 0; i < n.count; ++i) {
                double t, u, v;
                if (tri_hit(r, &s.tri[(size_t)(n.left_first + i) * 9], t, u, v) && accept(n.left_first + i, u, v)) {
                    r.tmax = t; hit.t = t; hit.u = u; hit.v = v; hit.tri = n.left_first + i; found = true;
                }
            }
        } else {
            double t0, t1;
            const Node &l = s.nodes[n.left_first], &rr = s.nodes[n.left_first + 1];
            bool hl = box_hit(r, l, r.tmax, t0), hr = box_hit(r, rr, r.tmax, t1);
            if (hl && hr) {
                if (t0 < t1) { stack[sp++] = n.left_first + 1; stack[sp++] = n.left_first; }
                else { stack[sp++] = n.left_first; stack[sp++] = n.left_first + 1; }
            } else if (hl) stack[sp++] = n.left_first;
            else if (hr) stack[sp++] = n.left_first + 1;
        }
    }
    return found;
}

bool trace_closest(const Scene &s, vec3 o, vec3 d, float tmin, float tmax, Hit &hit) {
    return trace_closest_filtered(s, o, d, tmin, tmax, hit, [](uint32_t, double, double) { return true; });
}

// reflection_hit.rchit:10-72 for triangle pid of geometry g at the barycentrics (hx, hy) of vertices 1 and 2
vec4 reflection_hit(const Scene &s, const PerFrameData &pfd, uint32_t g, uint32_t pid, float hx, float hy) {
    const Primitive &prim = s.primitives[g];
    uint32_t i0 = s.indices[prim.index_offset + 3 * pid + 0];
    uint32_t i1 = s.indices[prim.index_offset + 3 * pid + 1];
    uint32_t i2 = s.indices[prim.index_offset + 3 * pid + 2];
    const Vertex &v0 = s.vertices[prim.vertex_offset + i0];
    const Vertex &v1 = s.vertices[prim.vertex_offset + i1];
    const Vertex &v2 = s.vertices[prim.vertex_offset + i2];
    float b0 = 1.0f - hx - hy, b1 = hx, b2 = hy;
    vec3 normal = v3(v0.normal[0], v0.normal[1], v0.normal[2]) * b0 + v3(v1.normal[0], v1.normal[1], v1.normal[2]) * b1 +
                  v3(v2.normal[0], v2.normal[1], v2.normal[2]) * b2;
    vec3 pobj = v3(v0.pos[0], v0.pos[1], v0.pos[2]) * b0 + v3(v1.pos[0], v1.pos[1], v1.pos[2]) * b1 +
                v3(v2.pos[0], v2.pos[1], v2.pos[2]) * b2;
    vec4 pw = mul44(prim.transform, vec4{pobj.x, pobj.y, pobj.z, 1.0f});
    vec3 position = v3(pw.x, pw.y, pw.z);

    vec2 uv = {v0.uv0[0] * b0 + v1.uv0[0] * b1 + v2.uv0[0] * b2, v0.uv0[1] * b0 + v1.uv0[1] * b1 + v2.uv0[1] * b2};   // :22
    vec3 albedo = v3(prim.material.base_color[0], prim.material.base_color[1], prim.material.base_color[2]);
    if (has_texture(s, prim.material.base_color_texture)) {                                                       // :26-32
        vec4 c = sample_texture(s, prim.material.base_color_texture, uv);
        albedo = v3(c.x, c.y, c.z);
    }
    float metallic = prim.material.metallic_factor;
    float roughness = prim.material.roughness_factor;
    if (has_texture(s, prim.material.metallic_roughness_texture)) {                                               // :35-39
        vec4 mr = sample_texture(s, prim.material.metallic_roughness_texture, uv);
        metallic *= mr.y;
        roughness *= mr.z;
    }

    vec3 camera_position = v3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
    vec3 V = normalize(camera_position - position);
    vec3 L = -v3(pfd.directional_light.direction[0], pfd.directional_light.direction[1], pfd.directional_light.direction[2]);
    vec3 N = normal;
    vec3 H = normalize(L + V);

    roughness = std::min(std::max(roughness, 0.04f), 1.0f);
    metallic = std::min(std::max(metallic, 0.0f), 1.0f);
    float ambient_factor = PI_INVERSE_F * 0.2f;
    vec3 li = v3(pfd.directional_light.intensity[0], pfd.directional_light.intensity[1], pfd.directional_light.intensity[2]);
    vec3 lc = v3(pfd.directional_light.color[0], pfd.directional_light.color[1], pfd.directional_light.color[2]);
    vec3 f0 = v3(mixf(0.04f, albedo.x, metallic), mixf(0.04f, albedo.y, metallic), mixf(0.04f, albedo.z, metallic));
    vec3 F = fresnel_schlick(f0, H, V);
    vec3 ambient = albedo * ambient_factor;
    vec3 diffuse = diffuse_brdf(metallic, albedo, F);
    vec3 specular = specular_brdf(roughness, F, V, L, N, H);
    float ndl = gl_max(dot(N, L), 0.0f);
    vec3 lighting = ambient + (diffuse + specular) * ndl * li * lc;
    return vec4{lighting.x, lighting.y, lighting.z, 1.0f};
}

// gbuf.frag:19-32, the any-hit stage of the primary ray: a fragment failing the alpha-mask test, or with alpha exactly 0, is
// discarded. (c1, c2) = barycentrics of vertices 1 and 2.
bool gbuffer_alpha_test(const Scene &s, uint32_t g, uint32_t k, float c1, float c2) {
    const Primitive &pr = s.primitives[g];
    float alpha = pr.material.base_color[3];
    if (has_texture(s, pr.material.base_color_texture)) {
        const Vertex &a0 = s.vertices[pr.vertex_offset + s.indices[pr.index_offset + 3 * k + 0]];
        const Vertex &a1 = s.vertices[pr.vertex_offset + s.indices[pr.index_offset + 3 * k + 1]];
        const Vertex &a2 = s.vertices[pr.vertex_offset + s.indices[pr.index_offset + 3 * k + 2]];
        float c0 = 1.0f - c1 - c2;
        vec2 uvt = {a0.uv0[0] * c0 + a1.uv0[0] * c1 + a2.uv0[0] * c2, a0.uv0[1] * c0 + a1.uv0[1] * c1 + a2.uv0[1] * c2};
        alpha = sample_texture(s, pr.material.base_color_texture, uvt).w;
    }
    if (pr.material.alpha_mask == 1 && alpha < pr.material.alpha_cutoff) return false;
    return alpha != 0.0f;
}

// shadow_anyhit.rahit:22-26 (the shader samples textures[base_color_texture] unconditionally; index -1 counts as opaque here)
bool rahit_alpha_test(const Scene &s, uint32_t g, uint32_t k, float c1, float c2) {
    const Primitive &pr = s.primitives[g];
    if (pr.material.alpha_mask != 1 || !has_texture(s, pr.material.base_color_texture)) return true;
    const Vertex &a0 = s.vertices[pr.vertex_offset + s.indices[pr.index_offset + 3 * k + 0]];
    const Vertex &a1 = s.vertices[pr.vertex_offset + s.indices[pr.index_offset + 3 * k + 1]];
    const Vertex &a2 = s.vertices[pr.vertex_offset + s.indices[pr.index_offset + 3 * k + 2]];
    float c0 = 1.0f - c1 - c2;
    vec2 uvt = {a0.uv0[0] * c0 + a1.uv0[0] * c1 + a2.uv0[0] * c2, a0.uv0[1] * c0 + a1.uv0[1] * c1 + a2.uv0[1] * c2};
    return !(sample_texture(s, pr.material.base_color_texture, uvt).w < pr.material.alpha_cutoff);
}

// closesthit.rchit:11-41 for one hit: the albedo, the shading normal N and the world-space hit point (the shadow ray's origin)
struct RaytracedHit { vec3 albedo, N, position; };
RaytracedHit raytraced_hit(const Scene &s, uint32_t g, uint32_t pid, float b1, float b2) {
    const Primitive &prim = s.primitives[g];
    const Vertex &v0 = s.vertices[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 0]];
    const Vertex &v1 = s.vertices[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 1]];
    const Vertex &v2 = s.vertices[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 2]];
    float b0 = 1.0f - b1 - b2;
    vec2 tuv = {v0.uv0[0] * b0 + v1.uv0[0] * b1 + v2.uv0[0] * b2, v0.uv0[1] * b0 + v1.uv0[1] * b1 + v2.uv0[1] * b2};
    vec3 normal = v3(v0.normal[0], v0.normal[1], v0.normal[2]) * b0 + v3(v1.normal[0], v1.normal[1], v1.normal[2]) * b1 +
                  v3(v2.normal[0], v2.normal[1], v2.normal[2]) * b2;
    vec3 pobj = v3(v0.pos[0], v0.pos[1], v0.pos[2]) * b0 + v3(v1.pos[0], v1.pos[1], v1.pos[2]) * b1 +
                v3(v2.pos[0], v2.pos[1], v2.pos[2]) * b2;
    vec4 pw = mul44(prim.transform, vec4{pobj.x, pobj.y, pobj.z, 1.0f});
    RaytracedHit r;
    r.position = v3(pw.x, pw.y, pw.z);
    r.albedo = v3(prim.material.base_color[0], prim.material.base_color[1], prim.material.base_color[2]);
    if (has_texture(s, prim.material.base_color_texture)) {
        vec4 c = sample_texture(s, prim.material.base_color_texture, tuv);
        r.albedo = v3(c.x, c.y, c.z);
    }
    r.N = normal;
    if (has_texture(s, prim.material.normal_map)) {                                       // closesthit.rchit:35-41
        vec3 tan3 = v3(v0.tangent[0], v0.tangent[1], v0.tangent[2]) * b0 + v3(v1.tangent[0], v1.tangent[1], v1.tangent[2]) * b1 +
                    v3(v2.tangent[0], v2.tangent[1], v2.tangent[2]) * b2;
        float tw = v0.tangent[3] * b0 + v1.tangent[3] * b1 + v2.tangent[3] * b2;
        vec4 c = sample_texture(s, prim.material.normal_map, tuv);
        vec3 tsn = normalize(v3(c.x * 2.0f - 1.0f, c.y * 2.0f - 1.0f, c.z * 2.0f - 1.0f));
        vec3 bitangent = cross(tsn, tan3) * tw;
        vec3 tangent = normalize(tan3 - normal * dot(tan3, normal));
        r.N = tangent * tsn.x + bitangent * tsn.y + normal * tsn.z;
    }
    return r;
}

// closesthit.rchit:43-57 / closesthit_test_alpha.rchit:37-50: the payload of a shaded hit given the shadow ray's answer
vec4 raytraced_color(const PerFrameData &pfd, int alpha_test, vec3 albedo, vec3 N, bool occluded) {
    vec3 light_dir = -v3(pfd.directional_light.direction[0], pfd.directional_light.direction[1], pfd.directional_light.direction[2]);
    vec3 lc = v3(pfd.directional_light.color[0], pfd.directional_light.color[1], pfd.directional_light.color[2]);
    vec3 li = v3(pfd.directional_light.intensity[0], pfd.directional_light.intensity[1], pfd.directional_light.intensity[2]);
    vec3 albedo_lighting = albedo * (alpha_test ? 0.2f : PI_INVERSE_F);
    vec3 c = albedo_lighting;
    if (!occluded) {
        float ndl = gl_max(dot(N, light_dir), 0.0f);
        vec3 lit = alpha_test ? (albedo * ndl) * lc : ((albedo * ndl) * li) * lc;
        c = albedo_lighting + lit;
    }
    return vec4{c.x, c.y, c.z, 1.0f};
}

// imageStore to a B8G8R8A8_UNORM image: float -> UNORM8 (NaN -> 0), B first
inline void store_bgra8(uint8_t *o, vec4 payload) {
    auto q = [](float f) { f = (f == f) ? std::min(std::max(f, 0.0f), 1.0f) : 0.0f; return (uint8_t)std::lrintf(f * 255.0f); };
    o[0] = q(payload.z); o[1] = q(payload.y); o[2] = q(payload.x); o[3] = q(payload.w);
}

// gl_FragCoord.xy * display_size_inverse of pixel (x, y)
inline vec2 gbuffer_pixel_uv(const PerFrameData &pfd, int x, int y) {
    return vec2{((float)x + 0.5f) * pfd.display_size_inverse[0], ((float)y + 0.5f) * pfd.display_size_inverse[1]};
}

// gbuf.frag:33-58 for a primary hit seen through the pixel at uv (gbuffer_pixel_uv): albedo BGRA8 (albedo4 may be NULL),
// normals / object id RGBA16F, motion / metallic-roughness RGBA16F, depth D32
void gbuffer_hit(const Scene &s, const PerFrameData &pfd, uint32_t g, uint32_t pid, float b1, float b2, vec2 uv, uint8_t *albedo_out,
                 uint16_t *normals_out, uint16_t *motion_out, float *depth_out) {
    const Primitive &prim = s.primitives[g];
    const Vertex &v0 = s.vertices[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 0]];
    const Vertex &v1 = s.vertices[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 1]];
    const Vertex &v2 = s.vertices[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 2]];
    float b0 = 1.0f - b1 - b2;
    vec3 nobj = v3(v0.normal[0], v0.normal[1], v0.normal[2]) * b0 + v3(v1.normal[0], v1.normal[1], v1.normal[2]) * b1 +
                v3(v2.normal[0], v2.normal[1], v2.normal[2]) * b2;
    vec3 pobj = v3(v0.pos[0], v0.pos[1], v0.pos[2]) * b0 + v3(v1.pos[0], v1.pos[1], v1.pos[2]) * b1 +
                v3(v2.pos[0], v2.pos[1], v2.pos[2]) * b2;
    const Material &mat = prim.material;
    vec2 tuv = {v0.uv0[0] * b0 + v1.uv0[0] * b1 + v2.uv0[0] * b2, v0.uv0[1] * b0 + v1.uv0[1] * b1 + v2.uv0[1] * b2};
    vec4 albedo4 = {mat.base_color[0], mat.base_color[1], mat.base_color[2], mat.base_color[3]};
    if (has_texture(s, mat.base_color_texture)) albedo4 = sample_texture(s, mat.base_color_texture, tuv);       // gbuf.frag:20-26
    if (has_texture(s, mat.normal_map)) {                                                                     // gbuf.frag:35-41
        vec4 c = sample_texture(s, mat.normal_map, tuv);
        vec3 tsn = normalize(v3(c.x * 2.0f - 1.0f, c.y * 2.0f - 1.0f, c.z * 2.0f - 1.0f));
        vec3 tan3 = v3(v0.tangent[0], v0.tangent[1], v0.tangent[2]) * b0 + v3(v1.tangent[0], v1.tangent[1], v1.tangent[2]) * b1 +
                    v3(v2.tangent[0], v2.tangent[1], v2.tangent[2]) * b2;
        float tw = v0.tangent[3] * b0 + v1.tangent[3] * b1 + v2.tangent[3] * b2;
        vec3 bitangent = cross(tsn, tan3) * tw;
        vec3 tangent = normalize(tan3 - nobj * dot(tan3, nobj));
        nobj = tangent * tsn.x + bitangent * tsn.y + nobj * tsn.z;
    }
    float metallic = mat.metallic_factor, roughness = mat.roughness_factor;
    if (has_texture(s, mat.metallic_roughness_texture)) {                                                     // gbuf.frag:52-56
        vec4 c = sample_texture(s, mat.metallic_roughness_texture, tuv);
        metallic *= c.y;
        roughness *= c.z;
    }
    // normal_matrix = inverseTranspose(mat3(transform)) (hybrid_render_path.cpp:45) = cofactor(M) / det(M)
    const float *m = prim.transform;
    double a00 = m[0], a10 = m[1], a20 = m[2], a01 = m[4], a11 = m[5], a21 = m[6], a02 = m[8], a12 = m[9], a22 = m[10];
    double c00 = a11 * a22 - a21 * a12, c01 = -(a10 * a22 - a20 * a12), c02 = a10 * a21 - a20 * a11;
    double c10 = -(a01 * a22 - a21 * a02), c11 = a00 * a22 - a20 * a02, c12 = -(a00 * a21 - a20 * a01);
    double c20 = a01 * a12 - a11 * a02, c21 = -(a00 * a12 - a10 * a02), c22 = a00 * a11 - a10 * a01;
    double det = a00 * c00 + a01 * c01 + a02 * c02;
    // (M^-T)[r][c] = cof[r][c] / det, with cof indexed [row][col] of M (a_rc = m[c*4+r])
    float nm[9] = {(float)(c00 / det), (float)(c10 / det), (float)(c20 / det),    // column 0: rows 0..2
                   (float)(c01 / det), (float)(c11 / det), (float)(c21 / det),    // column 1
                   (float)(c02 / det), (float)(c12 / det), (float)(c22 / det)};   // column 2
    vec3 nw = {nm[0] * nobj.x + nm[3] * nobj.y + nm[6] * nobj.z,
               nm[1] * nobj.x + nm[4] * nobj.y + nm[7] * nobj.z,
               nm[2] * nobj.x + nm[5] * nobj.y + nm[8] * nobj.z};
    nw = normalize(nw);
    vec4 pw = mul44(prim.transform, vec4{pobj.x, pobj.y, pobj.z, 1.0f});
    vec4 clip = mul44(pfd.camera_proj, mul44(pfd.camera_view, pw));
    vec4 pclip = mul44(pfd.camera_proj_prev_frame, mul44(pfd.camera_view_prev_frame, pw));
    vec2 cur_ndc = uv;   // gl_FragCoord.xy * display_size_inverse
    vec2 prev_ndc = {(pclip.x / pclip.w) * 0.5f + 0.5f, (pclip.y / pclip.w) * 0.5f + 0.5f};
    if (albedo_out) {
        auto q = [](float f) { f = (f == f) ? std::min(std::max(f, 0.0f), 1.0f) : 0.0f; return (uint8_t)std::lrintf(f * 255.0f); };   // NaN -> 0
        albedo_out[0] = q(albedo4.z); albedo_out[1] = q(albedo4.y); albedo_out[2] = q(albedo4.x); albedo_out[3] = q(albedo4.w);
    }
    store_rgba16f(normals_out, 1, 0, 0, vec4{nw.x, nw.y, nw.z, (float)g});
    store_rgba16f(motion_out, 1, 0, 0, vec4{cur_ndc.x - prev_ndc.x, cur_ndc.y - prev_ndc.y, metallic, roughness});
    *depth_out = clip.z / clip.w;
}

}  // namespace

extern "C" {

// Host threads of every "#pragma omp" loop in the oracle. A launcher may have exported OMP_NUM_THREADS=1 (torchrun does for each rank);
// bench.py's CPU arm sets the count explicitly and reports what the runtime then uses. Returns omp_get_max_threads().
int vo_set_num_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
    return omp_get_max_threads();
#else
    (void)n;
    return 1;
#endif
}

struct vo_scene;

vo_scene *vo_scene_create(const Vertex *vertices, uint32_t n_vertices, const uint32_t *indices, uint32_t n_indices,
                          const Primitive *primitives, uint32_t n_primitives) {
    Scene *s = new Scene();
    s->vertices.assign(vertices, vertices + n_vertices);
    s->indices.assign(indices, indices + n_indices);
    s->primitives.assign(primitives, primitives + n_primitives);
    size_t n_tris = 0;
    for (uint32_t g = 0; g < n_primitives; ++g) n_tris += primitives[g].index_count / 3;
    std::vector<float> tri(n_tris * 9);
    std::vector<uint32_t> geom(n_tris), pid(n_tris);
    size_t t = 0;
    for (uint32_t g = 0; g < n_primitives; ++g) {
        const Primitive &p = primitives[g];
        for (uint32_t k = 0; k < p.index_count / 3; ++k, ++t) {
            for (int c = 0; c < 3; ++c) {
                uint32_t vi = p.vertex_offset + indices[p.index_offset + 3 * k + c];
                xform_point(p.transform, vertices[vi].pos, &tri[t * 9 + 3 * c]);
            }
            geom[t] = g; pid[t] = k;
        }
    }
    s->n_tris = (uint32_t)n_tris;
    if (n_tris == 0) return reinterpret_cast<vo_scene *>(s);

    BuildCtx c;
    c.tri = tri.data();
    c.cmin.resize(n_tris * 3); c.cmax.resize(n_tris * 3); c.cen.resize(n_tris * 3); c.idx.resize(n_tris);
#pragma omp parallel for
    for (long long i = 0; i < (long long)n_tris; ++i) {
        for (int a = 0; a < 3; ++a) {
            float x0 = tri[i * 9 + a], x1 = tri[i * 9 + 3 + a], x2 = tri[i * 9 + 6 + a];
            float mn = std::min(x0, std::min(x1, x2)), mx = std::max(x0, std::max(x1, x2));
            c.cmin[3 * i + a] = mn; c.cmax[3 * i + a] = mx; c.cen[3 * i + a] = 0.5f * (mn + mx);
        }
        c.idx[i] = (uint32_t)i;
    }
    c.nodes.resize(2 * n_tris + 2);
    c.next = 2;   // node 0 = root, node 1 unused (keeps sibling pairs aligned)
#pragma omp parallel
#pragma omp single
    build_rec(c, 0, 0, (uint32_t)n_tris, 0);
    c.nodes.resize(c.next.load());
    s->nodes.swap(c.nodes);
    // leaf order
    s->tri.resize(n_tris * 9); s->tri_geom.resize(n_tris); s->tri_prim.resize(n_tris);
#pragma omp parallel for
    for (long long i = 0; i < (long long)n_tris; ++i) {
        uint32_t src = c.idx[i];
        std::memcpy(&s->tri[i * 9], &tri[(size_t)src * 9], 36);
        s->tri_geom[i] = geom[src]; s->tri_prim[i] = pid[src];
    }
    return reinterpret_cast<vo_scene *>(s);
}

// ResourceManager::UploadTextureFromData: appends to textures[] and returns the index. format 43 = R8G8B8A8_SRGB, 37 = UNORM.
int vo_scene_add_texture(vo_scene *s_, uint32_t w, uint32_t h, const uint8_t *rgba, int vk_format, int mag_filter, int min_filter,
                         int address_mode_u, int address_mode_v) {
    Scene &s = *reinterpret_cast<Scene *>(s_);
    Scene::Texture t;
    t.w = w; t.h = h;
    t.rgba.assign(rgba, rgba + (size_t)w * h * 4);
    t.srgb = vk_format == 43;
    t.mag = mag_filter; t.min = min_filter; t.wrap_u = address_mode_u; t.wrap_v = address_mode_v;
    s.textures.push_back(std::move(t));
    return (int)s.textures.size() - 1;
}
// texture(textures[idx], uv) for unit tests
void vo_sample_texture(const vo_scene *s_, int idx, float u, float v, float *out4) {
    vec4 c = sample_texture(*reinterpret_cast<const Scene *>(s_), idx, vec2{u, v});
    out4[0] = c.x; out4[1] = c.y; out4[2] = c.z; out4[3] = c.w;
}

void vo_scene_destroy(vo_scene *s) { delete reinterpret_cast<Scene *>(s); }
uint32_t vo_scene_num_triangles(const vo_scene *s) { return reinterpret_cast<const Scene *>(s)->n_tris; }

// Single-ray entry points for unit tests. Returns 1 on hit.
int vo_trace_any(const vo_scene *s_, const float *o, const float *d, float tmin, float tmax) {
    return trace_any(*reinterpret_cast<const Scene *>(s_), v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), tmin, tmax) ? 1 : 0;
}
int vo_trace_closest(const vo_scene *s_, const float *o, const float *d, float tmin, float tmax, double *t_u_v,
                     uint32_t *geom_prim) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    Hit h;
    if (!trace_closest(s, v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), tmin, tmax, h)) return 0;
    t_u_v[0] = h.t; t_u_v[1] = h.u; t_u_v[2] = h.v;
    geom_prim[0] = s.tri_geom[h.tri]; geom_prim[1] = s.tri_prim[h.tri];
    return 1;
}

// Closest hit with an any-hit stage supplied by the caller (oracle/_ref runs the reference's shadow_anyhit.rahit through it):
// accept(user, geometry index, primitive id, u, v) != 0 keeps the candidate, 0 = ignoreIntersectionEXT.
typedef int (*vo_anyhit_fn)(void *user, uint32_t geometry_index, uint32_t primitive_id, double u, double v);
int vo_trace_closest_filtered(const vo_scene *s_, const float *o, const float *d, float tmin, float tmax, vo_anyhit_fn accept, void *user, double *t_u_v,
                              uint32_t *geom_prim) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    Hit h;
    auto f = [&](uint32_t tri, double u, double v) { return !accept || accept(user, s.tri_geom[tri], s.tri_prim[tri], u, v) != 0; };
    if (!trace_closest_filtered(s, v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), tmin, tmax, h, f)) return 0;
    t_u_v[0] = h.t; t_u_v[1] = h.u; t_u_v[2] = h.v;
    geom_prim[0] = s.tri_geom[h.tri]; geom_prim[1] = s.tri_prim[h.tri];
    return 1;
}

// raygen.rgen:14-66. Rows [y0, y1) only (bounded samples for the CPU baseline). `ao_spp` = 2 in the
// reference (:45,55); `flags` bit0 = trace shadow, bit1 = trace AO, bit2 = trace reflections (all set = reference).
// Optional outputs: refl_t (float per pixel: closest-hit distance of the reflection ray, -1 = miss / sky),
// ray_count (unique rays traced, SURVEY Q3 — the 4x duplicate shadow ray counts once).
void vo_raygen(const vo_scene *s_, const PerFrameData *pfd_, int W, int H, int y0, int y1, int ao_spp, int flags,
               const float *depth, const uint16_t *normals, uint16_t *shadow_ao, uint16_t *reflections,
               float *refl_t, uint64_t *ray_count) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    const PerFrameData &pfd = *pfd_;
    uint64_t rays = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : rays)
    for (int y = y0; y < y1; ++y) {
        for (int x = 0; x < W; ++x) {
            vec2 uv = {((float)x + 0.5f) / (float)W, ((float)y + 0.5f) / (float)H};
            uint32_t rng = seed_thread(((uint32_t)y * (uint32_t)H + (uint32_t)x) * pfd.frame_index);   // :17 (Q4)
            float current_depth = depth[(size_t)y * W + x];                                            // :19 (Q17)
            if (current_depth == 0.0f) {
                if (shadow_ao) store_rg16f(shadow_ao, W, x, y, vec4{1.0f, 1.0f, 0.0f, 1.0f});
                if (reflections) store_rgba16f(reflections, W, x, y, vec4{0, 0, 0, 0});
                if (refl_t) refl_t[(size_t)y * W + x] = -1.0f;
                continue;
            }
            vec3 P = get_world_space_position(pfd, current_depth, uv);
            vec3 L = -v3(pfd.directional_light.direction[0], pfd.directional_light.direction[1], pfd.directional_light.direction[2]);
            vec4 n4 = load_rgba16f(normals, W, x, y);
            vec3 N = v3(n4.x, n4.y, n4.z);
            vec3 origin = P + N * 0.1f;

            // :32-41 shadow (random numbers are always drawn, even when the ray is skipped)
            float rnd1 = random01(rng), rnd2 = random01(rng);
            float shadow_payload = 1.0f;
            if (flags & 1) {
                vec3 cone_dir = normalize(uniform_sample_cone(vec2{rnd1, rnd2}, 0.999995f));
                mat3 R = onb_from_unit_vector(L);
                shadow_payload = trace_any(s, origin, mul(R, cone_dir), 0.01f, 10000.0f) ? 0.0f : 1.0f;
                rays++;
            }
            // :44-55 AO
            float ao_payload = 0.0f;
            for (int i = 0; i < ao_spp; ++i) {
                rnd1 = random01(rng); rnd2 = random01(rng);
                if (flags & 2) {
                    vec3 rnd_dir = uniform_sample_cosine_weighted_hemisphere(vec2{rnd1, rnd2});
                    mat3 R = onb_from_unit_vector(N);
                    ao_payload += trace_any(s, origin, mul(R, rnd_dir), 0.01f, 5.0f) ? 0.0f : 1.0f;
                    rays++;
                } else {
                    ao_payload += 1.0f;
                }
            }
            ao_payload /= (float)ao_spp;
            if (shadow_ao) store_rg16f(shadow_ao, W, x, y, vec4{shadow_payload, ao_payload, 0.0f, 1.0f});

            // :59-65 reflection
            if (flags & 4) {
                vec3 cam = v3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
                vec3 I = normalize(P - cam);
                float ndi = dot(N, I);
                vec3 refl = I - N * (2.0f * ndi);      // GLSL reflect(I, N) = I - 2 dot(N, I) N
                Hit h;
                vec4 payload = {0, 0, 0, 0};
                float t = -1.0f;
                if (trace_closest(s, origin, refl, 0.01f, 10000.0f, h)) { payload = reflection_hit(s, pfd, s.tri_geom[h.tri], s.tri_prim[h.tri], (float)h.u, (float)h.v); t = (float)h.t; }
                rays++;
                if (reflections) store_rgba16f(reflections, W, x, y, payload);
                if (refl_t) refl_t[(size_t)y * W + x] = t;
            } else {
                if (reflections) store_rgba16f(reflections, W, x, y, vec4{0, 0, 0, 0});
                if (refl_t) refl_t[(size_t)y * W + x] = -1.0f;
            }
        }
    }
    if (ray_count) *ray_count = rays;
}

// The rays raygen.rgen:26-55 generates for ONE pixel, exactly as vo_raygen does (same statements, same order): ray 0 = shadow, rays
// 1..ao_spp = ambient occlusion; 8 floats each (origin xyz, tMin, direction xyz, tMax). Returns the number of rays (0 for a sky pixel).
// Tests use it to re-trace the pixels on which a GPU mask and the oracle disagree and to classify them (vo_brute_force).
int vo_raygen_pixel_rays(const PerFrameData *pfd_, int W, int H, int x, int y, const float *depth, const uint16_t *normals, int ao_spp, float *out_rays) {
    const PerFrameData &pfd = *pfd_;
    vec2 uv = {((float)x + 0.5f) / (float)W, ((float)y + 0.5f) / (float)H};
    uint32_t rng = seed_thread(((uint32_t)y * (uint32_t)H + (uint32_t)x) * pfd.frame_index);
    float current_depth = depth[(size_t)y * W + x];
    if (current_depth == 0.0f) return 0;
    vec3 P = get_world_space_position(pfd, current_depth, uv);
    vec3 L = -v3(pfd.directional_light.direction[0], pfd.directional_light.direction[1], pfd.directional_light.direction[2]);
    vec4 n4 = load_rgba16f(normals, W, x, y);
    vec3 N = v3(n4.x, n4.y, n4.z);
    vec3 origin = P + N * 0.1f;
    auto put = [&](int i, vec3 d, float tmax) {
        float *r = out_rays + 8 * i;
        r[0] = origin.x; r[1] = origin.y; r[2] = origin.z; r[3] = 0.01f; r[4] = d.x; r[5] = d.y; r[6] = d.z; r[7] = tmax;
    };
    float rnd1 = random01(rng), rnd2 = random01(rng);
    put(0, mul(onb_from_unit_vector(L), normalize(uniform_sample_cone(vec2{rnd1, rnd2}, 0.999995f))), 10000.0f);
    for (int i = 0; i < ao_spp; ++i) {
        rnd1 = random01(rng); rnd2 = random01(rng);
        put(1 + i, mul(onb_from_unit_vector(N), uniform_sample_cosine_weighted_hemisphere(vec2{rnd1, rnd2})), 5.0f);
    }
    return 1 + ao_spp;
}

// One ray against EVERY triangle in double precision (Moller-Trumbore, no acceleration structure): out[0] = 1 if any triangle is hit in
// (tmin, tmax), out[1] = closest such t (-1: none), out[2] = margin = the smallest distance of a nearby candidate from flipping its
// classification (normalised barycentric distance to an edge, or relative distance of t to an end of the interval). A small margin
// means the ray grazes an edge or an interval end: the self-intersection-epsilon / grazing cases north_star confines mismatches to.
void vo_brute_force(const vo_scene *s_, const float *o_, const float *d_, float tmin, float tmax, double *out) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    const double o[3] = {o_[0], o_[1], o_[2]}, d[3] = {d_[0], d_[1], d_[2]};
    int any = 0;
    double best = -1.0, margin = 1.0;
#pragma omp parallel
    {
        int l_any = 0;
        double l_best = -1.0, l_margin = 1.0;
#pragma omp for nowait
        for (long long i = 0; i < (long long)s.n_tris; ++i) {
            const float *t = &s.tri[(size_t)i * 9];
            const double v0[3] = {t[0], t[1], t[2]}, e1[3] = {t[3] - v0[0], t[4] - v0[1], t[5] - v0[2]}, e2[3] = {t[6] - v0[0], t[7] - v0[1], t[8] - v0[2]};
            const double pv[3] = {d[1] * e2[2] - d[2] * e2[1], d[2] * e2[0] - d[0] * e2[2], d[0] * e2[1] - d[1] * e2[0]};
            const double det = e1[0] * pv[0] + e1[1] * pv[1] + e1[2] * pv[2];
            if (det == 0.0) continue;
            const double inv = 1.0 / det, tv[3] = {o[0] - v0[0], o[1] - v0[1], o[2] - v0[2]};
            const double u = (tv[0] * pv[0] + tv[1] * pv[1] + tv[2] * pv[2]) * inv;
            const double qv[3] = {tv[1] * e1[2] - tv[2] * e1[1], tv[2] * e1[0] - tv[0] * e1[2], tv[0] * e1[1] - tv[1] * e1[0]};
            const double v = (d[0] * qv[0] + d[1] * qv[1] + d[2] * qv[2]) * inv;
            const double tt = (e2[0] * qv[0] + e2[1] * qv[1] + e2[2] * qv[2]) * inv, w = 1.0 - u - v;
            if (u >= 0 && v >= 0 && w >= 0 && tt > tmin && tt < tmax) { l_any = 1; if (l_best < 0 || tt < l_best) l_best = tt; }
            if (u > -1e-3 && v > -1e-3 && w > -1e-3 && tt > tmin - 1e-3 && tt < tmax + 1e-3) {
                const double bm = std::min(std::min(std::fabs(u), std::fabs(v)), std::fabs(w));
                const double tm = std::min(std::fabs(tt - tmin), std::fabs(tt - tmax)) / std::max(1.0, std::fabs(tt));
                l_margin = std::min(l_margin, std::min(bm, tm));
            }
        }
#pragma omp critical
        {
            any |= l_any;
            if (l_best >= 0 && (best < 0 || l_best < best)) best = l_best;
            margin = std::min(margin, l_margin);
        }
    }
    out[0] = any; out[1] = best; out[2] = margin;
}

// The fully ray-traced render path: raytraced_render_path/raygen.rgen:11-23, closesthit.rchit:10-58, miss.rmiss:6-8,
// shadow_miss.rmiss:6-8; alpha_test != 0 = raygen_test_alpha.rgen / closesthit_test_alpha.rchit / shadow_anyhit.rahit:9-27
// ("Raytracing Pass", src/render_paths/raytraced_render_path.cpp:12-47). Output: "RaytracedOutput", B8G8R8A8_UNORM.
void vo_raytraced(const vo_scene *s_, const PerFrameData *pfd_, int W, int H, int alpha_test, uint8_t *out_bgra8) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    const PerFrameData &pfd = *pfd_;
    auto rahit = [&](uint32_t tri, double hu, double hv) { return rahit_alpha_test(s, s.tri_geom[tri], s.tri_prim[tri], (float)hu, (float)hv); };
    auto opaque = [](uint32_t, double, double) { return true; };
#pragma omp parallel for schedule(dynamic, 1)
    for (int y = 0; y < H; ++y) {
        for (int x = 0; x < W; ++x) {
            vec2 uv_ = {((float)x + 0.5f) / (float)W, ((float)y + 0.5f) / (float)H};
            vec2 uv = {uv_.x * 2.0f - 1.0f, uv_.y * 2.0f - 1.0f};
            vec4 origin = mul44(pfd.camera_view_inverse, vec4{0, 0, 0, 1});
            vec4 target = mul44(pfd.camera_proj_inverse, vec4{uv.x, uv.y, 1, 1});
            vec3 tn = normalize(v3(target.x, target.y, target.z));
            vec4 direction = mul44(pfd.camera_view_inverse, vec4{tn.x, tn.y, tn.z, 0});
            vec4 payload = {0.3f, 0.8f, 0.2f, 1.0f};                                              // miss.rmiss:7
            Hit h;
            bool hit = alpha_test ? trace_closest_filtered(s, v3(origin.x, origin.y, origin.z), v3(direction.x, direction.y, direction.z), 0.1f, 10000.0f, h, rahit)
                                  : trace_closest_filtered(s, v3(origin.x, origin.y, origin.z), v3(direction.x, direction.y, direction.z), 0.1f, 10000.0f, h, opaque);
            if (hit) {
                RaytracedHit r = raytraced_hit(s, s.tri_geom[h.tri], s.tri_prim[h.tri], (float)h.u, (float)h.v);
                vec3 light_dir = -v3(pfd.directional_light.direction[0], pfd.directional_light.direction[1], pfd.directional_light.direction[2]);
                Hit sh;
                bool occluded = alpha_test ? trace_closest_filtered(s, r.position, light_dir, 0.1f, 10000.0f, sh, rahit) : trace_any(s, r.position, light_dir, 0.1f, 10000.0f);
                payload = raytraced_color(pfd, alpha_test, r.albedo, r.N, occluded);
            }
            store_bgra8(out_bgra8 + ((size_t)y * W + x) * 4, payload);
        }
    }
}

// The per-hit code of the passes on hits the caller chooses, kinds and outputs as vhr_debug_shade_hits (include/vhr_b200.h): record i =
// (g, pid, u, v, x, y) as uint32 g, uint32 pid, float u, float v, int32 x, int32 y; 8 words out per record, unwritten words 0. Returns 0,
// or -1 (nothing written) for an unknown kind or a record naming a texture, geometry or triangle that does not exist.
struct ShadeRecord { uint32_t g, pid; float u, v; int32_t x, y; };
int vo_shade_hits(const vo_scene *s_, const PerFrameData *pfd_, int kind, const ShadeRecord *rec, uint32_t n, uint32_t *out) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    const PerFrameData &pfd = *pfd_;
    if (kind < 0 || kind > 6) return -1;
    for (uint32_t i = 0; i < n; ++i) {
        if (kind == 0 ? !has_texture(s, (int)std::min<uint32_t>(rec[i].g, INT32_MAX))
                      : rec[i].g >= s.primitives.size() || rec[i].pid >= s.primitives[rec[i].g].index_count / 3)
            return -1;
    }
    std::memset(out, 0, (size_t)n * 8 * sizeof(uint32_t));
#pragma omp parallel for schedule(static)
    for (long long i = 0; i < (long long)n; ++i) {
        const ShadeRecord &r = rec[i];
        uint32_t *o = out + 8 * i;
        auto put4 = [&](vec4 c) { std::memcpy(o, &c, 16); };
        switch (kind) {
            case 0: put4(sample_texture(s, (int)r.g, vec2{r.u, r.v})); break;
            case 1: put4(reflection_hit(s, pfd, r.g, r.pid, r.u, r.v)); break;
            case 2: {
                uint16_t nrm[4], mot[4];
                float depth;
                gbuffer_hit(s, pfd, r.g, r.pid, r.u, r.v, gbuffer_pixel_uv(pfd, r.x, r.y), reinterpret_cast<uint8_t *>(o), nrm, mot, &depth);
                std::memcpy(o + 1, nrm, 8); std::memcpy(o + 3, mot, 8); std::memcpy(o + 5, &depth, 4);
                break;
            }
            case 3: o[0] = gbuffer_alpha_test(s, r.g, r.pid, r.u, r.v) ? 1u : 0u; break;
            case 4:
            case 5: {
                RaytracedHit t = raytraced_hit(s, r.g, r.pid, r.u, r.v);
                store_bgra8(reinterpret_cast<uint8_t *>(o), raytraced_color(pfd, kind == 5, t.albedo, t.N, false));
                store_bgra8(reinterpret_cast<uint8_t *>(o + 1), raytraced_color(pfd, kind == 5, t.albedo, t.N, true));
                std::memcpy(o + 2, &t.position, 12);
                break;
            }
            case 6: o[0] = rahit_alpha_test(s, r.g, r.pid, r.u, r.v) ? 1u : 0u; break;
        }
    }
    return 0;
}

// G-buffer scaffolding: primary rays through texel centres stand in for the rasteriser of the "G-Buffer Pass"
// (hybrid_render_path.cpp:13-56). Encodings follow gbuf.frag:33,43,46-58; clear values hybrid_render_path.cpp:16-19.
// Also returns the closest-hit record per pixel (tri_geom, tri_prim, t) for debugging when `hit_ids` != NULL.
void vo_gbuffer(const vo_scene *s_, const PerFrameData *pfd_, int W, int H, uint8_t *albedo_bgra8, uint16_t *normals,
                uint16_t *motion, float *depth, int32_t *hit_ids) {
    const Scene &s = *reinterpret_cast<const Scene *>(s_);
    const PerFrameData &pfd = *pfd_;
    vec3 cam = v3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
#pragma omp parallel for schedule(dynamic, 1)
    for (int y = 0; y < H; ++y) {
        for (int x = 0; x < W; ++x) {
            size_t pix = (size_t)y * W + x;
            vec2 uv = gbuffer_pixel_uv(pfd, x, y);
            vec3 pn = get_world_space_position(pfd, 1.0f, uv);   // point on the near plane (reverse-Z: depth 1)
            vec3 dir = pn - cam;
            Hit h;
            auto alpha_test = [&](uint32_t tri, double hu, double hv) { return gbuffer_alpha_test(s, s.tri_geom[tri], s.tri_prim[tri], (float)hu, (float)hv); };
            bool hit = trace_closest_filtered(s, cam, dir, 1.0f, FLT_MAX, h, alpha_test);
            if (hit_ids) { hit_ids[2 * pix] = hit ? (int32_t)s.tri_geom[h.tri] : -1; hit_ids[2 * pix + 1] = hit ? (int32_t)s.tri_prim[h.tri] : -1; }
            if (!hit) {
                if (albedo_bgra8) std::memset(albedo_bgra8 + pix * 4, 0, 4);
                store_rgba16f(normals, W, x, y, vec4{0, 0, 0, 0});
                store_rgba16f(motion, W, x, y, vec4{0, 0, -1.0f, -1.0f});
                depth[pix] = 0.0f;
                continue;
            }
            gbuffer_hit(s, pfd, s.tri_geom[h.tri], s.tri_prim[h.tri], (float)h.u, (float)h.v, uv, albedo_bgra8 ? albedo_bgra8 + pix * 4 : nullptr,
                        normals + pix * 4, motion + pix * 4, depth + pix);
        }
    }
}

}  // extern "C"
