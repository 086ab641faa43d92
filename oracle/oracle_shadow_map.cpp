// oracle/oracle_shadow_map.cpp — TEST INFRASTRUCTURE ONLY. CPU port of the "Shadow Map Pass" (hybrid_render_path.cpp:58-99,
// depth_prepass.vert/.frag) as DESIGN.md §2 "Shadow map" defines it. The reference's pass is fixed-function rasterisation,
// which oracle/_ref cannot compile for the CPU (the shim has no rasteriser stage), so this hand-written port IS the
// specification: the CUDA rasteriser (vulkanhybridrenderer_b200/csrc/shadow_map_kernels.cu) must match it bit for bit.
//
//   vo_shadow_map  <- the world-space triangle soup of vo_scene_create (same transform, same fp32 order), projected by
//                     directional_light.projview; two-sided, no depth bias or clamp; no Y flip; vertices snapped to 1/256 texel;
//                     samples at texel centres, exact integer edge functions, top-left fill rule; depth by fp32 barycentrics
//                     evaluated left to right; 0 <= z <= 1 kept; combined by max (reverse-Z, cleared to 0)
#include "oracle_common.h"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace vo;

namespace {

const float kGuardBand = 1048576.0f;      // 2^20 texels: triangles reaching further are clipped against it in double

struct RasterTri {
    int64_t X[3], Y[3];
    float z[3];
    int64_t A;
    int px0, px1, py0, py1;
};

// round-to-nearest-even of the exact product f * 256 (|f| <= 2^20: exact in float)
int64_t snap(float f) { return (int64_t)std::nearbyint((double)(f * 256.0f)); }

bool raster_setup(const float xf[3], const float yf[3], const float z[3], int W, int H, RasterTri &t) {
    if ((z[0] < 0.0f && z[1] < 0.0f && z[2] < 0.0f) || (z[0] > 1.0f && z[1] > 1.0f && z[2] > 1.0f)) return false;
    for (int k = 0; k < 3; ++k) { t.X[k] = snap(xf[k]); t.Y[k] = snap(yf[k]); t.z[k] = z[k]; }
    int64_t A = (t.X[1] - t.X[0]) * (t.Y[2] - t.Y[0]) - (t.Y[1] - t.Y[0]) * (t.X[2] - t.X[0]);
    if (A == 0) return false;
    if (A < 0) {
        std::swap(t.X[1], t.X[2]); std::swap(t.Y[1], t.Y[2]); std::swap(t.z[1], t.z[2]);
        A = -A;
    }
    t.A = A;
    const int64_t mnx = std::min({t.X[0], t.X[1], t.X[2]}), mxx = std::max({t.X[0], t.X[1], t.X[2]});
    const int64_t mny = std::min({t.Y[0], t.Y[1], t.Y[2]}), mxy = std::max({t.Y[0], t.Y[1], t.Y[2]});
    // texel centres 256 p + 128 within [mn, mx]: p from ceil((mn - 128) / 256) to floor((mx - 128) / 256)
    auto floor_div256 = [](int64_t v) { return v >= 0 ? v / 256 : -((-v + 255) / 256); };
    t.px0 = (int)std::max<int64_t>(0, floor_div256(mnx - 128 + 255));
    t.px1 = (int)std::min<int64_t>(W - 1, floor_div256(mxx - 128));
    t.py0 = (int)std::max<int64_t>(0, floor_div256(mny - 128 + 255));
    t.py1 = (int)std::min<int64_t>(H - 1, floor_div256(mxy - 128));
    return t.px0 <= t.px1 && t.py0 <= t.py1;
}

// top edge (horizontal, left to right) or left edge (going up) of a triangle with A > 0, x right and y = row down
inline bool top_left(int64_t ax, int64_t ay, int64_t bx, int64_t by) { return by - ay < 0 || (by - ay == 0 && bx - ax > 0); }
inline int64_t edge(int64_t ax, int64_t ay, int64_t bx, int64_t by, int64_t sx, int64_t sy) { return (bx - ax) * (sy - ay) - (by - ay) * (sx - ax); }
inline bool inside(int64_t w, bool tl) { return w > 0 || (w == 0 && tl); }

void rasterise_rows(const RasterTri &t, int y0, int y1, int W, float *out) {
    const int ya = std::max(t.py0, y0), yb = std::min(t.py1, y1 - 1);
    const bool tl0 = top_left(t.X[1], t.Y[1], t.X[2], t.Y[2]), tl1 = top_left(t.X[2], t.Y[2], t.X[0], t.Y[0]), tl2 = top_left(t.X[0], t.Y[0], t.X[1], t.Y[1]);
    for (int py = ya; py <= yb; ++py) {
        for (int px = t.px0; px <= t.px1; ++px) {
            const int64_t sx = (int64_t)px * 256 + 128, sy = (int64_t)py * 256 + 128;
            const int64_t w0 = edge(t.X[1], t.Y[1], t.X[2], t.Y[2], sx, sy), w1 = edge(t.X[2], t.Y[2], t.X[0], t.Y[0], sx, sy),
                          w2 = edge(t.X[0], t.Y[0], t.X[1], t.Y[1], sx, sy);
            if (!inside(w0, tl0) || !inside(w1, tl1) || !inside(w2, tl2)) continue;
            const float b1 = (float)w1 / (float)t.A, b2 = (float)w2 / (float)t.A;
            float z = (t.z[0] + b1 * (t.z[1] - t.z[0])) + b2 * (t.z[2] - t.z[0]);
            if (!(z >= 0.0f && z <= 1.0f)) continue;
            if (z == 0.0f) z = 0.0f;                     // -0.0 -> +0.0
            float &d = out[(size_t)py * W + px];
            if (z > d) d = z;                            // GREATER_OR_EQUAL, reverse-Z
        }
    }
}

// Sutherland-Hodgman against x >= -G, x <= G, y >= -G, y <= G in double, (x, y, z) interpolated together
int clip_guard_band(const double in[3][3], double out[9][3]) {
    double a[9][3], b[9][3];
    int n = 3;
    for (int k = 0; k < 3; ++k) for (int c = 0; c < 3; ++c) a[k][c] = in[k][c];
    const double G = kGuardBand;
    for (int plane = 0; plane < 4 && n > 0; ++plane) {
        const int axis = plane >> 1;
        const double s = (plane & 1) ? -1.0 : 1.0;
        int m = 0;
        for (int k = 0; k < n; ++k) {
            const double *u = a[k], *v = a[(k + 1) % n];
            const double du = s * u[axis] + G, dv = s * v[axis] + G;
            if (du >= 0.0) { for (int c = 0; c < 3; ++c) b[m][c] = u[c]; ++m; }
            if ((du >= 0.0) != (dv >= 0.0)) {
                const double t = du / (du - dv);
                for (int c = 0; c < 3; ++c) b[m][c] = u[c] + t * (v[c] - u[c]);
                ++m;
            }
        }
        n = m;
        for (int k = 0; k < n; ++k) for (int c = 0; c < 3; ++c) a[k][c] = b[k][c];
    }
    for (int k = 0; k < n; ++k) for (int c = 0; c < 3; ++c) out[k][c] = a[k][c];
    return n;
}

}  // namespace

extern "C" {

// out: W x H floats (row 0 = NDC y -1). Returns 0, or -1 when projview is not finite or its last row is neither (0, 0, 0, 1) nor
// zero (the library's VHR_ERR_INVALID). A zero last row (no light in the scene) leaves the cleared map.
int vo_shadow_map(const Vertex *vertices, uint32_t n_vertices, const uint32_t *indices, uint32_t n_indices, const Primitive *primitives,
                  uint32_t n_primitives, const PerFrameData *pfd, int W, int H, float *out) {
    (void)n_vertices; (void)n_indices;
    const float *m = pfd->directional_light.projview;
    for (int k = 0; k < 16; ++k)
        if (!std::isfinite(m[k])) return -1;
    const bool affine = m[3] == 0.0f && m[7] == 0.0f && m[11] == 0.0f && m[15] == 1.0f;
    const bool none = m[3] == 0.0f && m[7] == 0.0f && m[11] == 0.0f && m[15] == 0.0f;
    if (!affine && !none) return -1;
    std::fill(out, out + (size_t)W * H, 0.0f);
    if (none) return 0;
    const float hw = 0.5f * (float)W, hh = 0.5f * (float)H;
    std::vector<RasterTri> tris;
    for (uint32_t g = 0; g < n_primitives; ++g) {
        const Primitive &p = primitives[g];
        for (uint32_t k = 0; k < p.index_count / 3; ++k) {
            float xf[3], yf[3], z[3];
            bool in_band = true, finite = true;
            for (int c = 0; c < 3; ++c) {
                const float *v = vertices[p.vertex_offset + indices[p.index_offset + 3 * k + c]].pos;
                float w[3];
                for (int r = 0; r < 3; ++r) w[r] = ((p.transform[0 * 4 + r] * v[0] + p.transform[1 * 4 + r] * v[1]) + p.transform[2 * 4 + r] * v[2]) + p.transform[3 * 4 + r];
                const vec4 clip = mul44(m, vec4{w[0], w[1], w[2], 1.0f});     // w = 1 for an affine projview
                xf[c] = hw * clip.x + hw;
                yf[c] = hh * clip.y + hh;
                z[c] = clip.z;
                in_band = in_band && std::fabs(xf[c]) <= kGuardBand && std::fabs(yf[c]) <= kGuardBand;
                finite = finite && std::isfinite(xf[c]) && std::isfinite(yf[c]) && std::isfinite(z[c]);
            }
            RasterTri t;
            if (in_band) {
                if (raster_setup(xf, yf, z, W, H, t)) tris.push_back(t);
                continue;
            }
            if (!finite) continue;
            double in[3][3], poly[9][3];
            for (int c = 0; c < 3; ++c) { in[c][0] = xf[c]; in[c][1] = yf[c]; in[c][2] = z[c]; }
            const int n = clip_guard_band(in, poly);
            for (int f = 1; f + 1 < n; ++f) {       // fan (q0, q_f, q_f+1)
                const float sx[3] = {(float)poly[0][0], (float)poly[f][0], (float)poly[f + 1][0]};
                const float sy[3] = {(float)poly[0][1], (float)poly[f][1], (float)poly[f + 1][1]};
                const float sz[3] = {(float)poly[0][2], (float)poly[f][2], (float)poly[f + 1][2]};
                if (raster_setup(sx, sy, sz, W, H, t)) tris.push_back(t);
            }
        }
    }
    // bands of rows in parallel: every band sees every triangle in the same order, so the result does not depend on the threads
    const int band = 16;
#pragma omp parallel for schedule(dynamic, 1)
    for (int y0 = 0; y0 < H; y0 += band)
        for (const RasterTri &t : tris)
            if (t.py1 >= y0 && t.py0 < y0 + band) rasterise_rows(t, y0, std::min(H, y0 + band), W, out);
    return 0;
}

}  // extern "C"
