// shadow_map_kernels.cu — the "Shadow Map Pass" (hybrid_render_path.cpp:58-99, depth_prepass.vert/.frag) as a CUDA depth
// rasteriser (sm_100a): the world-space triangle soup of the BVH build, projected by directional_light.projview, into a D32
// map combined by max (reverse-Z, GREATER_OR_EQUAL, cleared to 0). Semantics: DESIGN.md §2 "Shadow map"; oracle/oracle_shadow_map.cpp
// restates them on the CPU and the kernels match it bit for bit.
//
// Every covered sample's depth is a pure function of the triangle and the sample, and the combine is an integer max on the bit
// patterns of non-negative floats, so the map does not depend on the order in which triangles or tiles are processed.
//
//   1. cudaMemsetAsync clears the map.
//   2. shadow_setup_kernel, one thread per triangle: project, snap, cull; a triangle whose bounding box holds at most
//      kSmallSamples texel centres is rasterised by its thread; a larger one stores a record and counts its 8 x 8 tiles; one
//      that reaches beyond the guard band goes to the clip list.
//   3. cub::DeviceScan::ExclusiveSum over the tile counts.
//   4. shadow_tile_kernel, one warp per (triangle, tile) item, 2 samples per lane.
//   5. shadow_clip_kernel, one block per triangle of the clip list (rare): clip against the guard band in double, rasterise the fan.
//
// Under a partition (world > 1, the map attached for every other rank) the map's rows are dealt in blocks of kTile rows, block b to
// rank b % world. Each rank projects every triangle but shades only the samples of its own rows (the <true> instances), then
// shadow_push_kernel stores those rows into the same rows of every other rank's map: every rank ends with the whole map, bit for bit
// the single-GPU one, because each texel is a max over triangles of a function of the triangle and the texel alone.
#include <cmath>
#include <type_traits>

#include <cub/cub.cuh>

#include "vhr_internal.h"

namespace vhr {

// kernels and helpers live in namespace vhr (not an anonymous one) so that their names in a profile are stable
constexpr float kGuardBand = 1048576.0f;      // 2^20 texels on each side of the map's origin
constexpr int kSmallSamples = 16;             // bounding boxes of at most this many texel centres: rasterised by the setup thread
constexpr int kTile = 8;                      // tile edge (texels) of the tile kernel's work items

// One triangle ready to rasterise: vertices snapped to 1/256 texel, oriented so that the doubled area A is positive.
struct RasterTri {
    int64_t X[3], Y[3];
    float z[3];
    int64_t A;
    int px0, px1, py0, py1;       // texel range of the bounding box, clamped to the map (empty: px0 > px1 or py0 > py1)
};

// 48-byte record of a large triangle for the tile kernel
struct TileRecord {
    int32_t X[3], Y[3];
    float z[3];
    uint32_t tx0, ty0, ntx;
};
static_assert(sizeof(TileRecord) == 48, "TileRecord layout");

__device__ __forceinline__ int64_t min2(int64_t a, int64_t b) { return a < b ? a : b; }
__device__ __forceinline__ int64_t max2(int64_t a, int64_t b) { return a > b ? a : b; }
__device__ __forceinline__ int64_t min3(int64_t a, int64_t b, int64_t c) { return min2(a, min2(b, c)); }
__device__ __forceinline__ int64_t max3(int64_t a, int64_t b, int64_t c) { return max2(a, max2(b, c)); }
__device__ __forceinline__ int64_t snap(float f) { return __float2ll_rn(mul_rn(f, 256.0f)); }

// false: the triangle draws nothing (all depths on one side of [0, 1], zero area, or no texel centre inside its box)
__device__ __forceinline__ bool raster_setup(const float xf[3], const float yf[3], const float zin[3], int W, int H, RasterTri &t) {
    if ((zin[0] < 0.0f && zin[1] < 0.0f && zin[2] < 0.0f) || (zin[0] > 1.0f && zin[1] > 1.0f && zin[2] > 1.0f)) return false;
    for (int k = 0; k < 3; ++k) { t.X[k] = snap(xf[k]); t.Y[k] = snap(yf[k]); t.z[k] = zin[k]; }
    int64_t A = (t.X[1] - t.X[0]) * (t.Y[2] - t.Y[0]) - (t.Y[1] - t.Y[0]) * (t.X[2] - t.X[0]);
    if (A == 0) return false;
    if (A < 0) {      // both windings are drawn (no culling): exchange vertices 1 and 2
        int64_t x = t.X[1], y = t.Y[1];
        float z = t.z[1];
        t.X[1] = t.X[2]; t.Y[1] = t.Y[2]; t.z[1] = t.z[2];
        t.X[2] = x; t.Y[2] = y; t.z[2] = z;
        A = -A;
    }
    t.A = A;
    const int64_t mnx = min3(t.X[0], t.X[1], t.X[2]), mxx = max3(t.X[0], t.X[1], t.X[2]);
    const int64_t mny = min3(t.Y[0], t.Y[1], t.Y[2]), mxy = max3(t.Y[0], t.Y[1], t.Y[2]);
    // texel centres 256 p + 128 inside [mn, mx] (>> 8 of a negative value rounds down)
    t.px0 = (int)max2(0, (mnx - 128 + 255) >> 8);
    t.px1 = (int)min2(W - 1, (mxx - 128) >> 8);
    t.py0 = (int)max2(0, (mny - 128 + 255) >> 8);
    t.py1 = (int)min2(H - 1, (mxy - 128) >> 8);
    return t.px0 <= t.px1 && t.py0 <= t.py1;
}

// edge a -> b of a triangle with A > 0 in the map's frame (x right, y = row down): top (horizontal, left to right) or left (upward)
__device__ __forceinline__ int64_t tie_bias(int64_t ax, int64_t ay, int64_t bx, int64_t by) {
    const int64_t dx = bx - ax, dy = by - ay;
    return (dy < 0 || (dy == 0 && dx > 0)) ? 0 : 1;
}
__device__ __forceinline__ int64_t edge(int64_t ax, int64_t ay, int64_t bx, int64_t by, int64_t sx, int64_t sy) {
    return (bx - ax) * (sy - ay) - (by - ay) * (sx - ax);
}

// depth of sample (px, py) if it is covered and in [0, 1]; else nothing. Atomic max on the bit pattern (non-negative floats).
__device__ __forceinline__ void shade_sample(const int64_t X[3], const int64_t Y[3], const float z[3], int64_t A, int px, int py,
                                             uint32_t *__restrict__ map, int W) {
    const int64_t sx = (int64_t)px * 256 + 128, sy = (int64_t)py * 256 + 128;
    const int64_t w0 = edge(X[1], Y[1], X[2], Y[2], sx, sy), w1 = edge(X[2], Y[2], X[0], Y[0], sx, sy), w2 = edge(X[0], Y[0], X[1], Y[1], sx, sy);
    if (w0 - tie_bias(X[1], Y[1], X[2], Y[2]) < 0 || w1 - tie_bias(X[2], Y[2], X[0], Y[0]) < 0 || w2 - tie_bias(X[0], Y[0], X[1], Y[1]) < 0) return;
    const float fa = __ll2float_rn(A);
    const float b1 = __fdiv_rn(__ll2float_rn(w1), fa), b2 = __fdiv_rn(__ll2float_rn(w2), fa);
    const float d = add_rn(add_rn(z[0], mul_rn(b1, sub_rn(z[1], z[0]))), mul_rn(b2, sub_rn(z[2], z[0])));
    if (!(d >= 0.0f && d <= 1.0f)) return;
    const uint32_t bits = d == 0.0f ? 0u : __float_as_uint(d);       // -0.0 -> +0.0
    if (bits) atomicMax(&map[(size_t)py * W + px], bits);            // 0 is the clear value: nothing to combine
}

struct ShadowParams {
    const float4 *tri_verts;
    uint32_t n_tris;
    float pv[12];                 // rows 0..2 of projview, column-major (m[c * 4 + r]); row 3 is (0, 0, 0, 1)
    int W, H;
    uint32_t *map;
    uint64_t *counts;             // n_tris + 1 tile counts (the last one 0); 64-bit so that their sum cannot wrap
    TileRecord *records;
    uint32_t *clip_list;          // [0] = count, then triangle indices
};
// partitioned instances: this rank shades only the samples of the map rows it owns
struct ShadowPartParams : ShadowParams {
    int world, rank;
};

// The one definition of row ownership under a partition: tile row ty (map rows [kTile ty, kTile ty + kTile)) belongs to rank
// ty % world. Interleaved rather than banded because coverage is concentrated in the middle of the map.
__host__ __device__ __forceinline__ bool owns_tile_row(int ty, int world, int rank) { return (uint32_t)ty % (uint32_t)world == (uint32_t)rank; }
__device__ __forceinline__ bool owns_row(int py, int world, int rank) { return owns_tile_row(py / kTile, world, rank); }
// the first tile row >= ty this rank owns
__device__ __forceinline__ int first_owned_tile_row(int ty, int world, int rank) {
    for (int k = 1; k < world && !owns_tile_row(ty, world, rank); ++k) ++ty;
    return ty;
}

// viewport transform of one world-space vertex: no Y flip (SURVEY Q24), x_ndc = clip x (w = 1)
__device__ __forceinline__ void project(const ShadowParams &p, float4 v, float &xf, float &yf, float &z) {
    const float *m = p.pv;        // m[c * 3 + r]
    const float x = dot4_rn(m[0], v.x, m[3], v.y, m[6], v.z, m[9], 1.0f);
    const float y = dot4_rn(m[1], v.x, m[4], v.y, m[7], v.z, m[10], 1.0f);
    z = dot4_rn(m[2], v.x, m[5], v.y, m[8], v.z, m[11], 1.0f);
    const float hw = 0.5f * (float)p.W, hh = 0.5f * (float)p.H;
    xf = add_rn(mul_rn(hw, x), hw);
    yf = add_rn(mul_rn(hh, y), hh);
}

// PART = false: the single-GPU pass, every sample of the map. PART = true (ShadowPartParams): only the samples of owned rows; a large
// triangle counts its tiles in owned tile rows and records the first of them (the tile kernel steps by world tile rows).
template <bool PART>
__global__ void __launch_bounds__(256) shadow_setup_kernel(const __grid_constant__ std::conditional_t<PART, ShadowPartParams, ShadowParams> p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > p.n_tris) return;
    if (i == p.n_tris) { p.counts[i] = 0; return; }
    uint64_t count = 0;
    float xf[3], yf[3], z[3];
    bool inside = true, finite = true;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        project(p, p.tri_verts[3 * (size_t)i + k], xf[k], yf[k], z[k]);
        inside = inside && fabsf(xf[k]) <= kGuardBand && fabsf(yf[k]) <= kGuardBand;
        finite = finite && isfinite(xf[k]) && isfinite(yf[k]) && isfinite(z[k]);
    }
    if (!inside) {
        if (finite) p.clip_list[1 + atomicAdd(&p.clip_list[0], 1u)] = i;
    } else {
        RasterTri t;
        if (raster_setup(xf, yf, z, p.W, p.H, t)) {
            const int nx = t.px1 - t.px0 + 1, ny = t.py1 - t.py0 + 1;
            if ((int64_t)nx * ny <= kSmallSamples) {
                if constexpr (PART) {      // the rows of owned tile rows only
                    for (int ty = first_owned_tile_row(t.py0 / kTile, p.world, p.rank); ty * kTile <= t.py1; ty += p.world)
                        for (int py = max(t.py0, ty * kTile); py <= min(t.py1, ty * kTile + kTile - 1); ++py)
                            for (int px = t.px0; px <= t.px1; ++px) shade_sample(t.X, t.Y, t.z, t.A, px, py, p.map, p.W);
                } else {
                    for (int py = t.py0; py <= t.py1; ++py)
                        for (int px = t.px0; px <= t.px1; ++px) shade_sample(t.X, t.Y, t.z, t.A, px, py, p.map, p.W);
                }
            } else {
                TileRecord r;
                for (int k = 0; k < 3; ++k) { r.X[k] = (int32_t)t.X[k]; r.Y[k] = (int32_t)t.Y[k]; r.z[k] = t.z[k]; }
                r.tx0 = (uint32_t)t.px0 / kTile; r.ty0 = (uint32_t)t.py0 / kTile;
                r.ntx = (uint32_t)t.px1 / kTile - r.tx0 + 1;
                if constexpr (PART) {
                    const int ty1 = t.py1 / kTile, ty = first_owned_tile_row((int)r.ty0, p.world, p.rank);
                    r.ty0 = (uint32_t)ty;
                    count = ty <= ty1 ? (uint64_t)r.ntx * (uint32_t)((ty1 - ty) / p.world + 1) : 0;
                } else {
                    count = (uint64_t)r.ntx * ((uint32_t)t.py1 / kTile - r.ty0 + 1);
                }
                p.records[i] = r;
            }
        }
    }
    p.counts[i] = count;
}

// Persistent warps over the scanned items: item k belongs to the last triangle whose offset is <= k. PART: the items of a triangle
// are its tiles in owned tile rows, which are world tile rows apart from the record's first one (`world` is unused otherwise).
template <bool PART>
__global__ void __launch_bounds__(256) shadow_tile_kernel(const uint64_t *__restrict__ offsets, const TileRecord *__restrict__ records,
                                                          uint32_t n_tris, uint32_t *__restrict__ map, int W, int H, int world) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint64_t total = offsets[n_tris];
    for (uint64_t item = warp; item < total; item += n_warps) {
        uint32_t lo = 0, hi = n_tris;           // offsets[lo] <= item < offsets[hi]
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(&offsets[mid]) <= item) lo = mid; else hi = mid;
        }
        const TileRecord r = records[lo];
        const uint32_t local = (uint32_t)(item - __ldg(&offsets[lo]));
        const int tx = (int)(r.tx0 + local % r.ntx);
        const int ty = PART ? (int)(r.ty0 + (local / r.ntx) * (uint32_t)world) : (int)(r.ty0 + local / r.ntx);
        const int64_t X[3] = {r.X[0], r.X[1], r.X[2]}, Y[3] = {r.Y[0], r.Y[1], r.Y[2]};
        const int64_t A = (X[1] - X[0]) * (Y[2] - Y[0]) - (Y[1] - Y[0]) * (X[2] - X[0]);
        const int px = tx * kTile + (int)(lane & 7u);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int py = ty * kTile + (int)(lane >> 3) + 4 * h;
            if (px < W && py < H) shade_sample(X, Y, r.z, A, px, py, map, W);
        }
    }
}

// Sutherland-Hodgman against |x| <= G, |y| <= G in double (xf, yf, z interpolated together); returns the polygon's vertex count
__device__ int clip_guard_band(const double in[3][3], double out[9][3]) {
    double a[9][3], b[9][3];
    int n = 3;
    for (int k = 0; k < 3; ++k) for (int c = 0; c < 3; ++c) a[k][c] = in[k][c];
    const double G = (double)kGuardBand;
    for (int plane = 0; plane < 4; ++plane) {
        const int axis = plane >> 1;
        const double s = (plane & 1) ? -1.0 : 1.0;        // distance s * v[axis] + G >= 0 is inside
        int m = 0;
        for (int k = 0; k < n; ++k) {
            const double *u = a[k], *v = a[(k + 1) % n];
            const double du = __dadd_rn(s * u[axis], G), dv = __dadd_rn(s * v[axis], G);
            if (du >= 0.0) { for (int c = 0; c < 3; ++c) b[m][c] = u[c]; ++m; }
            if ((du >= 0.0) != (dv >= 0.0)) {
                const double t = __ddiv_rn(du, __dsub_rn(du, dv));
                for (int c = 0; c < 3; ++c) b[m][c] = __dadd_rn(u[c], __dmul_rn(t, __dsub_rn(v[c], u[c])));      // no FMA: the oracle's rounding
                ++m;
            }
        }
        n = m;
        for (int k = 0; k < n; ++k) for (int c = 0; c < 3; ++c) a[k][c] = b[k][c];
        if (n == 0) break;
    }
    for (int k = 0; k < n; ++k) for (int c = 0; c < 3; ++c) out[k][c] = a[k][c];
    return n;
}

template <bool PART>
__global__ void __launch_bounds__(256) shadow_clip_kernel(const __grid_constant__ std::conditional_t<PART, ShadowPartParams, ShadowParams> p) {
    __shared__ float poly[9][3];
    __shared__ int n_poly;
    const uint32_t n_clip = p.clip_list[0];
    for (uint32_t c = blockIdx.x; c < n_clip; c += gridDim.x) {
        if (threadIdx.x == 0) {
            const uint32_t i = p.clip_list[1 + c];
            double in[3][3], out[9][3];
            for (int k = 0; k < 3; ++k) {
                float xf, yf, z;
                project(p, p.tri_verts[3 * (size_t)i + k], xf, yf, z);
                in[k][0] = xf; in[k][1] = yf; in[k][2] = z;
            }
            n_poly = clip_guard_band(in, out);
            for (int k = 0; k < n_poly; ++k) for (int e = 0; e < 3; ++e) poly[k][e] = (float)out[k][e];
        }
        __syncthreads();
        for (int f = 1; f + 1 < n_poly; ++f) {      // fan (q0, q_f, q_f+1)
            const float xf[3] = {poly[0][0], poly[f][0], poly[f + 1][0]}, yf[3] = {poly[0][1], poly[f][1], poly[f + 1][1]};
            const float z[3] = {poly[0][2], poly[f][2], poly[f + 1][2]};
            RasterTri t;
            if (!raster_setup(xf, yf, z, p.W, p.H, t)) continue;
            const int nx = t.px1 - t.px0 + 1;
            const int64_t ns = (int64_t)nx * (t.py1 - t.py0 + 1);
            for (int64_t s = threadIdx.x; s < ns; s += blockDim.x) {
                const int py = t.py0 + (int)(s / nx);
                if constexpr (PART)
                    if (!owns_row(py, p.world, p.rank)) continue;
                shade_sample(t.X, t.Y, t.z, t.A, t.px0 + (int)(s % nx), py, p.map, p.W);
            }
        }
        __syncthreads();
    }
}

// Partitioned pass, after rasterisation (a texel is final only once every triangle has been combined into it): the texels of this
// rank's tile rows go to the same texels of every other rank's map. Tile row ty is the contiguous span [kTile ty W, min(kTile ty +
// kTile, H) W) of texels; with vec (every map's base 16-byte aligned) its aligned middle moves in 16-byte words, its ends texel by texel.
struct ShadowPushParams {
    const uint32_t *map;
    uint32_t *map_of[VHR_MAX_RANKS];      // [r] = rank r's map; this rank's own entry is not used
    int W, H, world, rank, vec;
};

// blockIdx.y counts the rank's own tile rows: the first one, then every world-th.
__global__ void __launch_bounds__(256) shadow_push_kernel(const __grid_constant__ ShadowPushParams p) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    const int n_ty = (p.H + kTile - 1) / kTile;
    for (int ty = first_owned_tile_row(0, p.world, p.rank) + (int)blockIdx.y * p.world; ty < n_ty; ty += (int)gridDim.y * p.world) {
        const size_t begin = (size_t)ty * kTile * p.W, end = (size_t)min(ty * kTile + kTile, p.H) * p.W;
        const size_t a = p.vec ? min((begin + 3) & ~(size_t)3, end) : end;       // [begin, a) and [b, end): single texels
        const size_t b = p.vec ? max(a, end & ~(size_t)3) : end;
        for (size_t k = a / 4 + t; k < b / 4; k += stride) {
            const uint4 v = reinterpret_cast<const uint4 *>(p.map)[k];
#pragma unroll
            for (int r = 0; r < VHR_MAX_RANKS; ++r)
                if (r < p.world && r != p.rank) reinterpret_cast<uint4 *>(p.map_of[r])[k] = v;
        }
        for (size_t i = begin + t; i < a; i += stride) {
            const uint32_t v = p.map[i];
#pragma unroll
            for (int r = 0; r < VHR_MAX_RANKS; ++r)
                if (r < p.world && r != p.rank) p.map_of[r][i] = v;
        }
        for (size_t i = b + t; i < end; i += stride) {
            const uint32_t v = p.map[i];
#pragma unroll
            for (int r = 0; r < VHR_MAX_RANKS; ++r)
                if (r < p.world && r != p.rank) p.map_of[r][i] = v;
        }
    }
}

// Scratch buffers grow to the largest scene seen and stay with the context; a buffer is replaced only after the work that uses it.
// Replicated pass: the stream is synchronised and the old buffer freed (with every buffer retired earlier). Partitioned pass
// (`retire`): nothing here may synchronise the device, because with ranks driven by this thread an earlier rank's stream may
// already wait for this rank's signal, which is enqueued only after this call; cudaFree would wait for that stream. The old buffer
// is kept in `retired` instead, until a replicated pass grows a buffer or the context is destroyed.
static int grow(vhr_context *ctx, void *&buf, size_t &have, size_t need_bytes, bool retire) {
    if (buf && have >= need_bytes) return VHR_OK;
    ShadowScratch &s = ctx->shadow;
    if (buf && retire) {
        s.retired.push_back(buf);
    } else if (buf) {
        VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        cudaFree(buf);
        for (void *b : s.retired) cudaFree(b);
        s.retired.clear();
    }
    buf = nullptr; have = 0;
    VHR_CUDA_CHECK(cudaMalloc(&buf, std::max<size_t>(need_bytes, 16)));
    have = need_bytes;
    return VHR_OK;
}

// scratch for n triangles; scan_bytes = what CUB's scan of n + 1 counts needs
static int grow_scratch(vhr_context *ctx, uint32_t n, size_t &scan_bytes, bool retire) {
    ShadowScratch &s = ctx->shadow;
    if (int rc = grow(ctx, s.counts, s.counts_bytes, ((size_t)n + 1) * sizeof(uint64_t), retire)) return rc;
    if (int rc = grow(ctx, s.offsets, s.offsets_bytes, ((size_t)n + 1) * sizeof(uint64_t), retire)) return rc;
    if (int rc = grow(ctx, s.clip_list, s.clip_list_bytes, ((size_t)n + 1) * sizeof(uint32_t), retire)) return rc;
    if (int rc = grow(ctx, s.records, s.records_bytes, (size_t)n * sizeof(TileRecord), retire)) return rc;
    scan_bytes = 0;
    VHR_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (uint64_t *)s.counts, (uint64_t *)s.offsets, (int)n + 1, ctx->stream));
    if (int rc = grow(ctx, s.scan_tmp, s.scan_tmp_bytes, scan_bytes, retire)) return rc;
    if (!s.sms) VHR_CUDA_CHECK(cudaDeviceGetAttribute(&s.sms, cudaDevAttrMultiProcessorCount, ctx->device));
    return VHR_OK;
}

static void fill_params(vhr_context *ctx, Image *map, const float *m, uint32_t n, ShadowParams &p) {
    ShadowScratch &s = ctx->shadow;
    p.tri_verts = ctx->bvh.tri_verts;
    p.n_tris = n;
    for (int c = 0; c < 4; ++c)
        for (int r = 0; r < 3; ++r) p.pv[c * 3 + r] = m[c * 4 + r];
    p.W = (int)map->width; p.H = (int)map->height;
    p.map = (uint32_t *)map->ptr;
    p.counts = (uint64_t *)s.counts;
    p.records = (TileRecord *)s.records;
    p.clip_list = (uint32_t *)s.clip_list;
}

// setup, scan, tile and clip kernels over the n > 0 triangles into the cleared map (the instance PART selects)
template <bool PART>
static int rasterise(vhr_context *ctx, const std::conditional_t<PART, ShadowPartParams, ShadowParams> &p, size_t scan_bytes) {
    ShadowScratch &s = ctx->shadow;
    const uint32_t n = p.n_tris;
    uint64_t *offsets = (uint64_t *)s.offsets;
    int world = 1;
    if constexpr (PART) world = p.world;
    VHR_CUDA_CHECK(cudaMemsetAsync(p.clip_list, 0, sizeof(uint32_t), ctx->stream));
    shadow_setup_kernel<PART><<<(n + 256) / 256, 256, 0, ctx->stream>>>(p);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    VHR_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(s.scan_tmp, scan_bytes, p.counts, offsets, (int)n + 1, ctx->stream));
    ctx->launches += 2;      // CUB single-pass scan: init + scan kernels
    shadow_tile_kernel<PART><<<s.sms * 8, 256, 0, ctx->stream>>>(offsets, p.records, n, p.map, p.W, p.H, world);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    shadow_clip_kernel<PART><<<s.sms, 256, 0, ctx->stream>>>(p);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

// Partitioned pass (include/vhr_b200.h): wait for every rank, clear this rank's rows, rasterise them, push them to every rank, wait.
static int launch_shadow_map_partitioned(vhr_context *ctx, Image *map, const float *m, uint32_t n) {
    const Partition &pt = ctx->part;
    ShadowScratch &s = ctx->shadow;
    size_t scan_bytes = 0;
    if (int rc = grow_scratch(ctx, n, scan_bytes, true)) return rc;
    ShadowPartParams p;
    fill_params(ctx, map, m, n, p);
    p.world = pt.world; p.rank = pt.rank;
    ShadowPushParams q;
    q.map = p.map;
    q.W = p.W; q.H = p.H; q.world = pt.world; q.rank = pt.rank;
    uintptr_t bits = (uintptr_t)map->ptr;
    for (int r = 0; r < pt.world; ++r) {
        q.map_of[r] = r == pt.rank ? nullptr : (uint32_t *)map->peer[r];
        bits |= (uintptr_t)q.map_of[r];
    }
    q.vec = (bits & 15) == 0;
    // Load every kernel this call launches before a flag wait is enqueued: with lazy module loading a first launch would otherwise
    // wait for this stream, which then waits for the other ranks — a deadlock when they are contexts driven by this same thread and
    // have not issued their signals yet. CUB's scan kernels have no handle to load them by: one scan of one count loads them (the
    // offsets it writes are rewritten before they are read).
    static uint64_t loaded = 0;
    if (!(loaded >> (ctx->device & 63) & 1ull)) {
        cudaFuncAttributes attr;
        VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, shadow_setup_kernel<true>));
        VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, shadow_tile_kernel<true>));
        VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, shadow_clip_kernel<true>));
        VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, shadow_push_kernel));
        VHR_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(s.scan_tmp, scan_bytes, p.counts, (uint64_t *)s.offsets, 1, ctx->stream));
        ctx->launches += 2;
        loaded |= 1ull << (ctx->device & 63);
    }
    // WAR on the peers' maps: a peer's composition of the previous frame may still be reading any texel of its map
    if (int rc = peer_sync_all(ctx)) return rc;
    // clear this rank's rows only: a peer that is ahead may already have pushed its rows of this frame into this map
    const size_t row_bytes = (size_t)p.W * sizeof(uint32_t);
    const int n_ty = (p.H + kTile - 1) / kTile, full = p.H / kTile;      // tile rows; those with all kTile rows
    const int n_full_owned = full > pt.rank ? (full - pt.rank + pt.world - 1) / pt.world : 0;       // tile rows rank, rank + world, ...
    if (n_full_owned > 0)
        VHR_CUDA_CHECK(cudaMemset2DAsync((char *)map->ptr + (size_t)pt.rank * kTile * row_bytes, (size_t)pt.world * kTile * row_bytes, 0,
                                         kTile * row_bytes, n_full_owned, ctx->stream));
    if (full < n_ty && owns_tile_row(full, pt.world, pt.rank))      // the last, partial tile row
        VHR_CUDA_CHECK(cudaMemsetAsync((char *)map->ptr + (size_t)full * kTile * row_bytes, 0, (size_t)(p.H - full * kTile) * row_bytes, ctx->stream));
    if (n > 0)
        if (int rc = rasterise<true>(ctx, p, scan_bytes)) return rc;
    const int n_owned = (n_ty - pt.rank + pt.world - 1) / pt.world;      // tile rows rank, rank + world, ... below n_ty
    if (n_owned > 0) {      // the rank owns a tile row (the cleared ones too: the peers' copies hold the previous frame)
        dim3 grid((unsigned)std::min<size_t>(((size_t)kTile * p.W / 4 + 255) / 256, 1024), (unsigned)std::min(n_owned, 65535));
        shadow_push_kernel<<<grid, 256, 0, ctx->stream>>>(q);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
    }
    return peer_sync_all(ctx);      // every rank's rows have landed before SSAO, SSR or composition read the map
}

int launch_shadow_map(vhr_context *ctx) {
    if (ctx->n_bound < 1 || !ctx->bound[0]) return fail(VHR_ERR_STATE, "Shadow Map Pass: image 0 (the shadow map) is not bound");
    Image *map = ctx->bound[0];
    if (map->format != VHR_FORMAT_D32_SFLOAT) return fail(VHR_ERR_INVALID, "Shadow Map Pass: image 0 has format %d, expected D32_SFLOAT (126)", map->format);
    const float *m = ctx->pfd.directional_light.projview;
    for (int k = 0; k < 16; ++k)
        if (!std::isfinite(m[k])) return fail(VHR_ERR_INVALID, "Shadow Map Pass: directional_light.projview[%d] is not finite", k);
    const bool affine = m[3] == 0.0f && m[7] == 0.0f && m[11] == 0.0f && m[15] == 1.0f;
    const bool no_light = m[3] == 0.0f && m[7] == 0.0f && m[11] == 0.0f && m[15] == 0.0f;
    if (!affine && !no_light)
        return fail(VHR_ERR_INVALID, "Shadow Map Pass: projview's last row (%g, %g, %g, %g) is neither (0, 0, 0, 1) (orthographic light) nor zero (no light)",
                    m[3], m[7], m[11], m[15]);
    // Under a partition the map's attachments decide: attached for every other rank, the pass runs partitioned; for none, every rank
    // renders the whole map; for some, the call fails before any flag word is written or waited on.
    const Partition &pt = ctx->part;
    bool partitioned = false;
    if (pt.enabled && pt.world > 1) {
        int attached = 0, missing = -1;
        for (int r = 0; r < pt.world; ++r)
            if (r != pt.rank) {
                if (map->peer[r]) ++attached;
                else if (missing < 0) missing = r;
            }
        if (attached > 0 && missing >= 0)
            return fail(VHR_ERR_STATE, "Shadow Map Pass: binding 0 (%s) has no image of rank %d attached (vhr_image_attach_peer)",
                        image_label(ctx, map).c_str(), missing);
        partitioned = attached > 0;
    }
    if (int rc = make_writable(ctx, map, true)) return rc;
    const uint32_t n = ctx->bvh.n_tris;
    if (partitioned) return launch_shadow_map_partitioned(ctx, map, m, no_light ? 0 : n);
    VHR_CUDA_CHECK(cudaMemsetAsync(map->ptr, 0, map->bytes, ctx->stream));
    if (no_light || n == 0) return VHR_OK;      // every vertex has w = 0 (clipped) / nothing to draw: the cleared map

    size_t scan_bytes = 0;
    if (int rc = grow_scratch(ctx, n, scan_bytes, false)) return rc;
    ShadowParams p;
    fill_params(ctx, map, m, n, p);
    return rasterise<false>(ctx, p, scan_bytes);
}

void free_shadow_scratch(vhr_context *ctx) {
    ShadowScratch &s = ctx->shadow;
    for (void *b : {s.counts, s.offsets, s.clip_list, s.records, s.scan_tmp})
        if (b) cudaFree(b);
    for (void *b : s.retired) cudaFree(b);
    s = ShadowScratch();
}

}  // namespace vhr
