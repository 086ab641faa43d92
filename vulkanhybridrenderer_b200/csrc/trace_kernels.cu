// trace_kernels.cu — software ray traversal over the 8-wide quantised BVH and the ray-traced passes (sm_100a).
//
//   raygen_kernel   <- /root/reference/data/shaders/hybrid_render_path/raygen.rgen:14-66, miss.rmiss:6-8,
//                      reflection_miss.rmiss:6-8, reflection_hit.rchit:10-72 (one thread per pixel; the ray buffer
//                      is never materialised)
//   gbuffer_kernel  <- G-buffer encodings of gbuf.vert:19-28 / gbuf.frag:33,43,46-58 with primary rays standing in
//                      for the rasteriser ("G-Buffer Pass", hybrid_render_path.cpp:13-56)
//   trace_explicit  <- test/debug entry: explicit rays, any-hit or closest-hit
//
// traceRayEXT semantics restated from the Vulkan ray-tracing spec (the reference's traversal lives in the driver):
// opaque triangles, no culling (TLAS instance flag TRIANGLE_FACING_CULL_DISABLE, resource_manager.cpp:704-718),
// a triangle counts when tMin < t < tMax, shared edges are watertight (Woop/Benthin/Wald 2013 with the double
// fallback for zero edge functions).
#include <stdlib.h>

#include <algorithm>
#include <type_traits>
#include <vector>

#include "bvh.cuh"
#include "vhr_internal.h"

namespace vhr {

namespace {

struct Ray {
    float3 o, d;
    float tmin, tmax;
};

struct RayPre {
    float3 o;
    float3 idir;          // 1/d with zero components replaced by a huge finite value
    int kx, ky, kz;       // Woop permutation
    float Sx, Sy, Sz;
    uint32_t neg;         // bit a set: d[a] < 0
};

// MUFU.RCP (1 ulp): traversal set-up and hit distances are compared with an exact oracle under a tolerance, so the
// IEEE division's slow path (a CALL per use) buys nothing here.
__device__ __forceinline__ float rcp_fast(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float comp(float3 v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }
__device__ __forceinline__ float comp4(float4 v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }

__device__ __forceinline__ RayPre prepare(const Ray &r) {
    RayPre p;
    p.o = r.o;
    float3 d = r.d;
    const float tiny = 1e-30f;
    float dx = fabsf(d.x) < tiny ? copysignf(tiny, d.x) : d.x;
    float dy = fabsf(d.y) < tiny ? copysignf(tiny, d.y) : d.y;
    float dz = fabsf(d.z) < tiny ? copysignf(tiny, d.z) : d.z;
    p.idir = make_float3(rcp_fast(dx), rcp_fast(dy), rcp_fast(dz));
    // sign of the *adjusted* component: -0.0 becomes -tiny, so near/far must swap for it too
    p.neg = (dx < 0.0f ? 1u : 0u) | (dy < 0.0f ? 2u : 0u) | (dz < 0.0f ? 4u : 0u);
    float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    p.kz = (ax > ay) ? ((ax > az) ? 0 : 2) : ((ay > az) ? 1 : 2);
    p.kx = p.kz + 1; if (p.kx == 3) p.kx = 0;
    p.ky = p.kx + 1; if (p.ky == 3) p.ky = 0;
    float dkz = comp(d, p.kz);
    if (dkz < 0.0f) { int t = p.kx; p.kx = p.ky; p.ky = t; }
    p.Sz = rcp_fast(dkz);
    p.Sx = comp(d, p.kx) * p.Sz;
    p.Sy = comp(d, p.ky) * p.Sz;
    return p;
}

// Watertight ray/triangle test, two-sided. Returns true and (t, u, v) when tmin < t < tmax.
__device__ __forceinline__ bool intersect_tri(const RayPre &r, float tmin, float tmax, float4 v0, float4 v1, float4 v2,
                                              float &t_out, float &u_out, float &v_out) {
    const float3 A = make_float3(v0.x - r.o.x, v0.y - r.o.y, v0.z - r.o.z);
    const float3 B = make_float3(v1.x - r.o.x, v1.y - r.o.y, v1.z - r.o.z);
    const float3 C = make_float3(v2.x - r.o.x, v2.y - r.o.y, v2.z - r.o.z);
    const float Akz = comp(A, r.kz), Bkz = comp(B, r.kz), Ckz = comp(C, r.kz);
    const float Ax = comp(A, r.kx) - r.Sx * Akz, Ay = comp(A, r.ky) - r.Sy * Akz;
    const float Bx = comp(B, r.kx) - r.Sx * Bkz, By = comp(B, r.ky) - r.Sy * Bkz;
    const float Cx = comp(C, r.kx) - r.Sx * Ckz, Cy = comp(C, r.ky) - r.Sy * Ckz;
    // Edge functions: each product rounded on its own (no FMA contraction). With a fused multiply-add the two
    // triangles sharing an edge would see rn(p - rn(q)) and rn(q - rn(p)), which can have the SAME sign when p ~ q —
    // a crack. rn(p) - rn(q) and rn(q) - rn(p) are exact negations, which is what watertightness needs.
    float U = sub_rn(mul_rn(Cx, By), mul_rn(Cy, Bx));
    float V = sub_rn(mul_rn(Ax, Cy), mul_rn(Ay, Cx));
    float W = sub_rn(mul_rn(Bx, Ay), mul_rn(By, Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    const float det = U + V + W;
    if (det == 0.0f) return false;
    const float Az = r.Sz * Akz, Bz = r.Sz * Bkz, Cz = r.Sz * Ckz;
    const float T = U * Az + V * Bz + W * Cz;
    const float rdet = rcp_fast(det);
    const float t = T * rdet;
    if (!(t > tmin && t < tmax)) return false;
    t_out = t;
    u_out = V * rdet;
    v_out = W * rdet;
    return true;
}

// Byte -> float without the quarter-rate conversion unit: PRMT drops byte i of `w` into mantissa bits 8..15 of
// 0x47000000 (= 32768.0f), giving exactly 32768 + q on the integer pipe; the bias is folded into the slab offset.
// (I2F.U8 runs on the XU pipe at 16 lanes/clk/SM and was 73 % busy in the first profile — profiles/r01_*.)
// `bias` is 0x47000000 passed in through the kernel parameters (SceneRefs::bias) so that ptxas cannot fold it: PRMT takes one immediate, and
// with both the bias and the selector known it kept the four selectors in registers and re-materialised them around
// every use (~40 MOV / IMAD.U32 per node test in the second profile); now the selector is the immediate.
__device__ __forceinline__ float byte_biased(uint32_t w, int i, uint32_t bias) {
    return __uint_as_float(__byte_perm(w, bias, 0x7604u | ((uint32_t)i << 4)));
}
// Triangle records: 144 MB at 3 M triangles against 27 MB of nodes. VHR_TRI_LOAD_MODE (study, build-time): 0 = __ldg (default); 1 = __ldcs
// (evict-first: the records should not push the nodes out of L1 / L2); 2 = L1::no_allocate.
#ifndef VHR_TRI_LOAD_MODE
#define VHR_TRI_LOAD_MODE 0
#endif
__device__ __forceinline__ float4 tri_load_na(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
#if VHR_TRI_LOAD_MODE == 1
#define VHR_TRI_LOAD(p) __ldcs(p)
#elif VHR_TRI_LOAD_MODE == 2
#define VHR_TRI_LOAD(p) tri_load_na(p)
#else
#define VHR_TRI_LOAD(p) __ldg(p)
#endif
struct Hit {
    float t, u, v;
    uint32_t tri;
};
// Packed fp32x2 (Blackwell FFMA2): two IEEE fp32 fused multiply-adds per issue slot on an aligned register pair
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64 pfma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

// Intersects the ray with the 8 quantised child boxes of node `idx`. The builder stores internal children in the low
// slots, so the hit bits split into (internal children, by ordinal) and (leaf slots) with two ANDs; the leaf slots'
// triangle ranges are only decoded when the triangles are actually tested (expand_leaves).
__device__ __forceinline__ void intersect_node(const WideNode *__restrict__ nodes, uint32_t idx, const RayPre &r, float tmin,
                                               float tmax, uint32_t bias, uint32_t &child_base, uint32_t &child_hits, uint32_t &leaf_hits) {
    const uint4 *np = reinterpret_cast<const uint4 *>(nodes + idx);
    const uint4 n0 = __ldg(np + 0), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
    const uint32_t cb = __ldg(reinterpret_cast<const uint32_t *>(np + 1));
    // bit 31 of the returned base = "pop the highest hit child first": the slots ascend along axis cb >> 30 and the ray runs against it
    // (r.neg has no bit 3, so unsorted nodes, axis 3, are always popped lowest first)
    child_base = (cb & 0x3fffffffu) | (((r.neg >> (cb >> 30)) & 1u) << 31);
    const float sx = __uint_as_float((n0.w & 0xffu) << 23), sy = __uint_as_float(((n0.w >> 8) & 0xffu) << 23),
                sz = __uint_as_float(((n0.w >> 16) & 0xffu) << 23);
    const float ax = sx * r.idir.x, ay = sy * r.idir.y, az = sz * r.idir.z;
    // plane distance t(q) = q*a + b with b = (origin - o) * idir, evaluated as fma(32768 + q, a, b - 32768 a). The
    // rounding of the folded offset is < |a|/512 (1/512 of a quantisation step); the near offset is lowered and the
    // far offset raised by |a|/256 so the test only ever grows the box (conservative, like the builder's rounding).
    const float bx = fmaf(-32768.0f, ax, (__uint_as_float(n0.x) - r.o.x) * r.idir.x);
    const float by = fmaf(-32768.0f, ay, (__uint_as_float(n0.y) - r.o.y) * r.idir.y);
    const float bz = fmaf(-32768.0f, az, (__uint_as_float(n0.z) - r.o.z) * r.idir.z);
    const float ex = fabsf(ax) * 0.00390625f, ey = fabsf(ay) * 0.00390625f, ez = fabsf(az) * 0.00390625f;
    const float bnx = bx - ex, bny = by - ey, bnz = bz - ez;
    // Ize 2013: the exit distance is inflated by a few ulps so rounding never culls a box the exact test would enter;
    // the factor is folded into the far slope and offset (t_far * k = q * (a k) + (b k))
    const float kInfl = 1.0000004f;
    const float afx = ax * kInfl, afy = ay * kInfl, afz = az * kInfl;
    const float bfx = (bx + ex) * kInfl, bfy = (by + ey) * kInfl, bfz = (bz + ez) * kInfl;
    // qlo: x = n2.xy, y = n2.zw, z = n3.xy ; qhi: x = n3.zw, y = n4.xy, z = n4.zw
    const bool nx = r.neg & 1u, ny = r.neg & 2u, nz = r.neg & 4u;
    const uint32_t nearx[2] = {nx ? n3.z : n2.x, nx ? n3.w : n2.y}, farx[2] = {nx ? n2.x : n3.z, nx ? n2.y : n3.w};
    const uint32_t neary[2] = {ny ? n4.x : n2.z, ny ? n4.y : n2.w}, fary[2] = {ny ? n2.z : n4.x, ny ? n2.w : n4.y};
    const uint32_t nearz[2] = {nz ? n4.z : n3.x, nz ? n4.w : n3.y}, farz[2] = {nz ? n3.x : n4.z, nz ? n3.y : n4.w};
    uint32_t miss = 0u;
    // the near and the far plane of a child along one axis share an FFMA2: (q_near, q_far) * (a, a k) + (b_near, b_far k) — the slope /
    // offset pairs are the six values computed above, so the packed form needs no extra registers; 3 FFMA2 instead of 6 FFMA per child
    const u64 AX = pk2(ax, afx), AY = pk2(ay, afy), AZ = pk2(az, afz), BX = pk2(bnx, bfx), BY = pk2(bny, bfy), BZ = pk2(bnz, bfz);
#pragma unroll
    for (int s = 7; s >= 0; --s) {
        const int w = s >> 2, b = s & 3;
        float tnx, tfx, tny, tfy, tnz, tfz;
        upk2(pfma2(pk2(byte_biased(nearx[w], b, bias), byte_biased(farx[w], b, bias)), AX, BX), tnx, tfx);
        upk2(pfma2(pk2(byte_biased(neary[w], b, bias), byte_biased(fary[w], b, bias)), AY, BY), tny, tfy);
        upk2(pfma2(pk2(byte_biased(nearz[w], b, bias), byte_biased(farz[w], b, bias)), AZ, BZ), tnz, tfz);
        const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, tmin));
        const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tmax));
        // empty slots carry an inverted box (qlo = 255, qhi = 0) and can never pass this test.
        // tn <= tf  <=>  the sign bit of tf - tn is clear (x - x = +0 under round-to-nearest; both are finite); a funnel shift moves
        // that bit into the mask: FADD + SHF per child instead of FSETP + SEL + LOP3. Slots go 7 -> 0 so slot 0 ends in bit 0.
        miss = __funnelshift_l(__float_as_uint(tf - tn), miss, 1);
    }
    const uint32_t hits = ~miss & 0xffu;
    const uint32_t imask = n0.w >> 24;
    child_hits = hits & imask;
    leaf_hits = hits & ~imask;
}

// Takes the next child out of a (base | reverse << 31, hit mask) group: lowest slot first, or highest first when the node's slots are
// sorted along an axis the ray runs against. FIXED_ORDER (any-hit rays: their groups never carry the reverse bit) is the two-instruction
// lowest-first pop.
template <bool FIXED_ORDER>
__device__ __forceinline__ uint32_t pop_child(uint2 &group) {
    if (FIXED_ORDER) {
        const uint32_t k = (uint32_t)__ffs((int)group.y) - 1u;
        group.y &= group.y - 1u;
        return k;
    }
    const uint32_t k = (group.x >> 31) ? 31u - (uint32_t)__clz((int)group.y) : (uint32_t)__ffs((int)group.y) - 1u;
    group.y &= ~(1u << k);
    return k;
}

// Decodes the triangle ranges of the hit leaf slots of a node into a 24-bit mask over [tri_base, tri_base + 24).
__device__ __forceinline__ void expand_leaves(const WideNode *__restrict__ nodes, uint32_t idx, uint32_t leaf_hits, uint32_t &tri_base,
                                              uint32_t &tri_hits) {   // leaf_hits != 0
    const uint4 n1 = __ldg(reinterpret_cast<const uint4 *>(nodes + idx) + 1);
    tri_base = n1.y;
    tri_hits = 0u;
    // one short iteration per hit slot (usually one or two) instead of decoding all eight
    do {
        const uint32_t s = (uint32_t)__ffs((int)leaf_hits) - 1u;
        leaf_hits &= leaf_hits - 1u;
        const uint32_t m = __byte_perm(n1.z, n1.w, s) & 0xffu;
        tri_hits |= ((1u << (m >> 5)) - 1u) << (m & 31u);
    } while (leaf_hits);
}

// while-while traversal (Aila & Laine 2009) over the 8-wide nodes, one ray per lane; every lane of the warp calls
// trace() together (`alive` = this lane really has a ray) so callers never diverge before the loop.
// (a triangle whose record says no any-hit stage can reject it — v2.w = 0, bvh_build.cu — is accepted without the call)
// `accept(tri, u, v)` is the any-hit stage: a candidate it rejects is ignored and the traversal goes on (the G-buffer
// producer's alpha test, gbuf.frag:27-32). The hybrid path's own rays are gl_RayFlagsOpaqueEXT (raygen.rgen:39,51,64):
// AcceptAll, which compiles to nothing.
struct AcceptAll {
    __device__ __forceinline__ bool operator()(uint32_t, float, float) const { return true; }
};
// PACKED: stack entries of 4 bytes, (child base << 9) | (reverse bit << 8) | hit mask, instead of 8 (wide trees below 2^23 nodes): the
// per-thread stacks live in local memory, i.e. in L1 next to the nodes — 12 levels x 32 warps x 256 B = 98 KB per SM with 8-byte entries.
// SS > 0: the first SS stack entries of a thread live in SHARED memory (entry i of thread t at vhr_sstack[i * threads + t]: a warp's
// accesses fall into 32 different banks), deeper entries in local memory as before — the kernel is launched with SS * 8 * threads bytes of
// dynamic shared memory. The stack traffic of the default kernel is a third of its L1 sector traffic (ncu: 9.8 M local load + 11.4 M local
// store sectors against 44.8 M global), with write-allocate misses going to L2.
extern __shared__ uint2 vhr_sstack[];
template <bool ANY, class Accept = AcceptAll, bool PACKED = false, int SS = 0>
__device__ __forceinline__ bool trace(const WideNode *__restrict__ nodes, const float4 *__restrict__ tris, uint32_t n_wide,
                                      uint32_t bias, const Ray &ray, bool alive, Hit &hit, const Accept accept = Accept()) {
    if (!alive || n_wide == 0) return false;
    const RayPre r = prepare(ray);
    float tmax = ray.tmax;
    bool found = false;
    uint2 stack[PACKED ? 1 : kStackSize - SS];
    uint32_t stack32[PACKED ? kStackSize : 1];
    uint2 *const sstack = vhr_sstack + (threadIdx.y * blockDim.x + threadIdx.x);
    const int sstride = blockDim.x * blockDim.y;
    int sp = 0;
    uint2 group = make_uint2(0u, 1u);   // (child_base, hit mask over child ordinals): the root
    while (true) {
        if (group.y == 0u) {
            if (sp == 0) break;
            if (PACKED) {
                const uint32_t e = stack32[--sp];
                group = make_uint2((e >> 9) | ((e & 0x100u) << 23), e & 0xffu);
            } else if (SS > 0) {
                --sp;
                group = sp < SS ? sstack[sp * sstride] : stack[sp - SS];
            } else {
                group = stack[--sp];
            }
        }
        const uint32_t k = pop_child<ANY>(group);
        if (group.y != 0u && sp < kStackSize) {
            if (PACKED) stack32[sp++] = ((group.x & 0x7fffffffu) << 9) | ((group.x >> 31) << 8) | group.y;
            else if (SS > 0) {
                if (sp < SS) sstack[sp * sstride] = group; else stack[sp - SS] = group;
                ++sp;
            } else stack[sp++] = group;
        }
        const uint32_t node = (ANY ? group.x : (group.x & 0x7fffffffu)) + k;
        uint32_t child_base, child_hits, leaf_hits;
        intersect_node(nodes, node, r, ray.tmin, tmax, bias, child_base, child_hits, leaf_hits);
        // any-hit rays keep one fixed order (lowest slot first): measured faster than near-side-first for the incoherent AO rays
        // (0.496 -> 0.472 ms at 3 M triangles, profiles/traces/r01k_trace.log) — neighbouring lanes then fetch the same children
        if (ANY) child_base &= 0x7fffffffu;
        group = make_uint2(child_base, child_hits);
        if (leaf_hits) {
            uint32_t tri_base, tri_hits;
            expand_leaves(nodes, node, leaf_hits, tri_base, tri_hits);
            do {
                const uint32_t j = (uint32_t)__ffs((int)tri_hits) - 1u;
                tri_hits &= tri_hits - 1u;
                const float4 *tp = tris + (size_t)(tri_base + j) * 3;
                const float4 v0 = VHR_TRI_LOAD(tp), v1 = VHR_TRI_LOAD(tp + 1), v2 = VHR_TRI_LOAD(tp + 2);
                float t, u, v;
                if (intersect_tri(r, ray.tmin, tmax, v0, v1, v2, t, u, v) && (__float_as_uint(v2.w) == 0u || accept(tri_base + j, u, v))) {
                    if (ANY) return true;
                    tmax = t;
                    hit.t = t; hit.u = u; hit.v = v; hit.tri = tri_base + j;
                    found = true;
                }
            } while (tri_hits);
        }
    }
    return found;
}

// trace() with POSTPONED LEAVES (Aila & Laine's speculative traversal, adapted to leaf slots that live inside the wide
// node). The profile of trace() shows the triangle block (leaf-slot decode + fetch + watertight test, ~23 % of all issued
// instructions) running at 2-4 of 32 lanes: a lane tests its triangles the moment its node reports a leaf hit while the
// other lanes wait. Here a lane that finds leaf hits only notes them (node index + slot mask, two registers) and keeps
// traversing; the whole warp runs the triangle block together when a lane cannot go on without it (it found a second
// leaf node, or it has no nodes left) or when at least `batch` lanes have work noted. Every lane of the warp must call
// this together (full mask votes); `alive` = this lane really has a ray. Results are identical to trace(): the same
// nodes' leaves are tested, only later (a postponed any-hit leaf may cost the lane a few extra node steps that the warp
// was going to issue anyway).
template <bool ANY, class Accept = AcceptAll>
__device__ __forceinline__ bool trace_batched(const WideNode *__restrict__ nodes, const float4 *__restrict__ tris, uint32_t n_wide,
                                              uint32_t bias, const Ray &ray, bool alive, Hit &hit, int batch, const Accept accept = Accept()) {
    const unsigned FULL = 0xffffffffu;
    const RayPre r = prepare(ray);
    float tmax = ray.tmax;
    bool found = false;
    bool done = !alive || n_wide == 0;
    uint2 stack[kStackSize];
    int sp = 0;
    uint2 group = make_uint2(0u, 1u);   // (child_base, hit mask over child ordinals): the root
    uint32_t pend_node = 0u, pend_leaves = 0u;       // postponed leaf work: node index + hit leaf slots
    while (true) {
        uint32_t new_node = 0u, new_leaves = 0u;
        if (!done) {
            bool have = true;
            if (group.y == 0u) {
                if (sp == 0) have = false;
                else group = stack[--sp];
            }
            if (have) {
                const uint32_t k = pop_child<ANY>(group);
                if (group.y != 0u && sp < kStackSize) stack[sp++] = group;
                const uint32_t node = (ANY ? group.x : (group.x & 0x7fffffffu)) + k;
                uint32_t child_base, child_hits, leaf_hits;
                intersect_node(nodes, node, r, ray.tmin, tmax, bias, child_base, child_hits, leaf_hits);
                if (ANY) child_base &= 0x7fffffffu;           // same order policy as trace()
                group = make_uint2(child_base, child_hits);
                new_node = node; new_leaves = leaf_hits;
            }
        }
        const bool more_nodes = !done && (group.y != 0u || sp != 0);
        bool urgent = false;
        if (new_leaves) {
            if (pend_leaves) urgent = true;                       // second leaf node: the noted one has to be tested first
            else { pend_node = new_node; pend_leaves = new_leaves; new_leaves = 0u; }
        }
        if (!done && pend_leaves && !more_nodes) urgent = true;   // nothing left to traverse: the answer hangs on the noted leaves
        const unsigned pending = __ballot_sync(FULL, !done && pend_leaves != 0u);
        const bool run = __any_sync(FULL, urgent) || __popc(pending) >= batch;
        if (run && !done && pend_leaves) {
            uint32_t tri_base, tri_hits;
            expand_leaves(nodes, pend_node, pend_leaves, tri_base, tri_hits);
            do {
                const uint32_t j = (uint32_t)__ffs((int)tri_hits) - 1u;
                tri_hits &= tri_hits - 1u;
                const float4 *tp = tris + (size_t)(tri_base + j) * 3;
                const float4 v0 = VHR_TRI_LOAD(tp), v1 = VHR_TRI_LOAD(tp + 1), v2 = VHR_TRI_LOAD(tp + 2);
                float t, u, v;
                if (intersect_tri(r, ray.tmin, tmax, v0, v1, v2, t, u, v) && (__float_as_uint(v2.w) == 0u || accept(tri_base + j, u, v))) {
                    found = true;
                    if (ANY) { done = true; break; }
                    tmax = t;
                    hit.t = t; hit.u = u; hit.v = v; hit.tri = tri_base + j;
                }
            } while (tri_hits);
            pend_node = new_node; pend_leaves = new_leaves;       // the leaf node found this round (if any) is noted next
        }
        if (!done && !pend_leaves && group.y == 0u && sp == 0) done = true;
        if (__all_sync(FULL, done)) break;
    }
    return found;
}

// ---------------------------------------------------------------------------------------------------------------
// Shading of the reflection ray: reflection_hit.rchit:10-72
// ---------------------------------------------------------------------------------------------------------------
struct SceneRefs {
    const Vertex *verts;
    const uint32_t *indices;
    const Primitive *prims;
    const float *normal_mats;     // 9 floats per primitive, column-major inverseTranspose(mat3(transform))
    const WideNode *nodes;
    const float4 *tris;
    uint32_t n_wide;
    uint32_t bias;                // 0x47000000 (see byte_biased)
    const TextureDesc *textures;  // textures[] (glsl_common.h:104); entries without an image have texels == nullptr
    const float *lut;             // UNORM / sRGB decode tables (fetch_texel)
    uint32_t n_textures;
};

__device__ __forceinline__ bool has_texture(const SceneRefs &s, int idx) {
    return idx >= 0 && (uint32_t)idx < s.n_textures && s.textures[idx].texels != nullptr;
}
// v0.uv0 * b0 + v1.uv0 * b1 + v2.uv0 * b2 (reflection_hit.rchit:22; gbuf.vert:24 + the rasteriser's interpolation)
__device__ __forceinline__ float2 bary_uv(const Vertex &v0, const Vertex &v1, const Vertex &v2, float b0, float b1, float b2) {
    return make_float2(add_rn(add_rn(mul_rn(v0.uv0[0], b0), mul_rn(v1.uv0[0], b1)), mul_rn(v2.uv0[0], b2)),
                       add_rn(add_rn(mul_rn(v0.uv0[1], b0), mul_rn(v1.uv0[1], b1)), mul_rn(v2.uv0[1], b2)));
}

__device__ __forceinline__ float3 f3(const float *p) { return make_float3(p[0], p[1], p[2]); }
__device__ __forceinline__ float3 bary3(float3 a, float3 b, float3 c, float b0, float b1, float b2) {
    // (a*b0 + b*b1) + c*b2, componentwise, products and sums rounded like the oracle
    return make_float3(add_rn(add_rn(mul_rn(a.x, b0), mul_rn(b.x, b1)), mul_rn(c.x, b2)),
                       add_rn(add_rn(mul_rn(a.y, b0), mul_rn(b.y, b1)), mul_rn(c.y, b2)),
                       add_rn(add_rn(mul_rn(a.z, b0), mul_rn(b.z, b1)), mul_rn(c.z, b2)));
}

__device__ float4 reflection_hit(const SceneRefs &s, const PerFrameData &pfd, const Hit &h) {
    const float4 *tp = s.tris + (size_t)h.tri * 3;
    const uint32_t g = __float_as_uint(__ldg(tp).w), pid = __float_as_uint(__ldg(tp + 1).w);
    const Primitive &prim = s.prims[g];
    const uint32_t i0 = s.indices[prim.index_offset + 3 * pid + 0], i1 = s.indices[prim.index_offset + 3 * pid + 1],
                   i2 = s.indices[prim.index_offset + 3 * pid + 2];
    const Vertex &v0 = s.verts[prim.vertex_offset + i0], &v1 = s.verts[prim.vertex_offset + i1], &v2 = s.verts[prim.vertex_offset + i2];
    const float b1 = h.u, b2 = h.v, b0 = sub_rn(sub_rn(1.0f, b1), b2);
    const float3 normal = bary3(f3(v0.normal), f3(v1.normal), f3(v2.normal), b0, b1, b2);
    const float3 pobj = bary3(f3(v0.pos), f3(v1.pos), f3(v2.pos), b0, b1, b2);
    const float4 pw = mul44_rn(prim.transform, make_float4(pobj.x, pobj.y, pobj.z, 1.0f));
    const float3 position = make_float3(pw.x, pw.y, pw.z);
    float3 albedo = make_float3(prim.material.base_color[0], prim.material.base_color[1], prim.material.base_color[2]);
    float metallic = prim.material.metallic_factor, roughness = prim.material.roughness_factor;
    const bool tex_a = has_texture(s, prim.material.base_color_texture), tex_mr = has_texture(s, prim.material.metallic_roughness_texture);
    if (tex_a || tex_mr) {                                                                 // reflection_hit.rchit:26-39
        const float2 uv = bary_uv(v0, v1, v2, b0, b1, b2);
        if (tex_a) {
            const float4 c = sample_texture(s.textures, s.lut, prim.material.base_color_texture, uv.x, uv.y);
            albedo = make_float3(c.x, c.y, c.z);
        }
        if (tex_mr) {
            const float4 c = sample_texture(s.textures, s.lut, prim.material.metallic_roughness_texture, uv.x, uv.y);
            metallic = mul_rn(metallic, c.y);
            roughness = mul_rn(roughness, c.z);
        }
    }
    const float3 cam = make_float3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
    const float3 V = normalize_rn(make_float3(sub_rn(cam.x, position.x), sub_rn(cam.y, position.y), sub_rn(cam.z, position.z)));
    const float3 L = make_float3(-pfd.directional_light.direction[0], -pfd.directional_light.direction[1], -pfd.directional_light.direction[2]);
    const float3 N = normal;
    const float3 H = normalize_rn(make_float3(add_rn(L.x, V.x), add_rn(L.y, V.y), add_rn(L.z, V.z)));
    const float3 c = shade_direct_rn(albedo, metallic, roughness, N, V, L, H, pfd.directional_light.intensity, pfd.directional_light.color);
    return make_float4(c.x, c.y, c.z, 1.0f);
}

// ---------------------------------------------------------------------------------------------------------------
// raygen
// ---------------------------------------------------------------------------------------------------------------
struct RaygenParams {
    int W, H;                 // launch size (gl_LaunchSizeEXT)
    int y_begin, y_end;
    int ao_spp;
    int flags;                // bit0 shadows, bit1 AO, bit2 reflections
    int leaf_batch;           // trace_batched: lanes with noted leaf work that trigger the triangle block
    const uint2 *normals;     // binding 0
    const float *depth;       // binding 1
    uint32_t *shadow_ao;      // binding 2 (RG16F)
    uint2 *reflections;       // binding 3 (RGBA16F)
    float *refl_t;            // optional debug output: closest-hit distance of the reflection ray (-1 = miss/sky)
    SceneRefs scene;
    // multi-GPU (vhr_set_partition with ray_block_rows = 8): this rank traces the 8-row blocks b with b % world == rank and
    // stores every pixel into the image of the rank that OWNS the row (its SVGF band) over NVLink — the all-to-all that
    // would follow the pass is fused into it. world == 0: single-GPU addressing.
    int world, rank;
    int band_begin[VHR_MAX_RANKS + 1];
    uint32_t *shadow_ao_of[VHR_MAX_RANKS];
    uint2 *reflections_of[VHR_MAX_RANKS];
};

// 8x4-pixel warp tiles inside a 16x8-pixel macro block: neighbouring lanes trace neighbouring pixels. A macro block is one CTA of
// four warps (WPB = 4) or 4 / WPB consecutive CTAs of WPB warps — with one-warp CTAs a finished warp gives its registers back at
// once instead of waiting for the slowest warp of its CTA.
template <int WPB = 4>
__device__ __forceinline__ void tile_coords(int &x, int &y) {
    constexpr int kSplit = 4 / WPB;
    const int lane = threadIdx.x & 31;
    const int warp = (int)(blockIdx.x % kSplit) * WPB + (int)(threadIdx.x >> 5);
    x = (int)(blockIdx.x / kSplit) * 16 + (warp & 1) * 8 + (lane & 7);
    y = blockIdx.y * 8 + (warp >> 1) * 4 + (lane >> 3);
}

// ---- AO rays sorted by direction inside the CTA (VHR_OPT_RAYGEN_VARIANT 8) -------------------------------------------
// The AO rays of a warp tile start next to each other but leave over the whole hemisphere (15.7 of 32 lanes active in their node
// test, against 24.5 for the shadow rays, profiles/r01_ncu_raygen_segments.md). Here the CTA's 128 AO rays are counting-sorted by a
// 24-valued direction key (cube-map face of the direction x the signs of the two other components) before they are traced: thread t
// traces the t-th ray in key order and hands the result back to the pixel's thread through shared memory; lanes without a ray
// (sky, AO off) sort to the end, so whole warps of them do nothing. The rays and their any-hit answers are the same, only the
// thread that computes each one changes.
// Measured (profiles/traces/r01r_trace.log, 1080p): AO pass 0.467 -> 0.507 ms at 3 M triangles, 0.393 -> 0.422 ms at 260 k — slower: the rays of
// a warp now start up to 16 pixels apart, and that costs more than the common direction gains. Kept for study, not the default.
struct AoSortShared {
    float4 o[128];            // origin.xyz, tmin
    float4 d[128];            // direction.xyz, tmax
    uint16_t warp_count[4][32];
    uint16_t warp_base[4][32];
    uint16_t perm[128];
    uint8_t occluded[128];
};
__device__ __forceinline__ uint32_t direction_key(float3 d) {
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    const uint32_t sx = d.x < 0.0f, sy = d.y < 0.0f, sz = d.z < 0.0f;
    if (ax >= ay && ax >= az) return (0u + sx) * 4u + sy * 2u + sz;
    if (ay >= az) return (2u + sy) * 4u + sx * 2u + sz;
    return (4u + sz) * 4u + sx * 2u + sy;
}
// Every thread of the 128-thread CTA calls this together. Returns the any-hit answer of THIS thread's ray.
__device__ __forceinline__ bool trace_any_sorted(const SceneRefs &scene, const Ray &ray, bool alive, AoSortShared &sm) {
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t key = alive ? direction_key(ray.d) : 24u;
    sm.o[tid] = make_float4(ray.o.x, ray.o.y, ray.o.z, ray.tmin);
    sm.d[tid] = make_float4(ray.d.x, ray.d.y, ray.d.z, ray.tmax);
    sm.warp_count[warp][lane] = 0;
    __syncwarp();
    const unsigned same = __match_any_sync(FULL, key);
    const uint32_t rank = __popc(same & ((1u << lane) - 1u));
    if (rank == 0u) sm.warp_count[warp][key] = (uint16_t)__popc(same);
    __syncthreads();
    if (warp == 0) {
        // lane = key: total over the four warps, exclusive scan over the keys, then one base per (warp, key) in key-major order
        const uint32_t c0 = sm.warp_count[0][lane], c1 = sm.warp_count[1][lane], c2 = sm.warp_count[2][lane], c3 = sm.warp_count[3][lane];
        const uint32_t tot = c0 + c1 + c2 + c3;
        uint32_t incl = tot;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, incl, off);
            if (lane >= off) incl += v;
        }
        uint32_t run = incl - tot;
        sm.warp_base[0][lane] = (uint16_t)run; run += c0;
        sm.warp_base[1][lane] = (uint16_t)run; run += c1;
        sm.warp_base[2][lane] = (uint16_t)run; run += c2;
        sm.warp_base[3][lane] = (uint16_t)run;
    }
    __syncthreads();
    sm.perm[sm.warp_base[warp][key] + rank] = (uint16_t)tid;
    const uint32_t n_alive = sm.warp_base[0][24];                 // the rays without work sort last
    __syncthreads();
    const int j = sm.perm[tid];
    const float4 o = sm.o[j], d = sm.d[j];
    Ray r;
    r.o = make_float3(o.x, o.y, o.z); r.tmin = o.w;
    r.d = make_float3(d.x, d.y, d.z); r.tmax = d.w;
    Hit h;
    const bool occ = trace<true>(scene.nodes, scene.tris, scene.n_wide, scene.bias, r, (uint32_t)tid < n_alive, h);
    sm.occluded[j] = occ ? 1 : 0;
    __syncthreads();
    const bool mine = sm.occluded[tid] != 0;
    __syncthreads();                                               // the arrays are reused by the next AO sample
    return mine;
}

// MIN_BLOCKS is the occupancy target handed to ptxas (__launch_bounds__). Measured at 1080p / 3 M triangles (profiles/traces/r01c_trace.log):
//   8 (default): 64 registers, 8 blocks / SM, ~10 spilled words — 0.879 ms shadow+AO, 2.40 ms shadow + 2 AO + reflection;
//   0 (VHR_OPT_RAYGEN_VARIANT 2): unspecified, ptxas settles on 72 registers / 7 blocks — 0.883 / 2.47 ms;
//   1 (variant 3): no cap, 117 registers / 4 blocks — 1.16 / 3.39 ms (fewer warps to hide the node fetches);
//   BATCHED (variant 4): trace_batched — 1.00 / 2.57 ms: postponing leaves costs the any-hit rays more node steps than the fuller
//   triangle block saves. Same images in every variant.
template <int MIN_BLOCKS, bool BATCHED = false, int WPB = 4, bool SORT_AO = false, bool PACKED = false, bool MERGED = false, int SS = 0>
__global__ void __launch_bounds__(32 * WPB, MIN_BLOCKS * 4 / WPB) raygen_kernel(const __grid_constant__ RaygenParams p, const __grid_constant__ PerFrameData pfd) {
    static_assert(!SORT_AO || WPB == 4, "the AO sort works on 128-thread CTAs");
    int x, y;
    tile_coords<WPB>(x, y);
    uint32_t *__restrict__ out_sa = p.shadow_ao;
    uint2 *__restrict__ out_refl = p.reflections;
    if (p.world > 0) {
        // blockIdx.y counts this rank's 8-row blocks; the block's rows belong to one or two SVGF bands
        y = (y - blockIdx.y * 8) + (blockIdx.y * p.world + p.rank) * 8;
        int owner = 0;
#pragma unroll
        for (int r = 1; r < VHR_MAX_RANKS; ++r)
            if (r < p.world && y >= p.band_begin[r]) owner = r;
        out_sa = p.shadow_ao_of[owner];
        out_refl = p.reflections_of[owner];
    } else {
        y += p.y_begin;
    }
    // every lane stays in the kernel: trace() is warp-synchronous, lanes without a ray just pass alive = false
    const bool in_range = x < p.W && y < p.y_end;
    const size_t pix = in_range ? (size_t)y * p.W + x : 0;
    const float u = __fdiv_rn(add_rn((float)x, 0.5f), (float)p.W), v = __fdiv_rn(add_rn((float)y, 0.5f), (float)p.H);
    uint32_t rng = seed_thread(((uint32_t)y * (uint32_t)p.H + (uint32_t)x) * pfd.frame_index);   // raygen.rgen:17 (Q4)
    const float depth = in_range ? __ldg(&p.depth[pix]) : 0.0f;                                  // texel centre: exact texel (Q17)
    const bool lit = in_range && depth != 0.0f;
    if (in_range && !lit) {                                                                      // raygen.rgen:20-24
        if (!(p.flags & 8)) out_sa[pix] = pack_rg16f(1.0f, 1.0f);
        out_refl[pix] = make_uint2(0u, 0u);
        if (p.refl_t) p.refl_t[pix] = -1.0f;
    }
    const float3 P = unproject_rn(pfd.camera_viewproj_inverse, lit ? depth : 1.0f, u, v);
    const float3 L = make_float3(-pfd.directional_light.direction[0], -pfd.directional_light.direction[1], -pfd.directional_light.direction[2]);
    const float4 n4 = lit ? unpack_rgba16f(__ldg(&p.normals[pix])) : make_float4(0.0f, 0.0f, 1.0f, 0.0f);
    const float3 N = make_float3(n4.x, n4.y, n4.z);
    Ray ray;
    ray.o = make_float3(add_rn(P.x, mul_rn(N.x, 0.1f)), add_rn(P.y, mul_rn(N.y, 0.1f)), add_rn(P.z, mul_rn(N.z, 0.1f)));
    ray.tmin = 0.01f;
    Hit hit;

    float rnd1, rnd2, shadow = 1.0f, ao = 0.0f;
    if constexpr (MERGED) {
        // MERGED: the shadow ray and the AO rays go through ONE inlined copy of the any-hit traversal (a loop over the ray kinds) instead of
        // two: half the hot code in the instruction cache. Same rays, same RNG order.
#pragma unroll 1
        for (int k = 0; k <= p.ao_spp; ++k) {
            rnd1 = random01(rng);
            rnd2 = random01(rng);
            const bool is_shadow = k == 0;
            const bool enabled = is_shadow ? (p.flags & 1) != 0 : (p.flags & 2) != 0;
            bool occluded = false;
            if (enabled) {
                ray.d = is_shadow ? onb_apply(L, normalize_rn(uniform_sample_cone(rnd1, rnd2, 0.999995f))) : onb_apply(N, uniform_sample_cosine_weighted_hemisphere(rnd1, rnd2));
                ray.tmax = is_shadow ? 10000.0f : 5.0f;
                occluded = trace<true, AcceptAll, PACKED, SS>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit);
            }
            if (is_shadow) shadow = occluded ? 0.0f : 1.0f;
            else ao = add_rn(ao, occluded ? 0.0f : 1.0f);
        }
    } else {
    // shadow (raygen.rgen:32-41; the 4x loop re-traces one ray, Q3)
    rnd1 = random01(rng); rnd2 = random01(rng);
    if (p.flags & 1) {
        const float3 cone = normalize_rn(uniform_sample_cone(rnd1, rnd2, 0.999995f));
        ray.d = onb_apply(L, cone);
        ray.tmax = 10000.0f;
        const bool occluded = BATCHED ? trace_batched<true>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit, p.leaf_batch)
                                      : trace<true, AcceptAll, PACKED, SS>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit);
        shadow = occluded ? 0.0f : 1.0f;
    }
    // ambient occlusion (raygen.rgen:44-55)
    for (int i = 0; i < p.ao_spp; ++i) {
        rnd1 = random01(rng);
        rnd2 = random01(rng);
        if (p.flags & 2) {
            ray.d = onb_apply(N, uniform_sample_cosine_weighted_hemisphere(rnd1, rnd2));
            ray.tmax = 5.0f;
            bool occluded;
            if constexpr (SORT_AO) {
                __shared__ AoSortShared ao_sort;
                occluded = trace_any_sorted(p.scene, ray, lit, ao_sort);
            } else {
                occluded = BATCHED ? trace_batched<true>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit, p.leaf_batch)
                                   : trace<true, AcceptAll, PACKED, SS>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit);
            }
            ao = add_rn(ao, occluded ? 0.0f : 1.0f);
        } else {
            ao = add_rn(ao, 1.0f);
        }
    }
    }   // !MERGED
    ao = __fdiv_rn(ao, (float)p.ao_spp);
    if (lit && !(p.flags & 8)) out_sa[pix] = pack_rg16f(shadow, ao);      // bit 3: another kernel owns the shadow / AO texel (variant 9)

    // mirror reflection (raygen.rgen:59-65)
    if (p.flags & 4) {
        float4 payload = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        float rt = -1.0f;
        const float3 cam = make_float3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
        const float3 I = normalize_rn(make_float3(sub_rn(P.x, cam.x), sub_rn(P.y, cam.y), sub_rn(P.z, cam.z)));
        const float k2 = mul_rn(2.0f, dot3_rn(N, I));
        ray.d = make_float3(sub_rn(I.x, mul_rn(N.x, k2)), sub_rn(I.y, mul_rn(N.y, k2)), sub_rn(I.z, mul_rn(N.z, k2)));
        ray.tmax = 10000.0f;
        const bool refl_hit = BATCHED ? trace_batched<false>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit, p.leaf_batch)
                                      : trace<false, AcceptAll, PACKED, SS>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, lit, hit);
        if (refl_hit && lit) {
            payload = reflection_hit(p.scene, pfd, hit);
            rt = hit.t;
        }
        if (lit) {
            out_refl[pix] = pack_rgba16f(payload);
            if (p.refl_t) p.refl_t[pix] = rt;
        }
    } else if (lit) {
        out_refl[pix] = make_uint2(0u, 0u);
        if (p.refl_t) p.refl_t[pix] = -1.0f;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// raygen, persistent variant: warps pull pixels from a global queue and every lane runs its pixel's rays back to back
// ---------------------------------------------------------------------------------------------------------------
// The per-pixel kernel above synchronises the warp after every ray kind: all 32 shadow rays finish before the first AO
// ray starts, so a lane whose any-hit ray ended early idles until the slowest ray of the warp is done (the first
// profile shows the AO node test at 45 % lane utilisation). Here a lane owns a small state machine
//     pixel -> shadow ray -> AO ray x spp -> reflection ray -> write results -> next pixel
// and the warp alternates between two phases (Aila & Laine 2009, persistent threads with dynamic fetch):
//     refill   when at least kRefillIdle lanes have no ray in flight: finished pixels are written, new pixels are
//              handed out from the warp's chunk of the tile-ordered pixel queue (one atomicAdd per chunk), the next
//              ray of every idle lane is generated;
//     traverse node step + triangle tests for every lane with a ray, repeated until too many lanes have gone idle.
// Ray generation is the same arithmetic in the same RNG order as raygen_kernel, so both variants produce identical images.
constexpr int kChunkPixels = 64;      // pixels a warp takes from the queue per atomicAdd (two 8x4 tiles)

__global__ void __launch_bounds__(128) raygen_persistent_kernel(const __grid_constant__ RaygenParams p, const __grid_constant__ PerFrameData pfd,
                                                                uint32_t *__restrict__ queue_head, const int kRefillIdle, const int kBurst) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int tiles_x = (p.W + 7) >> 3;
    const int rows = p.y_end - p.y_begin;
    const uint32_t n_items = (uint32_t)tiles_x * (uint32_t)((rows + 3) >> 2) * 32u;
    const int last_stage = p.ao_spp + ((p.flags & 4) ? 1 : 0);     // stage 0 shadow, 1..spp AO, spp+1 reflection
    const WideNode *__restrict__ nodes = p.scene.nodes;
    const float4 *__restrict__ tris = p.scene.tris;

    // warp-uniform chunk of the pixel queue
    uint32_t chunk_next = 0u, chunk_end = 0u;
    bool queue_empty = p.scene.n_wide == 0 && false;
    // per-lane pixel state
    bool have_pixel = false;
    int stage = 0;
    size_t pix = 0;
    uint32_t rng = 0u;
    float3 P = make_float3(0.f, 0.f, 0.f), N = make_float3(0.f, 0.f, 1.f);
    float shadow = 1.0f, ao = 0.0f;
    // per-lane ray state
    bool ray_active = false, closest = false, found = false;
    RayPre r;
    r.o = P; r.idir = P; r.kx = 0; r.ky = 1; r.kz = 2; r.Sx = r.Sy = r.Sz = 0.f; r.neg = 0u;
    float tmin = 0.01f, tmax = 0.0f;
    Hit hit;
    hit.t = -1.f; hit.u = hit.v = 0.f; hit.tri = 0u;
    uint2 stack[kStackSize];
    int sp = 0;
    uint2 group = make_uint2(0u, 0u);
    const uint32_t bias = p.scene.bias;

    while (true) {
        // ================================ refill ==================================================================
        const uint32_t idle_mask = __ballot_sync(FULL, !ray_active);
        if (__popc(idle_mask) >= kRefillIdle) {
            // 1. idle lanes whose pixel has no rays left write it out and give it up
            if (!ray_active && have_pixel && stage > last_stage) {
                p.shadow_ao[pix] = pack_rg16f(shadow, __fdiv_rn(ao, (float)p.ao_spp));
                if (p.flags & 4) {
                    float4 payload = make_float4(0.f, 0.f, 0.f, 0.f);
                    float rt = -1.0f;
                    if (found) { payload = reflection_hit(p.scene, pfd, hit); rt = hit.t; }
                    p.reflections[pix] = pack_rgba16f(payload);
                    if (p.refl_t) p.refl_t[pix] = rt;
                } else {
                    p.reflections[pix] = make_uint2(0u, 0u);
                    if (p.refl_t) p.refl_t[pix] = -1.0f;
                }
                have_pixel = false;
            }
            // 2. hand out new pixels (warp-uniform control flow)
            bool want = !ray_active && !have_pixel;
            uint32_t item = 0xffffffffu;
            while (true) {
                const uint32_t wm = __ballot_sync(FULL, want);
                if (wm == 0u || queue_empty) break;
                if (chunk_next >= chunk_end) {
                    uint32_t base = 0u;
                    if (lane == 0) base = atomicAdd(queue_head, (uint32_t)kChunkPixels);
                    base = __shfl_sync(FULL, base, 0);
                    if (base >= n_items) { queue_empty = true; break; }
                    chunk_next = base;
                    chunk_end = min(base + (uint32_t)kChunkPixels, n_items);
                }
                const uint32_t rank = __popc(wm & ((1u << lane) - 1u));
                const uint32_t avail = chunk_end - chunk_next;
                if (want && rank < avail) { item = chunk_next + rank; want = false; }
                chunk_next += min((uint32_t)__popc(wm), avail);
            }
            // 3. set up the new pixel (raygen.rgen:15-29)
            if (item != 0xffffffffu) {
                const uint32_t tile = item >> 5, within = item & 31u;
                const int x = (int)(tile % (uint32_t)tiles_x) * 8 + (int)(within & 7u);
                const int y = p.y_begin + (int)(tile / (uint32_t)tiles_x) * 4 + (int)(within >> 3);
                if (x < p.W && y < p.y_end) {
                    pix = (size_t)y * p.W + x;
                    const float depth = __ldg(&p.depth[pix]);
                    if (depth == 0.0f) {                                   // sky: raygen.rgen:20-24
                        p.shadow_ao[pix] = pack_rg16f(1.0f, 1.0f);
                        p.reflections[pix] = make_uint2(0u, 0u);
                        if (p.refl_t) p.refl_t[pix] = -1.0f;
                    } else {
                        const float u = __fdiv_rn(add_rn((float)x, 0.5f), (float)p.W), v = __fdiv_rn(add_rn((float)y, 0.5f), (float)p.H);
                        rng = seed_thread(((uint32_t)y * (uint32_t)p.H + (uint32_t)x) * pfd.frame_index);
                        P = unproject_rn(pfd.camera_viewproj_inverse, depth, u, v);
                        const float4 n4 = unpack_rgba16f(__ldg(&p.normals[pix]));
                        N = make_float3(n4.x, n4.y, n4.z);
                        have_pixel = true;
                        stage = 0;
                        shadow = 1.0f; ao = 0.0f; found = false;
                    }
                }
            }
            // 4. generate the next ray of every idle lane that owns a pixel
            if (!ray_active && have_pixel) {
                Ray ray;
                ray.o = make_float3(add_rn(P.x, mul_rn(N.x, 0.1f)), add_rn(P.y, mul_rn(N.y, 0.1f)), add_rn(P.z, mul_rn(N.z, 0.1f)));
                ray.tmin = 0.01f;
                bool launch = false;
                while (!launch && stage <= last_stage) {
                    if (stage == 0) {                                      // shadow (raygen.rgen:32-41)
                        const float rnd1 = random01(rng), rnd2 = random01(rng);
                        if (p.flags & 1) {
                            const float3 L = make_float3(-pfd.directional_light.direction[0], -pfd.directional_light.direction[1], -pfd.directional_light.direction[2]);
                            ray.d = onb_apply(L, normalize_rn(uniform_sample_cone(rnd1, rnd2, 0.999995f)));
                            ray.tmax = 10000.0f;
                            closest = false; launch = true;
                        } else {
                            ++stage;
                        }
                    } else if (stage <= p.ao_spp) {                        // ambient occlusion (raygen.rgen:44-55)
                        const float rnd1 = random01(rng), rnd2 = random01(rng);
                        if (p.flags & 2) {
                            ray.d = onb_apply(N, uniform_sample_cosine_weighted_hemisphere(rnd1, rnd2));
                            ray.tmax = 5.0f;
                            closest = false; launch = true;
                        } else {
                            ao = add_rn(ao, 1.0f);
                            ++stage;
                        }
                    } else {                                               // mirror reflection (raygen.rgen:59-65)
                        const float3 cam = make_float3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
                        const float3 I = normalize_rn(make_float3(sub_rn(P.x, cam.x), sub_rn(P.y, cam.y), sub_rn(P.z, cam.z)));
                        const float k2 = mul_rn(2.0f, dot3_rn(N, I));
                        ray.d = make_float3(sub_rn(I.x, mul_rn(N.x, k2)), sub_rn(I.y, mul_rn(N.y, k2)), sub_rn(I.z, mul_rn(N.z, k2)));
                        ray.tmax = 10000.0f;
                        closest = true; launch = true;
                    }
                }
                if (launch) {
                    r = prepare(ray);
                    tmin = ray.tmin; tmax = ray.tmax;
                    found = false;
                    sp = 0;
                    group = make_uint2(0u, p.scene.n_wide ? 1u : 0u);
                    ray_active = true;
                }
            }
            if (__ballot_sync(FULL, ray_active) == 0u) {
                // nothing in flight: either pixels are still being finalised (loop again) or the queue is drained
                if (queue_empty && __ballot_sync(FULL, have_pixel) == 0u) break;
                continue;
            }
        }
        // ================================ traverse ================================================================
        // A burst of up to kBurst node steps per lane with no warp-level synchronisation in between (lanes in the
        // triangle test and lanes already in their next node test interleave under independent thread scheduling);
        // the warp only re-votes on refilling after the burst.
#pragma unroll 1
        for (int it = 0; it < kBurst && ray_active; ++it) {
            bool done = false, occluded = false;
            if (group.y == 0u) {
                if (sp == 0) done = true;
                else group = stack[--sp];
            }
            if (!done) {
                const uint32_t k = pop_child<false>(group);
                if (group.y != 0u && sp < kStackSize) stack[sp++] = group;
                const uint32_t node = (group.x & 0x7fffffffu) + k;
                uint32_t child_base, child_hits, leaf_hits;
                intersect_node(nodes, node, r, tmin, tmax, bias, child_base, child_hits, leaf_hits);
                if (!closest) child_base &= 0x7fffffffu;      // same order policy as trace()
                group = make_uint2(child_base, child_hits);
                if (leaf_hits) {
                    uint32_t tri_base, tri_hits;
                    expand_leaves(nodes, node, leaf_hits, tri_base, tri_hits);
                    do {
                        const uint32_t j = (uint32_t)__ffs((int)tri_hits) - 1u;
                        tri_hits &= tri_hits - 1u;
                        const float4 *tp = tris + (size_t)(tri_base + j) * 3;
                        const float4 v0 = VHR_TRI_LOAD(tp), v1 = VHR_TRI_LOAD(tp + 1), v2 = VHR_TRI_LOAD(tp + 2);
                        float t, u, v;
                        if (intersect_tri(r, tmin, tmax, v0, v1, v2, t, u, v)) {
                            if (!closest) { occluded = true; done = true; break; }
                            tmax = t;
                            hit.t = t; hit.u = u; hit.v = v; hit.tri = tri_base + j;
                            found = true;
                        }
                    } while (tri_hits);
                }
            }
            if (done) {
                // miss.rmiss: payload 1 (visible); any hit leaves it 0
                if (stage == 0) shadow = occluded ? 0.0f : 1.0f;
                else if (stage <= p.ao_spp) ao = add_rn(ao, occluded ? 0.0f : 1.0f);
                ++stage;
                ray_active = false;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// raygen, two-phase variant with RAY-level lane refill (VHR_OPT_RAYGEN_VARIANT 9): any-hit rays (shadow + AO)
// ---------------------------------------------------------------------------------------------------------------
// The per-pixel kernel traces one ray kind at a time and a warp iterates until its slowest ray is done: 15 of 32 lanes are active in an
// average instruction. The persistent variant above refills lanes with PIXELS, so its refill path carries the whole of raygen.rgen's ray
// generation at low utilisation and its per-lane state costs 96 registers (5 blocks / SM). Here the two jobs are separated:
//   A  every lane generates the rays of four pixels (its warp owns a 16 x 8 pixel block = four 8 x 4 tiles) exactly as raygen_kernel does —
//      same statements, same RNG order — and parks them in shared memory: origin per pixel, one direction per ray (12 B each);
//   B  the warp traverses its (1 + ao_spp) x 128 rays with per-lane refill: a lane whose ray is done takes the next ray of the warp's queue
//      (shadow rays of all lit pixels first, then the AO samples; a warp-uniform counter, no atomics) as soon as kRefill lanes are idle;
//      fetching a ray is two shared-memory loads + prepare(), nothing else. Any-hit answers land in a byte array;
//   C  every lane combines the answers of its four pixels and stores the texels.
// Same rays, same answers as raygen_kernel (an any-hit answer does not depend on when the ray is traced). Reflections (closest hit +
// shading) are not part of it: with them switched on the launcher runs raygen_kernel for that ray kind afterwards.
constexpr int kQueuePixels = 128;          // pixels per warp
struct QueueShared {                       // per warp; dynamic shared memory, sized by the launcher for (1 + ao_spp) ray kinds
    float o[kQueuePixels][3];              // origin = P + 0.1 N
    uint8_t list[kQueuePixels];            // lit pixels in queue order
};
template <int KINDS>                       // 1 + ao_spp (2, 3 or 5): ray kind 0 = shadow, k = AO sample k - 1
__global__ void __launch_bounds__(128, 8) raygen_queue_kernel(const __grid_constant__ RaygenParams p, const __grid_constant__ PerFrameData pfd, const int kRefill,
                                                              const int kBurst) {
    extern __shared__ __align__(16) unsigned char qsm[];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr size_t PER_WARP = sizeof(QueueShared) + (size_t)KINDS * kQueuePixels * 12 + (size_t)KINDS * kQueuePixels;
    unsigned char *base = qsm + (size_t)warp * ((PER_WARP + 15) & ~(size_t)15);
    QueueShared &q = *reinterpret_cast<QueueShared *>(base);
    float (*dirs)[3] = reinterpret_cast<float (*)[3]>(base + sizeof(QueueShared));                     // [KINDS * 128][3]
    uint8_t *occluded = base + sizeof(QueueShared) + (size_t)KINDS * kQueuePixels * 12;                // [KINDS * 128]
    // this warp's 16 x 8 pixel block inside the CTA's 32 x 16
    const int bx = blockIdx.x * 32 + (warp & 1) * 16, by = p.y_begin + blockIdx.y * 16 + (warp >> 1) * 8;
    const float3 L = make_float3(-pfd.directional_light.direction[0], -pfd.directional_light.direction[1], -pfd.directional_light.direction[2]);

    // ---- A: ray generation (raygen.rgen:15-55), four pixels per lane -------------------------------------------------------------------
    int n_lit = 0;
#pragma unroll 1
    for (int t = 0; t < 4; ++t) {
        const int i = t * 32 + lane;
        const int x = bx + (t & 1) * 8 + (lane & 7), y = by + (t >> 1) * 4 + (lane >> 3);
        const bool in_range = x < p.W && y < p.y_end;
        const size_t pix = in_range ? (size_t)y * p.W + x : 0;
        const float depth = in_range ? __ldg(&p.depth[pix]) : 0.0f;
        const bool lit = in_range && depth != 0.0f;
        if (in_range && !lit) {                                                                      // raygen.rgen:20-24
            p.shadow_ao[pix] = pack_rg16f(1.0f, 1.0f);
            p.reflections[pix] = make_uint2(0u, 0u);
            if (p.refl_t) p.refl_t[pix] = -1.0f;
        }
        if (lit) {
            const float u = __fdiv_rn(add_rn((float)x, 0.5f), (float)p.W), v = __fdiv_rn(add_rn((float)y, 0.5f), (float)p.H);
            uint32_t rng = seed_thread(((uint32_t)y * (uint32_t)p.H + (uint32_t)x) * pfd.frame_index);
            const float3 P = unproject_rn(pfd.camera_viewproj_inverse, depth, u, v);
            const float4 n4 = unpack_rgba16f(__ldg(&p.normals[pix]));
            const float3 N = make_float3(n4.x, n4.y, n4.z);
            q.o[i][0] = add_rn(P.x, mul_rn(N.x, 0.1f)); q.o[i][1] = add_rn(P.y, mul_rn(N.y, 0.1f)); q.o[i][2] = add_rn(P.z, mul_rn(N.z, 0.1f));
            float rnd1 = random01(rng), rnd2 = random01(rng);
            float3 d = onb_apply(L, normalize_rn(uniform_sample_cone(rnd1, rnd2, 0.999995f)));
            dirs[i][0] = d.x; dirs[i][1] = d.y; dirs[i][2] = d.z;
#pragma unroll
            for (int k = 1; k < KINDS; ++k) {
                rnd1 = random01(rng); rnd2 = random01(rng);
                d = onb_apply(N, uniform_sample_cosine_weighted_hemisphere(rnd1, rnd2));
                dirs[k * kQueuePixels + i][0] = d.x; dirs[k * kQueuePixels + i][1] = d.y; dirs[k * kQueuePixels + i][2] = d.z;
            }
        }
        const unsigned m = __ballot_sync(FULL, lit);
        if (lit) q.list[n_lit + __popc(m & ((1u << lane) - 1u))] = (uint8_t)i;
        n_lit += __popc(m);
    }
    __syncwarp();

    // ---- B: traversal with ray-level refill ------------------------------------------------------------------------------------------------
    // queue entry j: kind j / n_lit (skipping the kinds that are switched off), pixel list[j % n_lit]
    const int first_kind = (p.flags & 1) ? 0 : 1, end_kind = (p.flags & 2) ? KINDS : 1;
    const int n_rays = n_lit * max(end_kind - first_kind, 0);
    int next = 0;                                   // warp-uniform queue head
    bool active = false;
    int slot = 0;                                   // kind * 128 + pixel of the ray in flight
    RayPre r;
    r.o = make_float3(0.f, 0.f, 0.f); r.idir = r.o; r.kx = 0; r.ky = 1; r.kz = 2; r.Sx = r.Sy = r.Sz = 0.f; r.neg = 0u;
    float tmax = 0.0f;
    uint2 stack[kStackSize];
    int sp = 0;
    uint2 group = make_uint2(0u, 0u);
    const WideNode *__restrict__ nodes = p.scene.nodes;
    const float4 *__restrict__ tris = p.scene.tris;
    const uint32_t bias = p.scene.bias;
    while (true) {
        const unsigned idle = __ballot_sync(FULL, !active);
        if (idle == FULL || (next < n_rays && __popc(idle) >= kRefill)) {
            if (next >= n_rays) break;              // nothing in flight, nothing queued
            if (!active) {
                const int j = next + __popc(idle & ((1u << lane) - 1u));
                if (j < n_rays) {
                    const int kind = first_kind + j / n_lit, pixel = q.list[j - (j / n_lit) * n_lit];
                    slot = kind * kQueuePixels + pixel;
                    Ray ray;
                    ray.o = make_float3(q.o[pixel][0], q.o[pixel][1], q.o[pixel][2]);
                    ray.d = make_float3(dirs[slot][0], dirs[slot][1], dirs[slot][2]);
                    ray.tmin = 0.01f;
                    tmax = kind == 0 ? 10000.0f : 5.0f;
                    r = prepare(ray);
                    sp = 0;
                    group = make_uint2(0u, p.scene.n_wide ? 1u : 0u);
                    active = true;
                }
            }
            next += __popc(idle);
        }
#pragma unroll 1
        for (int it = 0; it < kBurst && active; ++it) {
            bool done = false, hit_any = false;
            if (group.y == 0u) {
                if (sp == 0) done = true;
                else group = stack[--sp];
            }
            if (!done) {
                const uint32_t k = pop_child<true>(group);
                if (group.y != 0u && sp < kStackSize) stack[sp++] = group;
                const uint32_t node = group.x + k;
                uint32_t child_base, child_hits, leaf_hits;
                intersect_node(nodes, node, r, 0.01f, tmax, bias, child_base, child_hits, leaf_hits);
                group = make_uint2(child_base & 0x7fffffffu, child_hits);
                if (leaf_hits) {
                    uint32_t tri_base, tri_hits;
                    expand_leaves(nodes, node, leaf_hits, tri_base, tri_hits);
                    do {
                        const uint32_t jt = (uint32_t)__ffs((int)tri_hits) - 1u;
                        tri_hits &= tri_hits - 1u;
                        const float4 *tp = tris + (size_t)(tri_base + jt) * 3;
                        const float4 v0 = VHR_TRI_LOAD(tp), v1 = VHR_TRI_LOAD(tp + 1), v2 = VHR_TRI_LOAD(tp + 2);
                        float tt, uu, vv;
                        if (intersect_tri(r, 0.01f, tmax, v0, v1, v2, tt, uu, vv)) { hit_any = true; done = true; break; }
                    } while (tri_hits);
                }
            }
            if (done) {
                occluded[slot] = hit_any ? 1 : 0;
                active = false;
            }
        }
    }
    __syncwarp();

    // ---- C: miss.rmiss / payload arithmetic of raygen.rgen:41-57 and the stores --------------------------------------------------------------
#pragma unroll 1
    for (int t = 0; t < 4; ++t) {
        const int i = t * 32 + lane;
        const int x = bx + (t & 1) * 8 + (lane & 7), y = by + (t >> 1) * 4 + (lane >> 3);
        if (!(x < p.W && y < p.y_end)) continue;
        const size_t pix = (size_t)y * p.W + x;
        if (__ldg(&p.depth[pix]) == 0.0f) continue;
        const float shadow = (p.flags & 1) ? (occluded[i] ? 0.0f : 1.0f) : 1.0f;
        float ao = 0.0f;
#pragma unroll
        for (int k = 1; k < KINDS; ++k) ao = add_rn(ao, (p.flags & 2) ? (occluded[k * kQueuePixels + i] ? 0.0f : 1.0f) : 1.0f);
        ao = __fdiv_rn(ao, (float)(KINDS - 1));
        p.shadow_ao[pix] = pack_rg16f(shadow, ao);
        if (!(p.flags & 4)) {
            p.reflections[pix] = make_uint2(0u, 0u);
            if (p.refl_t) p.refl_t[pix] = -1.0f;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// G-buffer producer (primary rays)
// ---------------------------------------------------------------------------------------------------------------
struct GbufferParams {
    int W, H;
    int y_begin, y_end;
    uint32_t *albedo;      // BGRA8
    uint2 *normals;
    uint2 *motion;
    float *depth;
    SceneRefs scene;
};
// multi-GPU (a partition with world > 1): this rank traces its rows and stores every texel into its own four images AND the same
// texel of every peer's, so each rank ends with the whole G-buffer. interleave = 1 (ray_block_rows = 8): the 8-row blocks b with
// b % world == rank, exactly the blocks this rank's ray pass traces; interleave = 0: the rank's band [y_begin, y_end).
struct GbufferPartParams : GbufferParams {
    int world, rank, interleave;
    uint32_t *albedo_of[VHR_MAX_RANKS];      // [rank] = this rank's own image
    uint2 *normals_of[VHR_MAX_RANKS];
    uint2 *motion_of[VHR_MAX_RANKS];
    float *depth_of[VHR_MAX_RANKS];
};

__device__ __forceinline__ uint32_t unorm8(float f) {
    f = fminf(fmaxf(f, 0.0f), 1.0f);
    return (uint32_t)__float2int_rn(f * 255.0f);
}

// The any-hit stage of the primary ray = the discards of gbuf.frag:19-32: a fragment whose albedo alpha is below the
// cutoff of an alpha-masked material, or exactly 0, is dropped and whatever lies behind it shows.
struct AlphaTest {
    const SceneRefs &s;
    __device__ __forceinline__ bool operator()(uint32_t tri, float u, float v) const {
        const float4 *tp = s.tris + (size_t)tri * 3;
        const uint32_t g = __float_as_uint(__ldg(tp).w), pid = __float_as_uint(__ldg(tp + 1).w);
        const Primitive &prim = s.prims[g];
        float alpha = prim.material.base_color[3];
        if (has_texture(s, prim.material.base_color_texture)) {
            const Vertex &v0 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 0]];
            const Vertex &v1 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 1]];
            const Vertex &v2 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 2]];
            const float2 uv = bary_uv(v0, v1, v2, sub_rn(sub_rn(1.0f, u), v), u, v);
            alpha = sample_texture(s.textures, s.lut, prim.material.base_color_texture, uv.x, uv.y).w;
        }
        if (prim.material.alpha_mask == 1 && alpha < prim.material.alpha_cutoff) return false;
        return alpha != 0.0f;
    }
};
__device__ __forceinline__ float3 cross_rn(float3 a, float3 b) {
    return make_float3(sub_rn(mul_rn(a.y, b.z), mul_rn(a.z, b.y)), sub_rn(mul_rn(a.z, b.x), mul_rn(a.x, b.z)), sub_rn(mul_rn(a.x, b.y), mul_rn(a.y, b.x)));
}

// partitioned instance: the texel goes to the same place in every rank's image (of[rank] is this rank's own)
template <typename T>
__device__ __forceinline__ void store_every_rank(T *const *of, int world, size_t i, T v) {
#pragma unroll
    for (int r = 0; r < VHR_MAX_RANKS; ++r)
        if (r < world) of[r][i] = v;
}

// PART = false: the single-GPU pass over the rows [y_begin, y_end). PART = true (GbufferPartParams): the rows dealt to this rank,
// every texel stored to every rank; the per-pixel arithmetic is the same.
template <bool PART>
__global__ void __launch_bounds__(128) gbuffer_kernel(const __grid_constant__ std::conditional_t<PART, GbufferPartParams, GbufferParams> p,
                                                      const __grid_constant__ PerFrameData pfd) {
    int x, y;
    tile_coords(x, y);
    if constexpr (PART) {
        if (p.interleave)      // blockIdx.y counts this rank's 8-row blocks, dealt as raygen_kernel deals them
            y = (y - blockIdx.y * 8) + (blockIdx.y * p.world + p.rank) * 8;
        else
            y += p.y_begin;
    } else {
        y += p.y_begin;
    }
    const bool in_range = x < p.W && y < p.y_end;       // trace() is warp-synchronous: no early return
    const size_t pix = in_range ? (size_t)y * p.W + x : 0;
    const float u = mul_rn(add_rn((float)x, 0.5f), pfd.display_size_inverse[0]);
    const float v = mul_rn(add_rn((float)y, 0.5f), pfd.display_size_inverse[1]);
    const float3 cam = make_float3(pfd.camera_view_inverse[12], pfd.camera_view_inverse[13], pfd.camera_view_inverse[14]);
    const float3 pn = unproject_rn(pfd.camera_viewproj_inverse, 1.0f, u, v);   // near plane (reverse-Z: depth 1)
    Ray ray;
    ray.o = cam;
    ray.d = make_float3(sub_rn(pn.x, cam.x), sub_rn(pn.y, cam.y), sub_rn(pn.z, cam.z));
    ray.tmin = 1.0f;
    ray.tmax = 3.0e38f;
    Hit h;
    const bool found = trace<false>(p.scene.nodes, p.scene.tris, p.scene.n_wide, p.scene.bias, ray, in_range, h, AlphaTest{p.scene});
    if (!in_range) return;
    if (!found) {
        // clear values of hybrid_render_path.cpp:16-19
        if constexpr (PART) {
            store_every_rank(p.albedo_of, p.world, pix, 0u);
            store_every_rank(p.normals_of, p.world, pix, make_uint2(0u, 0u));
            store_every_rank(p.motion_of, p.world, pix, pack_rgba16f(make_float4(0.0f, 0.0f, -1.0f, -1.0f)));
            store_every_rank(p.depth_of, p.world, pix, 0.0f);
        } else {
            if (p.albedo) p.albedo[pix] = 0u;
            p.normals[pix] = make_uint2(0u, 0u);
            p.motion[pix] = pack_rgba16f(make_float4(0.0f, 0.0f, -1.0f, -1.0f));
            p.depth[pix] = 0.0f;
        }
        return;
    }
    const SceneRefs &s = p.scene;
    const float4 *tp = s.tris + (size_t)h.tri * 3;
    const uint32_t g = __float_as_uint(__ldg(tp).w), pid = __float_as_uint(__ldg(tp + 1).w);
    const Primitive &prim = s.prims[g];
    const Vertex &v0 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 0]];
    const Vertex &v1 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 1]];
    const Vertex &v2 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 2]];
    const float b1 = h.u, b2 = h.v, b0 = sub_rn(sub_rn(1.0f, b1), b2);
    float3 nobj = bary3(f3(v0.normal), f3(v1.normal), f3(v2.normal), b0, b1, b2);
    const float3 pobj = bary3(f3(v0.pos), f3(v1.pos), f3(v2.pos), b0, b1, b2);
    const Material &mat = prim.material;
    const bool tex_a = has_texture(s, mat.base_color_texture), tex_n = has_texture(s, mat.normal_map), tex_mr = has_texture(s, mat.metallic_roughness_texture);
    float4 albedo = make_float4(mat.base_color[0], mat.base_color[1], mat.base_color[2], mat.base_color[3]);
    float metallic = mat.metallic_factor, roughness = mat.roughness_factor;
    if (tex_a || tex_n || tex_mr) {
        const float2 uv = bary_uv(v0, v1, v2, b0, b1, b2);
        if (tex_a) albedo = sample_texture(s.textures, s.lut, mat.base_color_texture, uv.x, uv.y);                  // gbuf.frag:24-26
        if (tex_n) {                                                                                               // gbuf.frag:35-41
            const float4 c = sample_texture(s.textures, s.lut, mat.normal_map, uv.x, uv.y);
            const float3 tsn = normalize_rn(make_float3(sub_rn(mul_rn(c.x, 2.0f), 1.0f), sub_rn(mul_rn(c.y, 2.0f), 1.0f), sub_rn(mul_rn(c.z, 2.0f), 1.0f)));
            const float3 tan3 = bary3(f3(v0.tangent), f3(v1.tangent), f3(v2.tangent), b0, b1, b2);
            const float tw = add_rn(add_rn(mul_rn(v0.tangent[3], b0), mul_rn(v1.tangent[3], b1)), mul_rn(v2.tangent[3], b2));
            const float3 cr = cross_rn(tsn, tan3);
            const float3 bitangent = make_float3(mul_rn(cr.x, tw), mul_rn(cr.y, tw), mul_rn(cr.z, tw));
            const float tn = dot3_rn(tan3, nobj);
            const float3 tangent = normalize_rn(make_float3(sub_rn(tan3.x, mul_rn(nobj.x, tn)), sub_rn(tan3.y, mul_rn(nobj.y, tn)), sub_rn(tan3.z, mul_rn(nobj.z, tn))));
            nobj = make_float3(add_rn(add_rn(mul_rn(tangent.x, tsn.x), mul_rn(bitangent.x, tsn.y)), mul_rn(nobj.x, tsn.z)),
                               add_rn(add_rn(mul_rn(tangent.y, tsn.x), mul_rn(bitangent.y, tsn.y)), mul_rn(nobj.y, tsn.z)),
                               add_rn(add_rn(mul_rn(tangent.z, tsn.x), mul_rn(bitangent.z, tsn.y)), mul_rn(nobj.z, tsn.z)));
        }
        if (tex_mr) {                                                                                              // gbuf.frag:52-56
            const float4 c = sample_texture(s.textures, s.lut, mat.metallic_roughness_texture, uv.x, uv.y);
            metallic = mul_rn(metallic, c.y);
            roughness = mul_rn(roughness, c.z);
        }
    }
    const float *nm = s.normal_mats + (size_t)g * 9;
    float3 nw = make_float3(add_rn(add_rn(mul_rn(nm[0], nobj.x), mul_rn(nm[3], nobj.y)), mul_rn(nm[6], nobj.z)),
                            add_rn(add_rn(mul_rn(nm[1], nobj.x), mul_rn(nm[4], nobj.y)), mul_rn(nm[7], nobj.z)),
                            add_rn(add_rn(mul_rn(nm[2], nobj.x), mul_rn(nm[5], nobj.y)), mul_rn(nm[8], nobj.z)));
    nw = normalize_rn(nw);
    const float4 pw = mul44_rn(prim.transform, make_float4(pobj.x, pobj.y, pobj.z, 1.0f));
    const float4 clip = mul44_rn(pfd.camera_proj, mul44_rn(pfd.camera_view, pw));
    const float4 pclip = mul44_rn(pfd.camera_proj_prev_frame, mul44_rn(pfd.camera_view_prev_frame, pw));
    const float pu = add_rn(mul_rn(__fdiv_rn(pclip.x, pclip.w), 0.5f), 0.5f);
    const float pv = add_rn(mul_rn(__fdiv_rn(pclip.y, pclip.w), 0.5f), 0.5f);
    if constexpr (PART) {
        store_every_rank(p.albedo_of, p.world, pix, unorm8(albedo.z) | (unorm8(albedo.y) << 8) | (unorm8(albedo.x) << 16) | (unorm8(albedo.w) << 24));
        store_every_rank(p.normals_of, p.world, pix, pack_rgba16f(make_float4(nw.x, nw.y, nw.z, (float)g)));
        store_every_rank(p.motion_of, p.world, pix, pack_rgba16f(make_float4(sub_rn(u, pu), sub_rn(v, pv), metallic, roughness)));
        store_every_rank(p.depth_of, p.world, pix, __fdiv_rn(clip.z, clip.w));
    } else {
        if (p.albedo) p.albedo[pix] = unorm8(albedo.z) | (unorm8(albedo.y) << 8) | (unorm8(albedo.x) << 16) | (unorm8(albedo.w) << 24);
        p.normals[pix] = pack_rgba16f(make_float4(nw.x, nw.y, nw.z, (float)g));
        p.motion[pix] = pack_rgba16f(make_float4(sub_rn(u, pu), sub_rn(v, pv), metallic, roughness));
        p.depth[pix] = __fdiv_rn(clip.z, clip.w);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The fully ray-traced render path (SURVEY 8f rank 4): raytraced_render_path/raygen.rgen:11-23 + closesthit.rchit:10-58 +
// miss.rmiss:6-8 + shadow_miss.rmiss:6-8, and the alpha-tested pipeline raygen_test_alpha.rgen / closesthit_test_alpha.rchit /
// shadow_anyhit.rahit:9-27 ("Raytracing Pass", src/render_paths/raytraced_render_path.cpp:12-47)
// ---------------------------------------------------------------------------------------------------------------
struct RaytracedParams {
    int W, H;
    int y_begin, y_end;
    uint32_t *out;            // binding 0: "RaytracedOutput", B8G8R8A8_UNORM storage image
    SceneRefs scene;
};

// shadow_anyhit.rahit:22-26: a candidate whose base-colour texel is below the cutoff of an alpha-masked material is ignored
// (ignoreIntersectionEXT). The shader samples textures[base_color_texture] unconditionally; without a texture (index -1, an
// out-of-bounds descriptor in the reference) the candidate counts as opaque here.
struct RahitAlphaTest {
    const SceneRefs &s;
    __device__ __forceinline__ bool operator()(uint32_t tri, float u, float v) const {
        const float4 *tp = s.tris + (size_t)tri * 3;
        const uint32_t g = __float_as_uint(__ldg(tp).w), pid = __float_as_uint(__ldg(tp + 1).w);
        const Primitive &prim = s.prims[g];
        if (prim.material.alpha_mask != 1 || !has_texture(s, prim.material.base_color_texture)) return true;
        const Vertex &v0 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 0]];
        const Vertex &v1 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 1]];
        const Vertex &v2 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 2]];
        const float2 uv = bary_uv(v0, v1, v2, sub_rn(sub_rn(1.0f, u), v), u, v);
        return !(sample_texture(s.textures, s.lut, prim.material.base_color_texture, uv.x, uv.y).w < prim.material.alpha_cutoff);
    }
};

template <bool ALPHA>
__global__ void __launch_bounds__(128) raytraced_kernel(const __grid_constant__ RaytracedParams p, const __grid_constant__ PerFrameData pfd) {
    int x, y;
    tile_coords(x, y);
    y += p.y_begin;
    const bool in_range = x < p.W && y < p.y_end;       // trace() is warp-synchronous: no early return
    const SceneRefs &s = p.scene;
    // raygen.rgen:12-18
    const float u = sub_rn(mul_rn(__fdiv_rn(add_rn((float)x, 0.5f), (float)p.W), 2.0f), 1.0f);
    const float v = sub_rn(mul_rn(__fdiv_rn(add_rn((float)y, 0.5f), (float)p.H), 2.0f), 1.0f);
    const float4 o4 = mul44_rn(pfd.camera_view_inverse, make_float4(0.0f, 0.0f, 0.0f, 1.0f));
    const float4 target = mul44_rn(pfd.camera_proj_inverse, make_float4(u, v, 1.0f, 1.0f));
    const float3 tn = normalize_rn(make_float3(target.x, target.y, target.z));
    const float4 d4 = mul44_rn(pfd.camera_view_inverse, make_float4(tn.x, tn.y, tn.z, 0.0f));
    Ray ray;
    ray.o = make_float3(o4.x, o4.y, o4.z);
    ray.d = make_float3(d4.x, d4.y, d4.z);
    ray.tmin = 0.1f;
    ray.tmax = 10000.0f;
    Hit h;
    const bool found = ALPHA ? trace<false>(s.nodes, s.tris, s.n_wide, s.bias, ray, in_range, h, RahitAlphaTest{s})
                             : trace<false>(s.nodes, s.tris, s.n_wide, s.bias, ray, in_range, h);
    float4 payload = make_float4(0.3f, 0.8f, 0.2f, 1.0f);                                    // miss.rmiss:7
    Ray sray;
    sray.o = make_float3(0.0f, 0.0f, 0.0f); sray.d = make_float3(0.0f, 1.0f, 0.0f); sray.tmin = 0.1f; sray.tmax = 10000.0f;
    float3 albedo = make_float3(0.0f, 0.0f, 0.0f), N = make_float3(0.0f, 0.0f, 0.0f);
    const float3 L = make_float3(-pfd.directional_light.direction[0], -pfd.directional_light.direction[1], -pfd.directional_light.direction[2]);
    const bool shade = in_range && found;
    if (shade) {                                                                             // closesthit.rchit:11-41
        const float4 *tp = s.tris + (size_t)h.tri * 3;
        const uint32_t g = __float_as_uint(__ldg(tp).w), pid = __float_as_uint(__ldg(tp + 1).w);
        const Primitive &prim = s.prims[g];
        const Vertex &v0 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 0]];
        const Vertex &v1 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 1]];
        const Vertex &v2 = s.verts[prim.vertex_offset + s.indices[prim.index_offset + 3 * pid + 2]];
        const float b1 = h.u, b2 = h.v, b0 = sub_rn(sub_rn(1.0f, b1), b2);
        const float2 uv = bary_uv(v0, v1, v2, b0, b1, b2);
        const float3 normal = bary3(f3(v0.normal), f3(v1.normal), f3(v2.normal), b0, b1, b2);
        const float3 pobj = bary3(f3(v0.pos), f3(v1.pos), f3(v2.pos), b0, b1, b2);
        const float4 pw = mul44_rn(prim.transform, make_float4(pobj.x, pobj.y, pobj.z, 1.0f));
        albedo = make_float3(prim.material.base_color[0], prim.material.base_color[1], prim.material.base_color[2]);
        if (has_texture(s, prim.material.base_color_texture)) {
            const float4 c = sample_texture(s.textures, s.lut, prim.material.base_color_texture, uv.x, uv.y);
            albedo = make_float3(c.x, c.y, c.z);
        }
        N = normal;
        if (has_texture(s, prim.material.normal_map)) {
            const float3 tan3 = bary3(f3(v0.tangent), f3(v1.tangent), f3(v2.tangent), b0, b1, b2);
            const float tw = add_rn(add_rn(mul_rn(v0.tangent[3], b0), mul_rn(v1.tangent[3], b1)), mul_rn(v2.tangent[3], b2));
            const float4 c = sample_texture(s.textures, s.lut, prim.material.normal_map, uv.x, uv.y);
            const float3 tsn = normalize_rn(make_float3(sub_rn(mul_rn(c.x, 2.0f), 1.0f), sub_rn(mul_rn(c.y, 2.0f), 1.0f), sub_rn(mul_rn(c.z, 2.0f), 1.0f)));
            const float3 cr = cross_rn(tsn, tan3);
            const float3 bitangent = make_float3(mul_rn(cr.x, tw), mul_rn(cr.y, tw), mul_rn(cr.z, tw));
            const float tdn = dot3_rn(tan3, normal);
            const float3 tangent = normalize_rn(make_float3(sub_rn(tan3.x, mul_rn(normal.x, tdn)), sub_rn(tan3.y, mul_rn(normal.y, tdn)), sub_rn(tan3.z, mul_rn(normal.z, tdn))));
            N = make_float3(add_rn(add_rn(mul_rn(tangent.x, tsn.x), mul_rn(bitangent.x, tsn.y)), mul_rn(normal.x, tsn.z)),
                            add_rn(add_rn(mul_rn(tangent.y, tsn.x), mul_rn(bitangent.y, tsn.y)), mul_rn(normal.y, tsn.z)),
                            add_rn(add_rn(mul_rn(tangent.z, tsn.x), mul_rn(bitangent.z, tsn.y)), mul_rn(normal.z, tsn.z)));
        }
        sray.o = make_float3(pw.x, pw.y, pw.z);
        sray.d = L;
    }
    // closesthit.rchit:48-50: the shadow ray (miss index 1 clears shadow_payload). Every lane takes part; only shaded ones are alive.
    Hit sh;
    const bool occluded = ALPHA ? trace<true>(s.nodes, s.tris, s.n_wide, s.bias, sray, shade, sh, RahitAlphaTest{s})
                                : trace<true>(s.nodes, s.tris, s.n_wide, s.bias, sray, shade, sh);
    if (!in_range) return;
    if (shade) {
        const float amb = ALPHA ? 0.2f : VHR_PI_INVERSE;                                     // closesthit_test_alpha.rchit:39 / closesthit.rchit:46
        float3 c = make_float3(mul_rn(amb, albedo.x), mul_rn(amb, albedo.y), mul_rn(amb, albedo.z));
        if (!occluded) {
            const float ndl = fmaxf(dot3_rn(N, L), 0.0f);
            const float *li = pfd.directional_light.intensity, *lc = pfd.directional_light.color;
            if (ALPHA) {
                c = make_float3(add_rn(c.x, mul_rn(mul_rn(ndl, albedo.x), lc[0])), add_rn(c.y, mul_rn(mul_rn(ndl, albedo.y), lc[1])),
                                add_rn(c.z, mul_rn(mul_rn(ndl, albedo.z), lc[2])));
            } else {
                c = make_float3(add_rn(c.x, mul_rn(mul_rn(mul_rn(ndl, albedo.x), li[0]), lc[0])), add_rn(c.y, mul_rn(mul_rn(mul_rn(ndl, albedo.y), li[1]), lc[1])),
                                add_rn(c.z, mul_rn(mul_rn(mul_rn(ndl, albedo.z), li[2]), lc[2])));
            }
        }
        payload = make_float4(c.x, c.y, c.z, 1.0f);
    }
    // imageStore to a B8G8R8A8_UNORM image: float -> UNORM8 (NaN -> 0), B in the low byte
    auto q = [](float f) { f = (f == f) ? fminf(fmaxf(f, 0.0f), 1.0f) : 0.0f; return (uint32_t)__float2int_rn(f * 255.0f); };
    p.out[(size_t)y * p.W + x] = q(payload.z) | (q(payload.y) << 8) | (q(payload.x) << 16) | (q(payload.w) << 24);
}

// ---------------------------------------------------------------------------------------------------------------
// explicit rays (tests)
// ---------------------------------------------------------------------------------------------------------------
__global__ void trace_explicit_kernel(const float *__restrict__ rays, uint32_t n, int any_hit, SceneRefs s, float *out_t,
                                      uint32_t *out_ids, float *out_uv) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = i < n;                         // trace() is warp-synchronous: no early return
    const uint32_t ii = in_range ? i : 0u;
    Ray r;
    r.o = make_float3(rays[8 * ii + 0], rays[8 * ii + 1], rays[8 * ii + 2]);
    r.tmin = rays[8 * ii + 3];
    r.d = make_float3(rays[8 * ii + 4], rays[8 * ii + 5], rays[8 * ii + 6]);
    r.tmax = rays[8 * ii + 7];
    Hit h;
    h.t = -1.0f; h.u = 0.0f; h.v = 0.0f; h.tri = 0xffffffffu;
    if (any_hit) {      // uniform across the launch
        const bool occluded = trace<true>(s.nodes, s.tris, s.n_wide, s.bias, r, in_range, h);
        if (in_range) out_t[i] = occluded ? 1.0f : 0.0f;
        return;
    }
    bool found = trace<false>(s.nodes, s.tris, s.n_wide, s.bias, r, in_range, h);
    if (!in_range) return;
    out_t[i] = found ? h.t : -1.0f;
    if (out_ids) {
        out_ids[2 * i] = found ? __float_as_uint(s.tris[(size_t)h.tri * 3].w) : 0xffffffffu;
        out_ids[2 * i + 1] = found ? __float_as_uint(s.tris[(size_t)h.tri * 3 + 1].w) : 0xffffffffu;
    }
    if (out_uv) { out_uv[2 * i] = h.u; out_uv[2 * i + 1] = h.v; }
}

SceneRefs scene_refs(vhr_context *ctx) {
    SceneRefs s;
    s.verts = ctx->d_vertices; s.indices = ctx->d_indices; s.prims = ctx->d_primitives;
    s.normal_mats = ctx->d_normal_mats;
    s.nodes = (const WideNode *)ctx->bvh.wide_nodes; s.tris = ctx->bvh.tri_verts; s.n_wide = ctx->bvh.n_wide;
    s.bias = 0x47000000u;
    s.textures = ctx->d_textures; s.lut = ctx->d_texel_lut; s.n_textures = ctx->d_textures ? VHR_MAX_GLOBAL_RESOURCES : 0u;
    return s;
}

bool band(vhr_context *ctx, uint32_t height, int &y0, int &y1) {
    y0 = std::max(0, ctx->opt.row_begin);
    y1 = ctx->opt.row_end < 0 ? (int)height : std::min((int)height, ctx->opt.row_end);
    return y1 > y0;
}

}  // namespace

int launch_trace_rays(vhr_context *ctx, uint32_t width, uint32_t height) {
    // descriptor set 3 of the "Raytrace Pass" (hybrid_render_path.cpp:102-110): 0 normals, 1 depth, 2 shadow/AO, 3 reflections
    if (ctx->n_bound < 4) return fail(VHR_ERR_STATE, "TraceRays: pass images not bound (need bindings 0..3)");
    if (!ctx->d_primitives && ctx->bvh.n_tris) return fail(VHR_ERR_STATE, "TraceRays: geometry not uploaded");
    Image *normals = ctx->bound[0], *depth = ctx->bound[1], *sa = ctx->bound[2], *refl = ctx->bound[3];
    if (normals->format != VHR_FORMAT_R16G16B16A16_SFLOAT || depth->format != VHR_FORMAT_D32_SFLOAT ||
        sa->format != VHR_FORMAT_R16G16_SFLOAT || refl->format != VHR_FORMAT_R16G16B16A16_SFLOAT)
        return fail(VHR_ERR_INVALID, "TraceRays: unexpected image formats");
    for (Image *im : {normals, depth, sa, refl})
        if (im->width != width || im->height != height)
            return fail(VHR_ERR_INVALID, "TraceRays: launch size %ux%u differs from image %ux%u", width, height, im->width, im->height);
    for (Image *im : {sa, refl})
        if (int rc = make_writable(ctx, im, covers_image(ctx, im, width, height))) return rc;
    RaygenParams p;
    p.W = (int)width; p.H = (int)height;
    if (!band(ctx, height, p.y_begin, p.y_end)) return VHR_OK;
    p.ao_spp = ctx->opt.ao_spp;
    p.flags = (ctx->opt.trace_shadows ? 1 : 0) | (ctx->opt.trace_ao ? 2 : 0) | (ctx->opt.trace_reflections ? 4 : 0);
    p.normals = (const uint2 *)normals->ptr; p.depth = (const float *)depth->ptr;
    p.shadow_ao = (uint32_t *)sa->ptr; p.reflections = (uint2 *)refl->ptr;
    p.refl_t = ctx->opt.debug_refl_t ? ctx->d_refl_t : nullptr;
    p.scene = scene_refs(ctx);
    p.world = 0; p.rank = 0;
    const Partition &pt = ctx->part;
    if (pt.enabled && pt.world > 1 && pt.ray_block_rows == 8) {
        p.world = pt.world; p.rank = pt.rank;
        p.y_begin = 0; p.y_end = (int)height;
        for (int r = 0; r <= pt.world; ++r) p.band_begin[r] = pt.band_begin[r];
        for (int r = 0; r < pt.world; ++r) {
            p.shadow_ao_of[r] = (uint32_t *)(r == pt.rank ? sa->ptr : sa->peer[r]);
            p.reflections_of[r] = (uint2 *)(r == pt.rank ? refl->ptr : refl->peer[r]);
            if (!p.shadow_ao_of[r] || !p.reflections_of[r])
                return fail(VHR_ERR_STATE, "TraceRays: rank %d's output images are not attached (vhr_image_attach_peer)", r);
        }
        const int n_blocks = ((int)height + 7) / 8;
        const int mine = (n_blocks - pt.rank + pt.world - 1) / pt.world;          // blocks b = rank, rank + world, ...
        dim3 block(128), grid((width + 15) / 16, mine);
        if (mine > 0) {
            raygen_kernel<8><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
            VHR_CUDA_CHECK(cudaGetLastError());
            ctx->launches++;
        }
        return peer_sync_all(ctx);      // every rank's rows have landed in their owners' images before anyone reads them
    }
    if (ctx->opt.raygen_variant == 1 && p.ao_spp >= 1) {
        if (!ctx->d_ray_queue) VHR_CUDA_CHECK(cudaMalloc(&ctx->d_ray_queue, sizeof(uint32_t)));
        if (ctx->raygen_blocks == 0) {
            int per_sm = 0, sms = 0;
            VHR_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, raygen_persistent_kernel, 128, 0));
            VHR_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
            ctx->raygen_blocks = std::max(1, per_sm) * std::max(1, sms);     // one resident wave: 148 SMs x blocks/SM
        }
        VHR_CUDA_CHECK(cudaMemsetAsync(ctx->d_ray_queue, 0, sizeof(uint32_t), ctx->stream));
        raygen_persistent_kernel<<<ctx->raygen_blocks, 128, 0, ctx->stream>>>(p, ctx->pfd, ctx->d_ray_queue, getenv("VHR_REFILL_IDLE") ? atoi(getenv("VHR_REFILL_IDLE")) : 16, getenv("VHR_BURST") ? atoi(getenv("VHR_BURST")) : 4);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
        return VHR_OK;
    }
    dim3 block(128), grid((width + 15) / 16, (p.y_end - p.y_begin + 7) / 8);
    p.leaf_batch = getenv("VHR_LEAF_BATCH") ? atoi(getenv("VHR_LEAF_BATCH")) : 16;
    if (ctx->opt.raygen_variant == 9 && (p.ao_spp == 1 || p.ao_spp == 2 || p.ao_spp == 4) && (p.flags & 3)) {
        // any-hit rays through the ray queue kernel; the reflection ray (closest hit + shading), if on, through the per-pixel kernel afterwards
        const int kinds = 1 + p.ao_spp;
        const size_t per_warp = (sizeof(QueueShared) + (size_t)kinds * kQueuePixels * 12 + (size_t)kinds * kQueuePixels + 15) & ~(size_t)15;
        const size_t smem = 4 * per_warp;
        const int refill = getenv("VHR_REFILL_IDLE") ? atoi(getenv("VHR_REFILL_IDLE")) : 8, burst = getenv("VHR_BURST") ? atoi(getenv("VHR_BURST")) : 4;
        dim3 qgrid((width + 31) / 32, (p.y_end - p.y_begin + 15) / 16);
        RaygenParams pq = p;
        pq.flags = p.flags & 7;
#define VHR_LAUNCH_QUEUE(K)                                                                                                         \
        do {                                                                                                                        \
            static uint64_t configured = 0;                                                                                         \
            if (!(configured >> (ctx->device & 63) & 1ull)) {                                                                       \
                VHR_CUDA_CHECK(cudaFuncSetAttribute(raygen_queue_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
                configured |= 1ull << (ctx->device & 63);                                                                           \
            }                                                                                                                       \
            raygen_queue_kernel<K><<<qgrid, block, smem, ctx->stream>>>(pq, ctx->pfd, refill, burst);                               \
        } while (0)
        if (kinds == 2) VHR_LAUNCH_QUEUE(2);
        else if (kinds == 3) VHR_LAUNCH_QUEUE(3);
        else VHR_LAUNCH_QUEUE(5);
#undef VHR_LAUNCH_QUEUE
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
        if (p.flags & 4) {
            RaygenParams pr = p;
            pr.flags = 4 | 8;                      // reflection ray only, leave the shadow / AO texel alone
            raygen_kernel<8><<<grid, block, 0, ctx->stream>>>(pr, ctx->pfd);
            VHR_CUDA_CHECK(cudaGetLastError());
            ctx->launches++;
        }
        return VHR_OK;
    }
    switch (ctx->opt.raygen_variant) {
        case 2: raygen_kernel<0><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;          // ptxas' own register choice (72)
        case 3: raygen_kernel<1><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;          // no register cap (117)
        case 4: raygen_kernel<8, true><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;    // postponed leaves
        case 8: raygen_kernel<8, false, 4, true><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;              // AO rays sorted by direction in the CTA
        case 6: raygen_kernel<8, false, 1><<<dim3(grid.x * 4, grid.y), 32, 0, ctx->stream>>>(p, ctx->pfd); break;   // one-warp CTAs, 32 / SM
        case 7: raygen_kernel<8, false, 2><<<dim3(grid.x * 2, grid.y), 64, 0, ctx->stream>>>(p, ctx->pfd); break;   // two-warp CTAs, 16 / SM
        case 12:                                                                                 // 4-byte stack entries (trees below 2^23 wide nodes)
            if (ctx->bvh.n_wide < (1u << 23)) { raygen_kernel<8, false, 4, false, true><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break; }
            raygen_kernel<8><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;
        case 13: raygen_kernel<8, false, 4, false, false, true><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;   // one inlined any-hit traversal for shadow + AO
        case 14: raygen_kernel<8, false, 4, false, false, false, 8><<<grid, block, 8 * sizeof(uint2) * 128, ctx->stream>>>(p, ctx->pfd); break;     // first 8 stack entries in shared memory
        case 15: raygen_kernel<8, false, 4, false, false, false, 12><<<grid, block, 12 * sizeof(uint2) * 128, ctx->stream>>>(p, ctx->pfd); break;   // first 12
        case 10: raygen_kernel<10><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;        // 48 registers, 10 blocks / SM
        case 11: raygen_kernel<12><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;        // 40 registers, 12 blocks / SM
        default: raygen_kernel<8><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd); break;         // 64 registers, 8 blocks / SM
    }
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

int launch_raytraced(vhr_context *ctx, uint32_t width, uint32_t height) {
    // descriptor set 3 of the "Raytracing Pass" (raytraced_render_path.cpp:13-16): 0 RaytracedOutput
    if (ctx->n_bound < 1 || !ctx->bound[0]) return fail(VHR_ERR_STATE, "Raytracing Pipeline: output image not bound");
    if (!ctx->d_primitives && ctx->bvh.n_tris) return fail(VHR_ERR_STATE, "TraceRays: geometry not uploaded");
    Image *out = ctx->bound[0];
    if (out->format != VHR_FORMAT_B8G8R8A8_UNORM) return fail(VHR_ERR_INVALID, "Raytracing Pipeline: output format %d, expected B8G8R8A8_UNORM", out->format);
    if (out->width != width || out->height != height)
        return fail(VHR_ERR_INVALID, "TraceRays: launch size %ux%u differs from image %ux%u", width, height, out->width, out->height);
    if (int rc = make_writable(ctx, out, covers_image(ctx, out, width, height))) return rc;
    RaytracedParams p;
    p.W = (int)width; p.H = (int)height;
    if (!band(ctx, height, p.y_begin, p.y_end)) return VHR_OK;
    p.out = (uint32_t *)out->ptr;
    p.scene = scene_refs(ctx);
    dim3 block(128), grid((width + 15) / 16, (p.y_end - p.y_begin + 7) / 8);
    if (ctx->opt.raytraced_alpha_test) raytraced_kernel<true><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
    else raytraced_kernel<false><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    return VHR_OK;
}

int launch_gbuffer(vhr_context *ctx, uint32_t width, uint32_t height) {
    if (ctx->n_bound < 4) return fail(VHR_ERR_STATE, "G-buffer pass: images not bound (need bindings 0..3)");
    Image *albedo = ctx->bound[0], *normals = ctx->bound[1], *motion = ctx->bound[2], *depth = ctx->bound[3];
    if (albedo->format != VHR_FORMAT_B8G8R8A8_UNORM || normals->format != VHR_FORMAT_R16G16B16A16_SFLOAT ||
        motion->format != VHR_FORMAT_R16G16B16A16_SFLOAT || depth->format != VHR_FORMAT_D32_SFLOAT)
        return fail(VHR_ERR_INVALID, "G-buffer pass: unexpected image formats");
    for (Image *im : {albedo, normals, motion, depth})
        if (im->width != width || im->height != height) return fail(VHR_ERR_INVALID, "G-buffer pass: image size mismatch");
    for (Image *im : {albedo, normals, motion, depth})      // e.g. the normals image still shared with the SVGF pass's previous-frame copy
        if (int rc = make_writable(ctx, im, covers_image(ctx, im, width, height))) return rc;
    GbufferPartParams p;      // its GbufferParams part is all the single-GPU instance takes
    p.W = (int)width; p.H = (int)height;
    if (!band(ctx, height, p.y_begin, p.y_end)) return VHR_OK;
    p.albedo = (uint32_t *)albedo->ptr; p.normals = (uint2 *)normals->ptr; p.motion = (uint2 *)motion->ptr; p.depth = (float *)depth->ptr;
    p.scene = scene_refs(ctx);
    const Partition &pt = ctx->part;
    if (!(pt.enabled && pt.world > 1)) {
        dim3 block(128), grid((width + 15) / 16, (p.y_end - p.y_begin + 7) / 8);
        gbuffer_kernel<false><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
        return VHR_OK;
    }
    // Partitioned: this rank's rows go to every rank's images (include/vhr_b200.h). Every peer image must be attached before
    // anything is enqueued, so that a failing call leaves no flag written and no stream waiting.
    Image *const imgs[4] = {albedo, normals, motion, depth};
    for (int i = 0; i < 4; ++i)
        for (int r = 0; r < pt.world; ++r)
            if (r != pt.rank && !imgs[i]->peer[r])
                return fail(VHR_ERR_STATE, "G-buffer pass: binding %d (%s) has no image of rank %d attached (vhr_image_attach_peer)", i,
                            image_label(ctx, imgs[i]).c_str(), r);
    // Load the kernel before a flag wait is enqueued: with lazy module loading its first launch would otherwise wait for this stream, which
    // then waits for the other ranks — a deadlock when they are contexts driven by this same thread and have not issued their signals yet.
    static uint64_t loaded = 0;
    if (!(loaded >> (ctx->device & 63) & 1ull)) {
        cudaFuncAttributes attr;
        VHR_CUDA_CHECK(cudaFuncGetAttributes(&attr, gbuffer_kernel<true>));
        loaded |= 1ull << (ctx->device & 63);
    }
    p.world = pt.world; p.rank = pt.rank;
    p.interleave = pt.ray_block_rows == 8;
    for (int r = 0; r < pt.world; ++r) {
        const bool own = r == pt.rank;
        p.albedo_of[r] = (uint32_t *)(own ? albedo->ptr : albedo->peer[r]);
        p.normals_of[r] = (uint2 *)(own ? normals->ptr : normals->peer[r]);
        p.motion_of[r] = (uint2 *)(own ? motion->ptr : motion->peer[r]);
        p.depth_of[r] = (float *)(own ? depth->ptr : depth->peer[r]);
    }
    // WAR on the peers' images: a peer may still be reading what the last partitioned G-buffer pass stored into these images. If that
    // pass wrote other images (alternating G-buffer sets), its trailing sync already ordered every rank's earlier work before this
    // one; otherwise (or with no such pass since the partition was installed) every rank first reaches this point.
    bool reused = !ctx->gbuffer_peer_written[0];
    for (Image *a : imgs)
        for (Image *b : ctx->gbuffer_peer_written) reused |= a == b;
    if (reused)
        if (int rc = peer_sync_all(ctx)) return rc;
    for (int i = 0; i < 4; ++i) ctx->gbuffer_peer_written[i] = imgs[i];
    int rows;
    if (p.interleave) {
        p.y_begin = 0; p.y_end = (int)height;
        const int n_blocks = ((int)height + 7) / 8;
        rows = (n_blocks - pt.rank + pt.world - 1) / pt.world * 8;        // blocks b = rank, rank + world, ...
    } else {
        rows = p.y_end - p.y_begin;
    }
    if (rows > 0) {
        dim3 block(128), grid((width + 15) / 16, (rows + 7) / 8);
        gbuffer_kernel<true><<<grid, block, 0, ctx->stream>>>(p, ctx->pfd);
        VHR_CUDA_CHECK(cudaGetLastError());
        ctx->launches++;
    }
    return peer_sync_all(ctx);      // later passes read rows the other ranks stored; the ray pass may not follow (rasterised shadows)
}

int launch_trace_explicit(vhr_context *ctx, const float *rays, uint32_t n, int any_hit, float *out_t, uint32_t *out_ids, float *out_uv) {
    if (n == 0) return VHR_OK;
    float *d_rays = nullptr, *d_t = nullptr, *d_uv = nullptr;
    uint32_t *d_ids = nullptr;
    VHR_CUDA_CHECK(cudaMalloc(&d_rays, (size_t)n * 8 * sizeof(float)));
    VHR_CUDA_CHECK(cudaMalloc(&d_t, (size_t)n * sizeof(float)));
    VHR_CUDA_CHECK(cudaMalloc(&d_ids, (size_t)n * 2 * sizeof(uint32_t)));
    VHR_CUDA_CHECK(cudaMalloc(&d_uv, (size_t)n * 2 * sizeof(float)));
    VHR_CUDA_CHECK(cudaMemcpyAsync(d_rays, rays, (size_t)n * 8 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    trace_explicit_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(d_rays, n, any_hit, scene_refs(ctx), d_t, d_ids, d_uv);
    VHR_CUDA_CHECK(cudaGetLastError());
    ctx->launches++;
    VHR_CUDA_CHECK(cudaMemcpyAsync(out_t, d_t, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (out_ids) VHR_CUDA_CHECK(cudaMemcpyAsync(out_ids, d_ids, (size_t)n * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (out_uv) VHR_CUDA_CHECK(cudaMemcpyAsync(out_uv, d_uv, (size_t)n * 2 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    VHR_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_rays); cudaFree(d_t); cudaFree(d_ids); cudaFree(d_uv);
    return VHR_OK;
}

}  // namespace vhr
