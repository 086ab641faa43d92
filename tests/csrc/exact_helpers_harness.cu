// Device test harness for the exactly-rounded helpers of vhr_common.cuh (div_exact*, sqrt_exact, bilinear_setup, wrap_repeat,
// wrap_texel) and for CUDA's sincosf. The header is included as the library compiles it; nothing is restated here except the
// references: IEEE operations (__fdiv_rn, __fsqrt_rn), the general filter-coordinate branch, and the Vulkan wrapping formulas in int64.
//
// Sweeps run on the device and report through a Report: a mismatch counter, a counter of checked inputs, and the first 64 offending
// inputs (four words each). The eval entry points write results for comparison with numpy on the host.
#include "../../vulkanhybridrenderer_b200/csrc/vhr_common.cuh"

#include <float.h>

using namespace vhr;

struct Report {
    unsigned long long mismatches, checked;
    uint32_t rec[64][4];
};

__device__ void report(Report *r, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
    const unsigned long long k = atomicAdd(&r->mismatches, 1ull);
    if (k < 64) {
        r->rec[k][0] = w0; r->rec[k][1] = w1; r->rec[k][2] = w2; r->rec[k][3] = w3;
    }
}

__device__ __forceinline__ bool same_bits(float x, float y) {       // bitwise, with NaN compared as a class
    return __float_as_uint(x) == __float_as_uint(y) || (x != x && y != y);
}

// ---------------------------------------------------------------------------------------------------------------------------------
// sqrt_exact against __fsqrt_rn on every bit pattern
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void sqrt_sweep_kernel(Report *r) {
    unsigned long long checked = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < (1ull << 32); i += (uint64_t)gridDim.x * blockDim.x) {
        const float x = __uint_as_float((uint32_t)i);
        const float got = sqrt_exact(x), want = __fsqrt_rn(x);
        if (!same_bits(got, want)) report(r, (uint32_t)i, __float_as_uint(got), __float_as_uint(want), 0);
        ++checked;
    }
    atomicAdd(&r->checked, checked);
}

__global__ void sqrt_eval_kernel(const float *x, float *ieee, float *exact, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        ieee[i] = __fsqrt_rn(x[i]);
        exact[i] = sqrt_exact(x[i]);
    }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// div_exact / div_exact_flag / div_exact_flag_bounded
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void div_eval_kernel(const float *a, const float *w, int n, float *q, float *qf, uint8_t *rf, float *qb, uint8_t *rb) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ExactDivisor d = exact_divisor(w[i]);
    q[i] = div_exact(a[i], d);
    bool rare = false;
    qf[i] = div_exact_flag(a[i], d, rare);
    rf[i] = rare;
    rare = false;
    qb[i] = div_exact_flag_bounded(a[i], d, rare);
    rb[i] = rare;
}

__device__ __forceinline__ bool fin_nz(float x) { return x != 0.0f && fabsf(x) <= FLT_MAX; }
__device__ __forceinline__ bool in_fast_range(float x) { return fabsf(x) >= 0x1p-40f && fabsf(x) < 0x1p40f; }

// The contracts of the flags (vhr_common.cuh): div_exact_flag raises `rare` exactly when both operands are finite and nonzero and one
// of them lies outside [2^-40, 2^40); div_exact_flag_bounded (dividend +0 or in that range) exactly when the divisor is finite, nonzero
// and outside it. Without `rare` the quotient is the IEEE one.
__device__ __forceinline__ bool rare_expected(float a, float w) {
    return fin_nz(w) && fin_nz(a) && (!in_fast_range(w) || !in_fast_range(a));
}
__device__ __forceinline__ bool rare_expected_bounded(float w) { return fin_nz(w) && !in_fast_range(w); }

// Every divisor significand (blockIdx.y picks the biased exponent from w_exps[]) over `n_sig` dividend significands at each biased
// exponent in a_exps[]; the dividend's low 11 significand bits and both signs come from a hash. Record: a, w, got, function (0, 1, 2;
// +16 when the flag was wrong).
__global__ void div_sweep_kernel(const int *w_exps, const int *a_exps, int n_a_exps, int n_sig, Report *r) {
    const uint32_t sig = blockIdx.x * blockDim.x + threadIdx.x;
    if (sig >= (1u << 23)) return;
    const uint32_t wsign = ((sig * 0x9E3779B1u) >> 31) << 31;
    const float w = __uint_as_float(wsign | ((uint32_t)w_exps[blockIdx.y] << 23) | sig);
    const ExactDivisor d = exact_divisor(w);
    unsigned long long checked = 0;
    for (int e = 0; e < n_a_exps; ++e) {
        for (int j = 0; j < n_sig; ++j) {
            const uint32_t h = seed_thread((uint32_t)j * 0x85EBCA6Bu ^ sig);
            uint32_t as = ((uint32_t)j * (1u << 23) / (uint32_t)n_sig) | (h & 0x7FFu);
            if (j == n_sig - 1) as = 0x7FFFFFu;
            const float a = __uint_as_float((h & 0x80000000u) | ((uint32_t)a_exps[e] << 23) | (as & 0x7FFFFFu));
            const float want = __fdiv_rn(a, w);
            const float q = div_exact(a, d);
            if (!same_bits(q, want)) report(r, __float_as_uint(a), __float_as_uint(w), __float_as_uint(q), 0);
            const bool exp_rare = rare_expected(a, w);
            bool rare = false;
            const float qf = div_exact_flag(a, d, rare);
            if (rare != exp_rare || (!rare && !same_bits(qf, want)))
                report(r, __float_as_uint(a), __float_as_uint(w), __float_as_uint(qf), 1 | (rare != exp_rare ? 16 : 0));
            if (__float_as_uint(a) == 0u || in_fast_range(a)) {      // div_exact_flag_bounded's precondition: +0 or in range
                rare = false;
                const float qb = div_exact_flag_bounded(a, d, rare);
                const bool exp_rare_b = rare_expected_bounded(w);
                if (rare != exp_rare_b || (!rare && !same_bits(qb, want)))
                    report(r, __float_as_uint(a), __float_as_uint(w), __float_as_uint(qb), 2 | (rare != exp_rare_b ? 16 : 0));
            }
            ++checked;
        }
    }
    atomicAdd(&r->checked, checked);
}

// ---------------------------------------------------------------------------------------------------------------------------------
// bilinear_setup: the fixed-point branch against the general branch (subtexel_rn + floor + wrap_repeat) on every float u with
// |fl(u n) - 0.5| < 2^14. Record: u, n, got (i0 | i1 << 16), want (i0 | i1 << 16); the weights are compared too (flag in bit 31).
// ---------------------------------------------------------------------------------------------------------------------------------
__global__ void bilinear_sweep_kernel(int n, Report *r) {
    const float nf = (float)n;
    unsigned long long checked = 0;
    for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < (1ull << 32); k += (uint64_t)gridDim.x * blockDim.x) {
        const float u = __uint_as_float((uint32_t)k);
        const float t = sub_rn(mul_rn(u, nf), 0.5f);
        if (!(fabsf(t) < 16384.0f)) continue;
        int i0, i1;
        float a;
        bilinear_setup(u, n, i0, i1, a);
        const float uu = subtexel_rn(t), fl = floorf(uu);
        const float ga = sub_rn(uu, fl);
        const int gi0 = wrap_repeat((int)fl, n), gi1 = wrap_repeat((int)fl + 1, n);
        if (i0 != gi0 || i1 != gi1 || __float_as_uint(a) != __float_as_uint(ga))
            report(r, (uint32_t)k, (uint32_t)n, (uint32_t)(i0 | (i1 << 16)) ^ (__float_as_uint(a) != __float_as_uint(ga) ? 0x80000000u : 0u),
                   (uint32_t)(gi0 | (gi1 << 16)));
        ++checked;
    }
    atomicAdd(&r->checked, checked);
}

__global__ void bilinear_eval_kernel(const float *u, int n, int count, int *i0, int *i1, float *a) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < count) bilinear_setup(u[k], n, i0[k], i1[k], a[k]);
}

// ---------------------------------------------------------------------------------------------------------------------------------
// wrap_repeat and wrap_texel on every int against the Vulkan spec's wrapping formulas evaluated in int64. Record: i, n, mode
// (4 = wrap_repeat), got.
// ---------------------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ long long spec_mod(long long i, long long n) { return ((i % n) + n) % n; }

__global__ void wrap_sweep_kernel(int n, Report *r) {
    const long long N = n;
    unsigned long long checked = 0;
    for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < (1ull << 32); k += (uint64_t)gridDim.x * blockDim.x) {
        const int i = (int)(uint32_t)k;
        const long long I = i;
        const long long rep = spec_mod(I, N);
        const long long mt = spec_mod(I, 2 * N) - N;
        const long long mir = (N - 1) - (mt >= 0 ? mt : -(1 + mt));
        const long long clamp = I < 0 ? 0 : (I > N - 1 ? N - 1 : I);
        const long long border = (I < 0 || I >= N) ? -1 : I;
        const long long want[5] = {rep, mir, clamp, border, rep};
        for (int m = 0; m < 5; ++m) {
            const int got = m < 4 ? wrap_texel(i, n, (uint32_t)m) : wrap_repeat(i, n);
            if ((long long)got != want[m]) report(r, (uint32_t)i, (uint32_t)n, (uint32_t)m, (uint32_t)got);
        }
        ++checked;
    }
    atomicAdd(&r->checked, checked);
}

// CUDA's sincosf, as the SSAO kernel calls it
__global__ void sincos_eval_kernel(const float *x, int n, float *s, float *c) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sincosf(x[i], &s[i], &c[i]);
}

static int last_error() { return (int)cudaGetLastError(); }
static dim3 blocks(long long n) { return dim3((unsigned)((n + 255) / 256)); }

extern "C" {
int eh_sqrt_sweep(Report *r) {
    sqrt_sweep_kernel<<<148 * 16, 256>>>(r);
    return last_error();
}
int eh_sqrt_eval(const float *x, float *ieee, float *exact, int n) {
    sqrt_eval_kernel<<<blocks(n), 256>>>(x, ieee, exact, n);
    return last_error();
}
int eh_div_eval(const float *a, const float *w, int n, float *q, float *qf, uint8_t *rf, float *qb, uint8_t *rb) {
    div_eval_kernel<<<blocks(n), 256>>>(a, w, n, q, qf, rf, qb, rb);
    return last_error();
}
int eh_div_sweep(const int *w_exps, int n_w_exps, const int *a_exps, int n_a_exps, int n_sig, Report *r) {
    div_sweep_kernel<<<dim3((1u << 23) / 256, n_w_exps), 256>>>(w_exps, a_exps, n_a_exps, n_sig, r);
    return last_error();
}
int eh_bilinear_sweep(int n, Report *r) {
    bilinear_sweep_kernel<<<148 * 16, 256>>>(n, r);
    return last_error();
}
int eh_bilinear_eval(const float *u, int n, int count, int *i0, int *i1, float *a) {
    bilinear_eval_kernel<<<blocks(count), 256>>>(u, n, count, i0, i1, a);
    return last_error();
}
int eh_wrap_sweep(int n, Report *r) {
    wrap_sweep_kernel<<<148 * 16, 256>>>(n, r);
    return last_error();
}
int eh_sincos_eval(const float *x, int n, float *s, float *c) {
    sincos_eval_kernel<<<blocks(n), 256>>>(x, n, s, c);
    return last_error();
}
int eh_report_size() { return (int)sizeof(Report); }
}
