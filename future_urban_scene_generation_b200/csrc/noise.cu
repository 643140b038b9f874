// noise.cu -- torch.randn on torch's CPU generator (MT19937 + normal_fill_AVX2), reproduced bit for bit on the device.
//
// The reference draws the VUNet Sampler noise with torch.randn on the CPU default generator (vunet/layers.py:166).  For a
// contiguous fp32 tensor whose numel is a multiple of 16 that is (oracle/noise_oracle.py restates it in numpy):
//   - one MT19937 word per element: --left; twist when it reaches 0 (left = 624, next = 0); temper state[next++];
//   - uniform u = (w & 0xFFFFFF) * 2^-24 (exact in fp32);
//   - per 16-element chunk, Box-Muller on elements j and j+8 (j < 8): u1 = 1 - u[j], u2 = u[j+8], radius =
//     sqrt(-2 log256_ps(u1)), (sin, cos) = sincos256_ps(2pi u2), out[j] = radius*cos, out[j+8] = radius*sin, each through
//     _mm256_fmadd_ps(n, 1, 0) (so -0 becomes +0).
// libtorch_cpu is built with GCC's default -ffp-contract=fast, which fuses some mul + add pairs of log256_ps / sincos256_ps
// into FMA (DESIGN.md §4.8 lists them).  The transform below spells every rounding out with __fmul_rn / __fadd_rn /
// __fmaf_rn / __fsqrt_rn, and the file is compiled with -fmad=false so that nothing else is contracted.
//
// Two kernels, because the MT19937 recurrence x[i] = x[i-227] ^ twist(x[i-624], x[i-623]) is sequential with a distance of
// 227 words:
//   k_mt_raw      one CTA walks the word stream 227 words per round (one __syncthreads per round) in a shared-memory ring
//                 and stores each UNTEMPERED word, as raw bits, at its element's final address;
//   k_box_muller  a grid-wide pass: one thread per (j, j+8) pair reads both raw words back, tempers them, and overwrites
//                 them with the two normals.
// So the generator needs no workspace, and an NHWC output (what the Sampler epilogues read) is written in place.
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>
#include "fusg.h"
#include "fusg_common.h"

namespace {

constexpr int MT_N = 624, MT_M = 397, MT_PAR = MT_N - MT_M;        // 227 words of the stream can be made at once
constexpr uint32_t MATRIX_A = 0x9908b0dfu;
constexpr int GEN_THREADS = 256, RING = 1024;                        // RING >= 624 + 227, a power of two
constexpr int BM_THREADS = 256;
constexpr uint32_t NAN_BITS = 0x7fc00000u;

struct RandnTable {
    fusg_randn_draw d[FUSG_RANDN_MAX_DRAWS];
    long long start[FUSG_RANDN_MAX_DRAWS + 1];    // first word of each draw; start[n] = all words
    int n;
};

__host__ __device__ __forceinline__ bool position_ok(uint32_t left, uint32_t next) {
    return left >= 1 && left <= (uint32_t)MT_N && next <= (uint32_t)MT_N && next + left - 1 <= (uint32_t)MT_N;
}

__host__ __device__ __forceinline__ uint32_t twist(uint32_t u, uint32_t v) {
    return (((u & 0x80000000u) | (v & 0x7fffffffu)) >> 1) ^ ((v & 1u) ? MATRIX_A : 0u);
}

__device__ __forceinline__ uint32_t *elem_addr(const RandnTable &t, int d, long long e) {
    const fusg_randn_draw &r = t.d[d];
    uint32_t *out = static_cast<uint32_t *>(r.out);
    if (!r.nhwc) return out + e;
    const long long hw = (long long)r.h * r.w, chw = hw * r.c;
    const long long b = e / chw, rem = e - b * chw, c = rem / hw, p = rem - c * hw;
    return out + b * chw + p * r.c + c;
}

__global__ void __launch_bounds__(GEN_THREADS, 1) k_mt_raw(const uint32_t *__restrict__ st, const RandnTable tab) {
    __shared__ uint32_t ring[RING];                   // x[i] at ring[i % RING]; x[0..623] is the state array
    const int t = threadIdx.x;
    const uint32_t left = st[MT_N], next = st[MT_N + 1];
    const long long total = tab.start[tab.n];
    int d = 0;                                        // draw of this thread's current word (its words only increase)
    auto emit = [&](long long w, uint32_t v) {
        while (w >= tab.start[d + 1]) ++d;
        *elem_addr(tab, d, w - tab.start[d]) = v;
    };
    if (!position_ok(left, next)) {                   // not a position torch's generator reaches: every output is NaN
        for (long long w = t; w < total; w += GEN_THREADS) emit(w, NAN_BITS);
        return;
    }
    for (int k = t; k < MT_N; k += GEN_THREADS) ring[k] = st[k];
    __syncthreads();
    // the left - 1 words already twisted: state[next .. next + left - 2]
    const long long l0 = min((long long)left - 1, total);
    for (long long w = t; w < l0; w += GEN_THREADS) emit(w, ring[next + w]);
    // then the stream x[624 + k], 227 words a round.  A round reads x[i - 624 .. i - 1] and writes x[i .. i + 226], which
    // lie less than RING apart, so one barrier per round orders everything.
    for (long long i0 = MT_N, w0 = l0; w0 < total; i0 += MT_PAR, w0 += MT_PAR) {
        uint32_t x = 0;
        if (t < MT_PAR) {
            const long long i = i0 + t;
            x = ring[(i - MT_N + MT_M) & (RING - 1)] ^ twist(ring[(i - MT_N) & (RING - 1)], ring[(i - MT_N + 1) & (RING - 1)]);
            ring[i & (RING - 1)] = x;
        }
        __syncthreads();
        if (t < MT_PAR && w0 + t < total) emit(w0 + t, x);
    }
}

// ---- log256_ps / sincos256_ps (ATen/native/cpu/avx_mathfun.h) as libtorch_cpu evaluates them ----------------------
// Constants are the header's double literals rounded to float, as its _PS256_CONST arrays hold them.
__device__ __forceinline__ float log256(float x) {                  // x in (0, 1]
    constexpr float P[9] = {(float)7.0376836292E-2, (float)-1.1514610310E-1, (float)1.1676998740E-1, (float)-1.2420140846E-1,
                            (float)1.4249322787E-1, (float)-1.6668057665E-1, (float)2.0000714765E-1, (float)-2.4999993993E-1,
                            (float)3.3333331174E-1};
    constexpr float Q1 = (float)-2.12194440e-4, Q2 = (float)0.693359375, SQRTHF = (float)0.707106781186547524;
    x = fmaxf(x, __uint_as_float(0x00800000u));
    const uint32_t bits = __float_as_uint(x);
    float e = __fadd_rn(__int2float_rn((int)(bits >> 23) - 0x7f), 1.0f);
    x = __uint_as_float((bits & ~0x7f800000u) | 0x3f000000u);
    const bool mask = x < SQRTHF;
    const float tmp = mask ? x : 0.0f;
    x = __fsub_rn(x, 1.0f);
    e = __fsub_rn(e, mask ? 1.0f : 0.0f);
    x = __fadd_rn(x, tmp);
    const float z = __fmul_rn(x, x);
    float y = P[0];
#pragma unroll
    for (int k = 1; k < 9; ++k) y = __fmaf_rn(y, x, P[k]);           // y*x + p_k: fused
    y = __fmul_rn(y, x);
    y = __fmaf_rn(y, z, __fmul_rn(e, Q1));                           // y*z + e*q1: the first product fused
    y = __fmaf_rn(-z, 0.5f, y);                                      // y - z*0.5: fused
    x = __fadd_rn(x, y);
    return __fmaf_rn(e, Q2, x);                                      // x + e*q2: fused
}

__device__ __forceinline__ void sincos256(float x, float *s, float *c) {   // x >= 0
    constexpr float DP1 = (float)-0.78515625, DP2 = (float)-2.4187564849853515625e-4, DP3 = (float)-3.77489497744594108e-8;
    constexpr float S0 = (float)-1.9515295891E-4, S1 = (float)8.3321608736E-3, S2 = (float)-1.6666654611E-1;
    constexpr float C0 = (float)2.443315711809948E-005, C1 = (float)-1.388731625493765E-003, C2 = (float)4.166664568298827E-002;
    constexpr float FOPI = (float)1.27323954473516;
    const uint32_t sign_in = __float_as_uint(x) & 0x80000000u;
    x = fabsf(x);
    int j = __float2int_rz(__fmul_rn(x, FOPI));
    j = (j + 1) & ~1;
    const float y = __int2float_rn(j);
    const uint32_t sign_sin = sign_in ^ ((uint32_t)(j & 4) << 29);
    const bool poly = (j & 2) == 0;
    const uint32_t sign_cos = (uint32_t)(~(j - 2) & 4) << 29;
    x = __fmaf_rn(y, DP1, x);                                        // x + y*DP_k: fused
    x = __fmaf_rn(y, DP2, x);
    x = __fmaf_rn(y, DP3, x);
    const float z = __fmul_rn(x, x);
    float yc = __fmaf_rn(__fmaf_rn(C0, z, C1), z, C2);
    yc = __fmul_rn(yc, z);
    yc = __fmaf_rn(yc, z, -__fmul_rn(z, 0.5f));                      // yc*z - z*0.5: the first product fused
    yc = __fadd_rn(yc, 1.0f);
    float ys = __fmaf_rn(__fmaf_rn(S0, z, S1), z, S2);
    ys = __fmul_rn(ys, z);
    ys = __fmaf_rn(ys, x, x);                                        // ys*x + x: fused
    // the header's masked select, additions of +0 included
    const float ysin2 = poly ? ys : 0.0f, ysin1 = poly ? 0.0f : yc;
    *s = __uint_as_float(__float_as_uint(__fadd_rn(ysin1, ysin2)) ^ sign_sin);
    *c = __uint_as_float(__float_as_uint(__fadd_rn(__fsub_rn(yc, ysin1), __fsub_rn(ys, ysin2))) ^ sign_cos);
}

__device__ __forceinline__ float uniform(uint32_t y) {
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return __fmul_rn(__uint2float_rn(y & 0xFFFFFFu), 5.9604644775390625e-8f);   // * 2^-24, exact
}

__global__ void __launch_bounds__(BM_THREADS) k_box_muller(const uint32_t *__restrict__ st, const RandnTable tab) {
    if (!position_ok(st[MT_N], st[MT_N + 1])) return;               // k_mt_raw wrote NaN
    constexpr float TWO_PI = (float)(2.0 * 3.14159265358979323846);  // 2.0f * c10::pi<double>, rounded by _mm256_set1_ps
    const long long pairs = tab.start[tab.n] / 2;
    for (long long q = (long long)blockIdx.x * BM_THREADS + threadIdx.x; q < pairs; q += (long long)gridDim.x * BM_THREADS) {
        const long long w1 = (q >> 3) * 16 + (q & 7);               // a 16-word chunk never straddles two draws
        int d = 0;
        while (w1 >= tab.start[d + 1]) ++d;
        uint32_t *a1 = elem_addr(tab, d, w1 - tab.start[d]), *a2 = elem_addr(tab, d, w1 + 8 - tab.start[d]);
        const float u1 = __fsub_rn(1.0f, uniform(*a1)), u2 = uniform(*a2);
        const float radius = __fsqrt_rn(__fmul_rn(log256(u1), -2.0f));
        float s, c;
        sincos256(__fmul_rn(TWO_PI, u2), &s, &c);
        *reinterpret_cast<float *>(a1) = __fadd_rn(__fmul_rn(radius, c), 0.0f);   // _mm256_fmadd_ps(n, 1, 0)
        *reinterpret_cast<float *>(a2) = __fadd_rn(__fmul_rn(radius, s), 0.0f);
    }
}

}  // namespace

extern "C" size_t fusg_sizeof_randn_draw(void) { return sizeof(fusg_randn_draw); }

extern "C" int fusg_randn_mt19937(const uint32_t *state, const fusg_randn_draw *draws, int ndraw, void *stream) {
    if (!state || !draws || ndraw <= 0 || ndraw > FUSG_RANDN_MAX_DRAWS) return FUSG_ERR_ARG;
    RandnTable tab = {};
    tab.n = ndraw;
    for (int i = 0; i < ndraw; ++i) {
        const fusg_randn_draw &r = draws[i];
        if (!r.out || r.b <= 0 || r.c <= 0 || r.h <= 0 || r.w <= 0 || (r.nhwc != 0 && r.nhwc != 1)) return FUSG_ERR_ARG;
        if (reinterpret_cast<uintptr_t>(r.out) & 3) return FUSG_ERR_ARG;
        const long long n = (long long)r.b * r.c * r.h * r.w;
        if (n < 16 || n % 16 != 0) return FUSG_ERR_UNSUPPORTED;      // torch draws such a tensor another way
        tab.d[i] = r;
        tab.start[i + 1] = tab.start[i] + n;
    }
    if (tab.start[ndraw] > (1ll << 40)) return FUSG_ERR_UNSUPPORTED;
    const int sms = fusg_num_sms();
    const long long pairs = tab.start[ndraw] / 2;
    long long grid = (pairs + BM_THREADS - 1) / BM_THREADS;
    if (grid > 8ll * sms) grid = 8ll * sms;
    cudaStream_t st = (cudaStream_t)stream;
    k_mt_raw<<<1, GEN_THREADS, 0, st>>>(state, tab);
    k_box_muller<<<(unsigned)grid, BM_THREADS, 0, st>>>(state, tab);
    fusg_count_launch(2);
    return fusg_check_launch();
}

extern "C" int fusg_mt19937_advance(const uint32_t *state, int left, long long next, long long n, uint32_t *state_out, int *left_out,
                                    long long *next_out) {
    if (!state || !state_out || !left_out || !next_out || n < 0 || next < 0 || next > MT_N) return FUSG_ERR_ARG;
    if (!position_ok((uint32_t)left, (uint32_t)next)) return FUSG_ERR_ARG;
    uint32_t s[MT_N];
    std::memcpy(s, state, sizeof(s));
    const long long k = n < left - 1 ? n : left - 1;
    left -= (int)k;
    next += k;
    n -= k;
    while (n > 0) {                                   // MT19937RNGEngine::next_state
        uint32_t *p = s;
        for (int j = MT_N - MT_M + 1; --j; p++) *p = p[MT_M] ^ twist(p[0], p[1]);
        for (int j = MT_M; --j; p++) *p = p[MT_M - MT_N] ^ twist(p[0], p[1]);
        *p = p[MT_M - MT_N] ^ twist(p[0], s[0]);
        const long long t = n < MT_N ? n : MT_N;
        n -= t;
        left = MT_N - (int)t + 1;
        next = t;
    }
    std::memcpy(state_out, s, sizeof(s));
    *left_out = left;
    *next_out = next;
    return FUSG_OK;
}
