// conv.cu -- VUNet convolution engine for sm_100a (include/fusg.h: fusg_conv2d and helpers).
//
// Reference semantics: MyConv2d / NiN / Residual / DownSample / UpSample('subpixel') / Sampler /
// DepthToSpace / SpaceToDepth of vunet/layers.py:21-221, as they are composed by
// vunet/models.py:17-484.  One launch = one convolution with everything the reference wraps
// around it fused in: channel concat of two inputs (K-loop over two TMA descriptors), bias,
// residual add, Sampler noise, ELU for the next pre-activated layer, sub-pixel addressing.
//
// Two kernels, same epilogue:
//   k_conv_tc      implicit GEMM on the 5th-gen tensor cores: M = 128 output pixels
//                  (Wt x Ht x Bt box), N = up to 128 output channels, K = taps x channels.
//                  A tiles are fetched by 4-D tiled TMA straight from the NHWC activation with the
//                  tap offset folded into the box coordinate -- out-of-bounds zero fill IS the
//                  convolution padding (and elementStrides = 2 IS the stride) -- B tiles by 2-D TMA
//                  from the folded weight matrix; both land 128B/64B-swizzled, K-major, and are
//                  consumed by tcgen05.mma (kind::f16, bf16 x bf16 -> fp32) with the accumulator in
//                  TMEM (double buffered).  Warp roles: 0 = TMA producer, 1 = MMA issuer (+ TMEM
//                  alloc), 2..5 = epilogue (tcgen05.ld -> registers -> global).  Persistent over tiles.
//   k_conv_direct  CUDA-core direct convolution with fp32 accumulation; used for the fp32
//                  verification build and as the in-library cross-check of k_conv_tc.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <type_traits>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include "../../include/fusg.h"
#include "fusg_common.h"

namespace fusg {

// ------------------------------------------------------------------------------------------------
// shared epilogue
// ------------------------------------------------------------------------------------------------
// ELU(x) = x > 0 ? x : exp(x) - 1.  __expf (ex2.approx) has ~2 ulp error at 1.0, i.e. an absolute error of
// ~2e-7 on the negative branch: far below bf16 resolution and below the 1e-4 fp32 verification bar.
__device__ __forceinline__ float elu1(float x) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 1.4426950408889634f));
    return x > 0.f ? x : e - 1.f;
}

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }

struct OutAddr { size_t pix; int ch; int Ct, Ht, Wt, py, px; };

// fusg_conv_out.elu: 0 raw, 1 ELU, 2 tanh
__device__ __forceinline__ float out_act(int kind, float v) { return kind == 1 ? elu1(v) : (kind == 2 ? tanhf(v) : v); }

// logical destination of output channel group starting at n (16-aligned) for pixel (y,x)
__device__ __forceinline__ OutAddr out_address(const fusg_conv_out &o, int cout, int Ho, int Wo, int b, int y, int x, int n) {
    OutAddr a;
    switch (o.mode) {
        default:
        case FUSG_OUT_PLAIN: a.Ct = cout; a.Ht = Ho; a.Wt = Wo; a.py = y; a.px = x; a.ch = n; break;
        case FUSG_OUT_D2S: {
            const int cq = cout >> 2, blk = n / cq;
            a.Ct = cq; a.Ht = 2 * Ho; a.Wt = 2 * Wo; a.py = 2 * y + (blk >> 1); a.px = 2 * x + (blk & 1); a.ch = n - blk * cq;
            break;
        }
        case FUSG_OUT_S2D:
            a.Ct = 4 * cout; a.Ht = Ho >> 1; a.Wt = Wo >> 1; a.py = y >> 1; a.px = x >> 1; a.ch = (((y & 1) << 1) + (x & 1)) * cout + n;
            break;
        case FUSG_OUT_D2S_BLOCK:
            a.Ct = cout; a.Ht = 2 * Ho; a.Wt = 2 * Wo; a.py = 2 * y + (o.blk >> 1); a.px = 2 * x + (o.blk & 1); a.ch = n;
            break;
    }
    a.pix = ((size_t)b * a.Ht + a.py) * a.Wt + a.px;
    return a;
}

// v[16]: fp32 accumulators of channels n..n+15 of output pixel (b,y,x); applies bias, residual,
// noise and writes every output slot.
template <typename T>
__device__ __forceinline__ void epilogue16(const fusg_conv_desc &d, const float *bias, int Ho, int Wo, int b, int y, int x, int n, float *v) {
    const int nvalid = min(16, d.cout - n);
    if (nvalid <= 0) return;
    const size_t opix = ((size_t)b * Ho + y) * Wo + x;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += bias[n + i];
    if (d.residual) {
        const T *r = reinterpret_cast<const T *>(d.residual) + opix * d.cout + n;
        if (nvalid == 16) {
            if constexpr (std::is_same<T, __nv_bfloat16>::value) {
                const uint4 q0 = __ldg(reinterpret_cast<const uint4 *>(r)), q1 = __ldg(reinterpret_cast<const uint4 *>(r) + 1);
                const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162 *>(&w[i]);
                    v[2 * i] += __bfloat162float(h.x);
                    v[2 * i + 1] += __bfloat162float(h.y);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] += to_f<T>(r[i]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < nvalid) v[i] += to_f<T>(r[i]);
        }
    }
    float z[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) z[i] = 0.f;
    bool need_z = false;
#pragma unroll
    for (int s = 0; s < FUSG_CONV_MAX_OUTS; ++s) need_z = need_z || (d.outs[s].ptr != nullptr && d.outs[s].source == 1);
    if (need_z) {
        const float *e = d.noise + opix * d.cout + n;
#pragma unroll
        for (int i = 0; i < 16; ++i) z[i] = v[i] + (i < nvalid ? __ldg(e + i) : 0.f);
    }
#pragma unroll
    for (int s = 0; s < FUSG_CONV_MAX_OUTS; ++s) {
        const fusg_conv_out &o = d.outs[s];
        if (o.ptr == nullptr) continue;
        float val[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) val[i] = o.source == 1 ? z[i] : v[i];
        const OutAddr a = out_address(o, d.cout, Ho, Wo, b, y, x, n);
        if (o.layout == 1 && o.mode == FUSG_OUT_UNPAIR) {    // pixel-pair packed layer -> NCHW fp32
            float *p = reinterpret_cast<float *>(o.ptr);
            const int cq = d.cout >> 1;
#pragma unroll
            for (int i = 0; i < 16; ++i) {             // constant trip count keeps val[] in registers
                if (i < nvalid) {
                    const int nn = n + i, dx = nn >= cq ? 1 : 0, c = nn - dx * cq;   // nn < 2*cq
                    p[(((size_t)b * cq + c) * Ho + y) * (2 * Wo) + 2 * x + dx] = out_act(o.elu, val[i]);
                }
            }
        } else if (o.layout == 1) {                          // NCHW fp32, unrounded
            float *p = reinterpret_cast<float *>(o.ptr);
            const size_t plane = (size_t)a.Ht * a.Wt;
            const size_t base = ((size_t)b * a.Ct + a.ch) * plane + (size_t)a.py * a.Wt + a.px;
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < nvalid) p[base + (size_t)i * plane] = out_act(o.elu, val[i]);
        } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
            __nv_bfloat16 *p = reinterpret_cast<__nv_bfloat16 *>(o.ptr) + a.pix * a.Ct + a.ch;
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                // ELU is taken of the bf16-rounded raw value, so a consumer that re-derives it from
                // the stored raw tensor gets the same bits.
                float f0 = __bfloat162float(__float2bfloat16_rn(val[2 * i])), f1 = __bfloat162float(__float2bfloat16_rn(val[2 * i + 1]));
                if (o.elu) { f0 = out_act(o.elu, f0); f1 = out_act(o.elu, f1); }
                const __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);
                w[i] = *reinterpret_cast<const uint32_t *>(&h);
            }
            if (nvalid == 16) {
                reinterpret_cast<uint4 *>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
                reinterpret_cast<uint4 *>(p)[1] = make_uint4(w[4], w[5], w[6], w[7]);
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (i < nvalid) p[i] = __ushort_as_bfloat16((unsigned short)((i & 1) ? (w[i >> 1] >> 16) : (w[i >> 1] & 0xffffu)));
            }
        } else {
            T *p = reinterpret_cast<T *>(o.ptr) + a.pix * a.Ct + a.ch;       // fp32 / fp16 NHWC (activation of the rounded value)
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < nvalid) p[i] = from_f<T>(out_act(o.elu, to_f<T>(from_f<T>(val[i]))));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_conv_direct: thread = (output pixel, group of 16 output channels)
// ------------------------------------------------------------------------------------------------
constexpr int DC_CHUNK = 32;   // channels staged per step

template <typename T>
__global__ void __launch_bounds__(128) k_conv_direct(const __grid_constant__ fusg_conv_desc d, int Ho, int Wo) {
    __shared__ float s_w[16][DC_CHUNK + 1];
    const long long total = (long long)d.B * Ho * Wo;
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int n0 = blockIdx.y * 16;
    const bool active = pix < total;
    int b = 0, y = 0, x = 0;
    if (active) { b = (int)(pix / ((long long)Ho * Wo)); const int r = (int)(pix - (long long)b * Ho * Wo); y = r / Wo; x = r - y * Wo; }
    // pad_mode 1: the padding values live in the input tensor's own border (fusg.h)
    const int pad = d.pad_mode ? d.pad : d.ksize >> 1, bd = d.pad_mode ? d.border : 0, ctot = d.c0 + d.c1, taps = d.ksize * d.ksize;
    const int Hp = d.H + 2 * bd, Wp = d.W + 2 * bd;
    const int cph0 = d.cphys0 ? d.cphys0 : d.c0, cph1 = d.cphys1 ? d.cphys1 : d.c1;   // channels beyond these read as zero
    const T *wbase = reinterpret_cast<const T *>(d.weight);
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    for (int tap = 0; tap < taps; ++tap) {
        const int ky = tap / d.ksize, kx = tap - ky * d.ksize;
        const int iy = y * d.stride + ky - pad + bd, ix = x * d.stride + kx - pad + bd;      // physical coordinates
        const bool inb = active && iy >= 0 && iy < Hp && ix >= 0 && ix < Wp;
        for (int c0 = 0; c0 < ctot; c0 += DC_CHUNK) {
            const int cn = min(DC_CHUNK, ctot - c0);
            __syncthreads();
            for (int i = threadIdx.x; i < 16 * DC_CHUNK; i += blockDim.x) {
                const int n = i / DC_CHUNK, c = i - n * DC_CHUNK;
                float w = 0.f;
                if (c < cn && n0 + n < d.cout_pad) w = to_f<T>(wbase[((size_t)(n0 + n) * taps + tap) * ctot + c0 + c]);
                s_w[n][c] = w;
            }
            __syncthreads();
            if (inb) {
                for (int c = 0; c < cn; ++c) {
                    const int cc = c0 + c;
                    float a;
                    if (cc < d.c0) a = cc < cph0 ? to_f<T>(reinterpret_cast<const T *>(d.in0)[(((size_t)b * Hp + iy) * Wp + ix) * d.pitch0 + cc]) : 0.f;
                    else a = cc - d.c0 < cph1 ? to_f<T>(reinterpret_cast<const T *>(d.in1)[(((size_t)b * Hp + iy) * Wp + ix) * d.pitch1 + (cc - d.c0)]) : 0.f;
#pragma unroll
                    for (int n = 0; n < 16; ++n) acc[n] = fmaf(a, s_w[n][c], acc[n]);
                }
            }
        }
    }
    if (active) epilogue16<T>(d, d.bias, Ho, Wo, b, y, x, n0, acc);
}

// ------------------------------------------------------------------------------------------------
// PTX wrappers (tcgen05 / TMA / mbarrier)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_addr(bar)) : "memory");
}
// the barriers of a CTA live in one 1024-byte aligned block: [full | empty | tfull[2] | tempty[2] | w_bar | tmem_slot[6]];
// tmem_slot[4] holds the kernel's start time for the bounded waits (fusg_wait_failed)
constexpr unsigned TC_WAIT_COUNTER_OFF = 312;        // (2 * TC_MAX_STAGES + 5) * 8 + 16, checked below
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(s_addr(bar)), "r"(parity), "r"(0x989680u)
            : "memory");
        if (!done) fusg_wait_failed((s_addr(bar) & ~1023u) + TC_WAIT_COUNTER_OFF);
    }
}
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
            s_addr(dst)),
        "l"(tm), "r"(s_addr(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(s_addr(dst)),
        "l"(tm), "r"(s_addr(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// one lane of the (converged) warp; keeps the surrounding control flow warp-uniform so that TMA / MMA
// operands stay in uniform registers (no per-instruction waterfall loop)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_addr(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s_addr(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t *r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA-pair (cta_group::2) variants: the two CTAs of a cluster share one M = 256 MMA; each holds its own 128 A rows
// and HALF of the weight rows; TMA loads of both CTAs signal the leader's mbarrier; the leader's commit arrives on the
// barriers of both CTAs (multicast).  Checked in isolation by scripts/umma_2cta_probe.cu.
__device__ __forceinline__ void tmem_alloc2(uint32_t *dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_addr(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(void *dst, const CUtensorMap *tm, uint32_t bar_cluster_addr, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
            s_addr(dst)),
        "l"(tm), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void *dst, const CUtensorMap *tm, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(s_addr(dst)),
        "l"(tm), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2cta(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(s_addr(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
// wait on a barrier of this CTA that a PEER CTA arrives on (cluster-scope acquire)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(s_addr(bar)), "r"(parity), "r"(0x989680u)
            : "memory");
        if (!done) fusg_wait_failed((s_addr(bar) & ~1023u) + TC_WAIT_COUNTER_OFF);
    }
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

// thread-block cluster helpers (split-K layers)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t dsmem_addr(uint32_t local_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//  [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) swizzle mode
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout_type) {
    uint64_t desc = 0;
    desc |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    desc |= (uint64_t)1 << 16;                          // LBO (ignored for swizzled K-major; canonical value 1)
    desc |= (uint64_t)(sbo_bytes >> 4) << 32;
    desc |= (uint64_t)1 << 46;
    desc |= (uint64_t)layout_type << 61;
    return desc;
}


// ------------------------------------------------------------------------------------------------
// Lean epilogue of k_conv_tc for the common layer shape: no noise, outputs are at most one raw and
// one ELU NHWC bf16 tensor sharing the same addressing mode, cout a multiple of 16.
// ------------------------------------------------------------------------------------------------
struct FastEpi {
    __nv_bfloat16 *raw, *elu;
    const __nv_bfloat16 *res;
    int mode, blk, cq_shift;
    int f16;                  // activation dtype is fp16 (raw outputs only: no residual / ELU copy on this path)
    int stride_a, stride_b;   // elements between output pixels x -> x+2 and x -> x+1 (x even) of one image row under `mode`
};

__device__ __forceinline__ float bf16lo_to_f(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16hi_to_f(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// fp16 activations (ICN): saturate instead of overflowing to inf -- a pre-norm convolution output beyond +-65504 would
// otherwise turn the whole InstanceNorm plane into NaN (random-init weights stay below ~1e2; real checkpoints are unverified)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    uint32_t r;
    lo = fminf(fmaxf(lo, -65504.f), 65504.f);
    hi = fminf(fmaxf(hi, -65504.f), 65504.f);
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}

__device__ __forceinline__ uint4 elu_piece(uint4 v) {
    uint4 o;
    o.x = pack_bf16x2(elu1(bf16lo_to_f(v.x)), elu1(bf16hi_to_f(v.x)));
    o.y = pack_bf16x2(elu1(bf16lo_to_f(v.y)), elu1(bf16hi_to_f(v.y)));
    o.z = pack_bf16x2(elu1(bf16lo_to_f(v.z)), elu1(bf16hi_to_f(v.z)));
    o.w = pack_bf16x2(elu1(bf16lo_to_f(v.w)), elu1(bf16hi_to_f(v.w)));
    return o;
}

// element offset (in channels) of output channel n of plain-output pixel (b,y,x) under `mode`
__device__ __forceinline__ size_t fast_out_offset(const FastEpi &fe, int cout, int Ho, int Wo, int b, int y, int x, int n) {
    switch (fe.mode) {
        default:
        case FUSG_OUT_PLAIN: return (((size_t)b * Ho + y) * Wo + x) * cout + n;
        case FUSG_OUT_D2S: {
            const int blk = n >> fe.cq_shift, cq = 1 << fe.cq_shift;
            return (((size_t)b * 2 * Ho + 2 * y + (blk >> 1)) * (2 * Wo) + 2 * x + (blk & 1)) * cq + (n & (cq - 1));
        }
        case FUSG_OUT_S2D:
            return ((((size_t)b * (Ho >> 1) + (y >> 1)) * (Wo >> 1) + (x >> 1)) * 4 + (((y & 1) << 1) + (x & 1))) * cout + n;
        case FUSG_OUT_D2S_BLOCK:
            return (((size_t)b * 2 * Ho + 2 * y + (fe.blk >> 1)) * (2 * Wo) + 2 * x + (fe.blk & 1)) * cout + n;
    }
}

__device__ __forceinline__ void fast_chunk16(const FastEpi &fe, const float *s_bias, int cout, int Ho, int Wo, size_t opix, int b, int y, int x,
                                             int n, const uint32_t *acc) {
    float v[16];
    const float4 *b4 = reinterpret_cast<const float4 *>(s_bias + n);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 bb = b4[i];
        v[4 * i] = __uint_as_float(acc[4 * i]) + bb.x;
        v[4 * i + 1] = __uint_as_float(acc[4 * i + 1]) + bb.y;
        v[4 * i + 2] = __uint_as_float(acc[4 * i + 2]) + bb.z;
        v[4 * i + 3] = __uint_as_float(acc[4 * i + 3]) + bb.w;
    }
    if (fe.res) {
        const uint4 *r = reinterpret_cast<const uint4 *>(fe.res + opix * cout + n);
        const uint4 q0 = __ldg(r), q1 = __ldg(r + 1);
        const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) { v[2 * i] += bf16lo_to_f(w[i]); v[2 * i + 1] += bf16hi_to_f(w[i]); }
    }
    uint32_t pk[8];
    if (fe.f16) {
#pragma unroll
        for (int i = 0; i < 8; ++i) pk[i] = pack_f16x2(v[2 * i], v[2 * i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) pk[i] = pack_bf16x2(v[2 * i], v[2 * i + 1]);
    }
    const size_t off = fast_out_offset(fe, cout, Ho, Wo, b, y, x, n);
    if (fe.raw) {
        uint4 *o = reinterpret_cast<uint4 *>(fe.raw + off);
        o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    }
    if (fe.elu) {
        uint32_t ek[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) ek[i] = pack_bf16x2(elu1(bf16lo_to_f(pk[i])), elu1(bf16hi_to_f(pk[i])));   // ELU of the rounded value
        uint4 *o = reinterpret_cast<uint4 *>(fe.elu + off);
        o[0] = make_uint4(ek[0], ek[1], ek[2], ek[3]);
        o[1] = make_uint4(ek[4], ek[5], ek[6], ek[7]);
    }
}

// fast_epi == 3: the network's last layer (shape_decoder_6.conv, 32 -> 3, run on pixel pairs: n = dx * cq + c, cq = cout / 2 <= 8)
// straight to the NCHW fp32 API tensor.  A thread holds both pixels of its pair for every channel: one 8-byte store per
// channel, and the 32 lanes of a warp (consecutive pairs of one image row) cover 256 contiguous bytes.  The generic
// epilogue spent 160 us on this layer's 50 MB (scalar stores, per-element index arithmetic, a code path that does not fit
// the instruction cache).
__device__ __forceinline__ void unpair_chunk(float *out, const float *s_bias, int cq, int Ho, int Wo, int b, int y, int x, const uint32_t *acc) {
    float *p = out + (((size_t)b * cq) * Ho + y) * (size_t)(2 * Wo) + 2 * x;
    const size_t plane = (size_t)Ho * (2 * Wo);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        if (c < cq) {
            float2 v;
            v.x = __uint_as_float(acc[c]) + s_bias[c];
            v.y = __uint_as_float(acc[cq + c]) + s_bias[cq + c];
            *reinterpret_cast<float2 *>(p + c * plane) = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_conv_tc
// ------------------------------------------------------------------------------------------------
constexpr int TC_EPI_WARPS = 8;                         // warps 2..9; warp 0 TMA, warp 1 MMA
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
constexpr int TC_STAGING_BYTES = 32768;                  // shared memory of the staged epilogue
constexpr int TC_STAGE_BYTES = TC_STAGING_BYTES / TC_EPI_WARPS;     // per-warp staging block
constexpr int TC_BLOCK_M = 128;
constexpr int TC_HALO_ROWS_MAX = TC_BLOCK_M + 6;                   // pixels of one halo A buffer: 128 + ksize - 1, ksize <= 7
constexpr int TC_HALO_BYTES = ((TC_HALO_ROWS_MAX * 128 + 1023) / 1024) * 1024;   // 128-byte rows (kc = 64), 1024-aligned
constexpr int TC_MAX_STAGES = 16;
static_assert(TC_WAIT_COUNTER_OFF == (2 * TC_MAX_STAGES + 5) * 8 + 16, "the wait guard's start-time slot must be tmem_slot[4]");

struct alignas(64) ConvTcParams {
    CUtensorMap tmA0, tmA1, tmW;
    fusg_conv_desc d;
    int Ho, Wo;
    int Wt, Ht, Bt;                 // tile box (output pixels): Wt*Ht*Bt = 128*msub
    int wt_shift, ht_shift;         // log2(Wt), log2(Ht): Ho, Wo and the tile box are powers of two on this path
    int txs, tys;                   // log2(tiles_x), log2(tiles_y)
    int msub;                       // 128-row MMA sub-tiles per CTA tile (1 or 2): two sub-tiles share every B k-block
    int tiles_x, tiles_y, tiles_b;  // M-tile grid
    int n_tiles, block_n;           // N tiling
    int kc;                         // channels per k-block (64: 128B swizzle, 32: 64B swizzle)
    int chunks0, chunks1;           // k-blocks per tap from in0 / in1
    int num_kblocks;                // taps * (chunks0 + chunks1)
    int stages;
    int a_bytes, b_bytes;           // per k-block
    int group;                      // k-blocks per pipeline stage (one barrier round trip)
    int w_resident;                 // 1: the whole weight matrix of the (single) N tile stays in shared memory
    int halo;                       // 1: sliding-window A tiles -- one TMA load of an image-row segment + 2 halo pixels serves the
                                    //    three horizontal taps (3x3, stride 1, Wt = 128, one image row per 128-row sub-tile)
    int hks;                        // halo mode: kernel size (3; 5 or 7 for the bordered ICN layers) -- hks horizontal taps per loaded row segment
    uint32_t halo_skip;             // halo mode: bit (ky * chunks + chunk) set = all three taps of that stage have zero weights -> skipped
    int pair;                       // halo mode on CTA pairs (cta_group::2): M = 256 per MMA, each CTA holds half of the weight rows
    int epi_smem;                   // bytes past the bias: the staged epilogue's staging blocks (reserved whenever the plan wanted
                                    // it, even if the lean epilogue was then refused) or the split-K receive buffer
    unsigned long long w_prefetch_bytes;   // > 0: bytes of the weight matrix the grid pulls into L2 before the dependency wait
    int ksplit;                     // > 1: thread-block cluster of `ksplit` CTAs per tile, each reducing 1/ksplit of K (few-tile layers)
    int kb_local;                   // k-blocks per CTA = num_kblocks / ksplit
    int tmem_cols;
    int fast_epi;                   // 1: lean epilogue, 2: lean + warp-staged epilogue (every global access covers whole 128-byte lines)
    FastEpi fe;
};

// Shared-memory layout of k_conv_tc, in bytes from the kernel's 1024-aligned base: barriers (first KB) | A pipeline |
// B region | bias | staging / split-K receive buffer.  `total` is the launch's dynamic shared-memory size, alignment
// slack included.
struct TcSmem { size_t b, bias, stage, total; };
__host__ __device__ __forceinline__ TcSmem tc_smem(const ConvTcParams &p) {
    const size_t pipe_a = p.halo ? (size_t)p.stages * 2 * TC_HALO_BYTES : (size_t)p.stages * p.group * p.a_bytes;
    // B k-blocks: [stages][hks] in halo mode, [stages][group] streamed, or [num_kblocks] resident
    const size_t pipe_b = p.w_resident ? (size_t)p.num_kblocks * p.b_bytes
                                       : (p.halo ? (size_t)p.stages * p.hks * p.b_bytes : (size_t)p.stages * p.group * p.b_bytes);
    TcSmem s;
    s.b = 1024 + pipe_a;
    s.bias = s.b + ((pipe_b + 15) & ~(size_t)15);              // cout_pad floats, 16-byte aligned (float4 reads)
    s.stage = s.bias + (size_t)p.d.cout_pad * 4;
    s.total = 1024 /*alignment slack*/ + s.b + pipe_b + 16 /*bias alignment*/ + (size_t)p.d.cout_pad * 4 + (size_t)p.epi_smem;
    return s;
}

// MMA-issuer role of k_conv_tc.  Everything the loop needs is hoisted into registers and the
// (sub-tile, k-step) MMAs of a k-block are fully unrolled: the single issuing thread must stay well
// under the tensor-pipe time of a k-block (KSTEPS*MSUB*64 cycles at N=128) or it becomes the bottleneck.
template <int KSTEPS, int MSUB>
__device__ __forceinline__ void mma_role(const ConvTcParams &p, uint8_t *sA, uint8_t *sB, uint64_t *full_bar, uint64_t *empty_bar,
                                         uint64_t *tfull_bar, uint64_t *tempty_bar, uint64_t *w_bar, uint32_t tmem_base, int total_tiles) {
    const uint32_t block_n = (uint32_t)p.block_n;
    // instruction descriptor: fp32 accumulate | A/B format (1 = bf16, 0 = fp16) | N >> 3 | M >> 4
    const uint32_t idesc = (1u << 4) | (p.fe.f16 ? 0u : ((1u << 7) | (1u << 10))) | ((block_n >> 3) << 17) | ((uint32_t)(TC_BLOCK_M >> 4) << 24);
    const uint32_t kc = KSTEPS * 16;
    // descriptor high bits: LBO=1 | SBO = 8 rows of one swizzle span | version 1 | swizzle mode
    const uint64_t desc_hi = ((uint64_t)1 << 16) | ((uint64_t)((kc * 2u * 8u) >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)(KSTEPS == 4 ? 2u : 4u) << 61);
    const uint32_t sub16 = (TC_BLOCK_M * kc * 2u) >> 4;                 // next 128-row sub-tile, in 16-byte units
    const int group = p.group, stages = p.stages, groups = p.kb_local / p.group;
    const uint32_t a_kb16 = (uint32_t)p.a_bytes >> 4, b_kb16 = (uint32_t)p.b_bytes >> 4;
    const uint32_t a_stage16 = a_kb16 * group, b_stage16 = b_kb16 * group;
    const bool resident = p.w_resident != 0;
    const uint32_t sA16 = (s_addr(sA) & 0x3FFFF) >> 4, sB16 = (s_addr(sB) & 0x3FFFF) >> 4;
    const uint32_t acc_cols = (uint32_t)MSUB * block_n;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t acc = 0, acc_phase = 0;
    if (resident) mbar_wait(w_bar, 0);
    for (int tile = blockIdx.x / p.ksplit; tile < total_tiles; tile += gridDim.x / p.ksplit) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * acc_cols;
        for (int grp = 0; grp < groups; ++grp) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            if (elect_one()) {
                uint32_t a16 = sA16 + (uint32_t)stage * a_stage16;
                uint32_t b16 = sB16 + (resident ? (uint32_t)grp * b_stage16 : (uint32_t)stage * b_stage16);
                for (int g = 0; g < group; ++g) {
                    const uint64_t a_desc = desc_hi | (uint64_t)a16, b_desc = desc_hi | (uint64_t)b16;
                    const uint32_t first = (grp | g) != 0 ? 1u : 0u;
#pragma unroll
                    for (int sub = 0; sub < MSUB; ++sub) {
#pragma unroll
                        for (int ks = 0; ks < KSTEPS; ++ks) {
                            // +2 (x16 bytes) per 16-element K step inside the swizzle span
                            umma_bf16(d_tmem + (uint32_t)sub * block_n, a_desc + (uint64_t)(sub * sub16 + ks * 2), b_desc + (uint64_t)(ks * 2), idesc,
                                      ks == 0 ? first : 1u);
                        }
                    }
                    a16 += a_kb16;
                    b16 += b_kb16;
                }
                umma_commit(&empty_bar[stage]);                // frees the smem stage when these MMAs retire
                if (grp == groups - 1) umma_commit(&tfull_bar[acc]);   // accumulator complete
            }
            __syncwarp();
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
    }
}

// MMA issuer of the sliding-window (halo) mode: a pipeline stage holds, for one (tap row ky, 64-channel chunk), the
// two image-row segments of the CTA tile with one extra pixel on each side, and the three weight k-blocks kx = 0..2.
// The A descriptor of tap kx simply starts kx rows (kx * 128 bytes) into the buffer: the 128-byte swizzle is a
// function of the absolute shared-memory address, so a start address that is 128- but not 1024-byte aligned
// addresses the same swizzled rows (checked on the device by scripts/umma_shift_probe.cu).
template <bool PAIR, int KS>
__device__ __forceinline__ void mma_role_halo(const ConvTcParams &p, uint8_t *sA, uint8_t *sB, uint64_t *full_bar, uint64_t *empty_bar,
                                              uint64_t *tfull_bar, uint64_t *tempty_bar, uint64_t *w_bar, uint32_t tmem_base, int total_tiles) {
    const uint32_t block_n = (uint32_t)p.block_n;
    constexpr bool pair = PAIR;
    if (pair && cluster_ctarank() != 0) return;                        // the leader CTA issues for the pair
    const uint32_t idesc = (1u << 4) | (p.fe.f16 ? 0u : ((1u << 7) | (1u << 10))) | ((block_n >> 3) << 17) | ((uint32_t)((pair ? 2 * TC_BLOCK_M : TC_BLOCK_M) >> 4) << 24);
    const uint64_t desc_hi = ((uint64_t)1 << 16) | ((uint64_t)(1024u >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2u << 61);
    const int stages = p.stages, cpt = p.chunks0 + p.chunks1, nst = KS * cpt;
    const uint32_t skip = p.halo_skip;
    int st_first = 0, st_last = nst - 1;                       // first / last stage that is actually executed
    while ((skip >> st_first) & 1u) ++st_first;
    while ((skip >> st_last) & 1u) --st_last;
    const uint32_t b_kb16 = (uint32_t)p.b_bytes >> 4;
    const uint32_t a_stage16 = (2u * TC_HALO_BYTES) >> 4, b_stage16 = (uint32_t)KS * b_kb16;
    const bool resident = p.w_resident != 0;
    const uint32_t sA16 = (s_addr(sA) & 0x3FFFF) >> 4, sB16 = (s_addr(sB) & 0x3FFFF) >> 4;
    const uint32_t acc_cols = 2u * block_n;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t acc = 0, acc_phase = 0;
    if (resident) mbar_wait(w_bar, 0);
    const int tstep = pair ? (int)gridDim.x >> 1 : (int)gridDim.x, tcount = pair ? total_tiles >> 1 : total_tiles;
    for (int tile = pair ? (int)blockIdx.x >> 1 : (int)blockIdx.x; tile < tcount; tile += tstep) {
        if constexpr (PAIR) mbar_wait_cluster(&tempty_bar[acc], acc_phase ^ 1);
        else mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * acc_cols;
        for (int st = 0; st < nst; ++st) {
            if ((skip >> st) & 1u) continue;
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t a16 = sA16 + (uint32_t)stage * a_stage16;
                // weight k-block index of (ky, kx, chunk) is (ky*3 + kx)*cpt + chunk; st = ky*cpt + chunk
                const int ky = st / cpt, c = st - ky * cpt;
                const uint32_t b16 = resident ? sB16 + (uint32_t)(ky * KS * cpt + c) * b_kb16 : sB16 + (uint32_t)stage * b_stage16;
                const uint32_t b_step = resident ? (uint32_t)cpt * b_kb16 : b_kb16;
                auto issue_tap = [&](int kx) {
#pragma unroll
                    for (int sub = 0; sub < 2; ++sub) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint64_t a_desc = desc_hi | (uint64_t)(a16 + (uint32_t)sub * (TC_HALO_BYTES >> 4) + (uint32_t)kx * 8u + (uint32_t)ks * 2u);
                            const uint64_t b_desc = desc_hi | (uint64_t)(b16 + (uint32_t)kx * b_step + (uint32_t)ks * 2u);
                            if constexpr (PAIR) umma_bf16_2cta(d_tmem + (uint32_t)sub * block_n, a_desc, b_desc, idesc, (st != st_first || (kx | ks) != 0) ? 1u : 0u);
                            else umma_bf16(d_tmem + (uint32_t)sub * block_n, a_desc, b_desc, idesc, (st != st_first || (kx | ks) != 0) ? 1u : 0u);
                        }
                    }
                };
                if constexpr (KS == 3) {
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) issue_tap(kx);
                } else {
#pragma unroll 1
                    for (int kx = 0; kx < KS; ++kx) issue_tap(kx);
                }
                if constexpr (PAIR) {
                    umma_commit_2cta(&empty_bar[stage]);
                    if (st == st_last) umma_commit_2cta(&tfull_bar[acc]);
                } else {
                    umma_commit(&empty_bar[stage]);
                    if (st == st_last) umma_commit(&tfull_bar[acc]);
                }
            }
            __syncwarp();
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
    }
}

// PAIR = true is the cta_group::2 instantiation: it must be launched as clusters of two CTAs (the driver rejects a
// kernel that contains 2-CTA tcgen05 instructions otherwise), so the single-CTA paths keep their own instantiation.
template <bool PAIR>
__global__ void __launch_bounds__(TC_THREADS, 1) k_conv_tc(const __grid_constant__ ConvTcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte aligned base (swizzle atoms)
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    // barriers first: mbar_wait finds the CTA's wait-failure counter from a barrier's address, so the block must sit on a
    // 1024-byte boundary (tc_smem)
    const TcSmem lay = tc_smem(p);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);
    uint8_t *sA = smem + 1024;
    uint8_t *sB = smem + lay.b;
    uint64_t *full_bar = bars, *empty_bar = bars + TC_MAX_STAGES, *tfull_bar = bars + 2 * TC_MAX_STAGES, *tempty_bar = tfull_bar + 2;
    uint64_t *w_bar = tempty_bar + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(w_bar + 1);
    float *s_bias = reinterpret_cast<float *>(smem + lay.bias);
    // lay.stage, fast_epi == 2: 32 KB of per-warp staging blocks.  Taken from s_bias because the same address written as
    // smem + lay.stage makes k_conv_tc<true> spill registers
    uint8_t *s_stage = reinterpret_cast<uint8_t *>(s_bias + p.d.cout_pad);
    float *s_recv = reinterpret_cast<float *>(s_stage);                      // ksplit > 1: block_n x 128 fp32 receive buffer (no staging then)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const fusg_conv_desc &d = p.d;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA0);
        if (d.in1) tma_prefetch_desc(&p.tmA1);
        tma_prefetch_desc(&p.tmW);
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], PAIR ? 2 * TC_EPI_WARPS : TC_EPI_WARPS); }
        mbar_init(w_bar, 1);
        fusg_wait_guard_start(tmem_slot + 4);      // kernel start time, at bars + TC_WAIT_COUNTER_OFF
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if constexpr (PAIR) tmem_alloc2(tmem_slot, (uint32_t)p.tmem_cols);
        else tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    }
    for (int i = threadIdx.x; i < p.d.cout_pad; i += TC_THREADS) s_bias[i] = p.d.bias[i];
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // the peer's barriers exist before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // programmatic dependent launch: everything above (barriers, TMEM, tensor-map prefetch, bias) touched nothing the
    // previous kernel of the stream produces; wait for it here, then let the next kernel start its own prologue.
    // Few-CTA layers (the coarse scales and the auto-regressive tail) are bound by how fast a handful of SMs can pull their
    // weight slabs (K up to 4608) from HBM: the weights do not depend on the previous kernel, so the grid pulls the whole
    // matrix into L2 NOW, underneath that kernel's tail -- each CTA an equal share, as bulk prefetches
    if (p.w_prefetch_bytes && threadIdx.x == 32) {
        const unsigned long long total = p.w_prefetch_bytes, per = ((total / gridDim.x) + 15ull) & ~15ull;
        unsigned long long lo = per * blockIdx.x, hi = lo + per < total ? lo + per : total;
        const char *wb = reinterpret_cast<const char *>(d.weight);
        for (; lo < hi; lo += 32768ull) {
            const unsigned n = (unsigned)(hi - lo < 32768ull ? hi - lo : 32768ull) & ~15u;
            if (n) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(wb + lo), "r"(n) : "memory");
        }
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // split-K: every CTA of the cluster must be running before a peer writes into its shared memory; arrive now,
    // wait just before the first remote store
    if (p.ksplit > 1) asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");

    const int m_tiles = p.tiles_x * p.tiles_y * p.tiles_b;
    const int total_tiles = m_tiles * p.n_tiles;
    const int pad = d.pad_mode ? d.pad - d.border : d.ksize >> 1;    // pad_mode 1: TMA coordinates are physical (bordered tensor)
    const int cpt = p.chunks0 + p.chunks1;        // k-blocks per tap
    int split_tile = -1;                          // split-K: the tile whose partial accumulator this epilogue warp parked

    if (warp == 0) {
        // =================== TMA producer (whole warp runs the loop; one elected lane issues) ===================
        {
            const int groups = p.kb_local / p.group;
            const int kb0 = p.ksplit > 1 ? (int)cluster_ctarank() * p.kb_local : 0;     // first k-block of this CTA
            const uint32_t stage_tx = (uint32_t)(p.group * (p.a_bytes + (p.w_resident ? 0 : p.b_bytes)));
            if (p.w_resident) {
                // the weight matrix of this N tile is loaded once per CTA
                if (elect_one()) {
                    mbar_arrive_expect_tx(w_bar, (uint32_t)(p.num_kblocks * p.b_bytes));
                    for (int kb = 0; kb < p.num_kblocks; ++kb) tma_load_2d(sB + (size_t)kb * p.b_bytes, &p.tmW, w_bar, kb * p.kc, 0);
                }
                __syncwarp();
            }
            int stage = 0;
            uint32_t phase = 0;
            if (p.halo) {
                const int hks = p.hks;
                // physical coordinate of the first loaded pixel / row: pad_mode 0 -> one pixel of zero fill, pad_mode 1 -> the stored border
                const int hoff = d.pad_mode ? d.border - d.pad : -(hks >> 1);
                const uint32_t tx_bytes = 2u * (uint32_t)((TC_BLOCK_M + hks - 1) * 128) + (p.w_resident ? 0u : (uint32_t)hks * (uint32_t)p.b_bytes);
                constexpr bool pair = PAIR;
                const int rank = pair ? (int)cluster_ctarank() : 0;
                const int tstep = pair ? (int)gridDim.x >> 1 : (int)gridDim.x, tcount = pair ? total_tiles >> 1 : total_tiles;
                for (int it = pair ? (int)blockIdx.x >> 1 : (int)blockIdx.x; it < tcount; it += tstep) {
                    const int tile = pair ? 2 * it + rank : it;        // the two CTAs of a pair take neighbouring M tiles
                    const int mt = p.n_tiles == 1 ? tile : tile / p.n_tiles, nt = tile - mt * p.n_tiles;
                    const int tx = mt & (p.tiles_x - 1), ty = (mt >> p.txs) & (p.tiles_y - 1), tb = mt >> (p.txs + p.tys);
                    const int ox0 = tx * p.Wt, oy0 = ty * p.Ht, b0 = tb * p.Bt, n0 = nt * p.block_n;
                    for (int ky = 0; ky < hks; ++ky) {
                        for (int c = 0; c < cpt; ++c) {
                            if ((p.halo_skip >> (ky * cpt + c)) & 1u) continue;      // all-zero weights: nothing to accumulate
                            mbar_wait(&empty_bar[stage], phase ^ 1);
                            if (elect_one()) {
                                uint8_t *a_dst = sA + (size_t)stage * 2 * TC_HALO_BYTES;
                                uint8_t *b_dst = sB + (size_t)stage * hks * p.b_bytes;
                                if constexpr (PAIR) {
                                    // both CTAs' bytes land on the leader's barrier; only the leader arrives on it
                                    const uint32_t lead = dsmem_addr(s_addr(&full_bar[stage]), 0);
                                    if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2u * tx_bytes);
                                    for (int sub = 0; sub < 2; ++sub) {
                                        if (c < p.chunks0) tma_load_4d_2sm(a_dst + sub * TC_HALO_BYTES, &p.tmA0, lead, c * 64, ox0 + hoff, oy0 + sub + ky + hoff, b0);
                                        else tma_load_4d_2sm(a_dst + sub * TC_HALO_BYTES, &p.tmA1, lead, (c - p.chunks0) * 64, ox0 + hoff, oy0 + sub + ky + hoff, b0);
                                    }
                                    for (int kx = 0; kx < hks; ++kx)     // this CTA's half of the weight rows
                                        tma_load_2d_2sm(b_dst + (size_t)kx * p.b_bytes, &p.tmW, lead, ((ky * hks + kx) * cpt + c) * 64, n0 + rank * (p.block_n >> 1));
                                } else {
                                mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
                                for (int sub = 0; sub < 2; ++sub) {      // sub-tile = image row oy0 + sub, pixels ox0-1 .. ox0+128
                                    if (c < p.chunks0) tma_load_4d(a_dst + sub * TC_HALO_BYTES, &p.tmA0, &full_bar[stage], c * 64, ox0 + hoff, oy0 + sub + ky + hoff, b0);
                                    else tma_load_4d(a_dst + sub * TC_HALO_BYTES, &p.tmA1, &full_bar[stage], (c - p.chunks0) * 64, ox0 + hoff, oy0 + sub + ky + hoff, b0);
                                }
                                if (!p.w_resident) {
                                    for (int kx = 0; kx < hks; ++kx)
                                        tma_load_2d(b_dst + (size_t)kx * p.b_bytes, &p.tmW, &full_bar[stage], ((ky * hks + kx) * cpt + c) * 64, n0);
                                }
                                }
                            }
                            __syncwarp();
                            if (++stage == p.stages) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            } else
            for (int tile = blockIdx.x / p.ksplit; tile < total_tiles; tile += gridDim.x / p.ksplit) {
                const int mt = p.n_tiles == 1 ? tile : tile / p.n_tiles, nt = tile - mt * p.n_tiles;
                const int tx = mt & (p.tiles_x - 1), ty = (mt >> p.txs) & (p.tiles_y - 1), tb = mt >> (p.txs + p.tys);
                const int ox0 = tx * p.Wt, oy0 = ty * p.Ht, b0 = tb * p.Bt;
                const int ixb = ox0 * d.stride - pad, iyb = oy0 * d.stride - pad, n0 = nt * p.block_n;
                // running k-block coordinates (no div/mod in the loop)
                const int tap0 = kb0 / cpt;
                int ky = tap0 / d.ksize, kx = tap0 - ky * d.ksize, cidx = kb0 - tap0 * cpt, kcol = kb0 * p.kc;
                for (int grp = 0; grp < groups; ++grp) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    const bool leader = elect_one();
                    if (leader) mbar_arrive_expect_tx(&full_bar[stage], stage_tx);
                    uint8_t *a_dst = sA + (size_t)stage * p.group * p.a_bytes;
                    uint8_t *b_dst = sB + (size_t)stage * p.group * p.b_bytes;
                    for (int g = 0; g < p.group; ++g) {
                        if (leader) {
                            if (cidx < p.chunks0) tma_load_4d(a_dst, &p.tmA0, &full_bar[stage], cidx * p.kc, ixb + kx, iyb + ky, b0);
                            else tma_load_4d(a_dst, &p.tmA1, &full_bar[stage], (cidx - p.chunks0) * p.kc, ixb + kx, iyb + ky, b0);
                            if (!p.w_resident) tma_load_2d(b_dst, &p.tmW, &full_bar[stage], kcol, n0);
                        }
                        b_dst += p.b_bytes;
                        a_dst += p.a_bytes;
                        kcol += p.kc;                              // weight columns are ordered (tap, in0 channels, in1 channels)
                        if (++cidx == cpt) { cidx = 0; if (++kx == d.ksize) { kx = 0; ++ky; } }
                    }
                    __syncwarp();
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // =================== MMA issuer (whole warp runs the loop; one elected lane issues) ===================
        if (p.halo) {
            if constexpr (PAIR) mma_role_halo<true, 3>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
            else if (p.hks == 3) mma_role_halo<false, 3>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
            else if (p.hks == 5) mma_role_halo<false, 5>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
            else mma_role_halo<false, 7>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
        }
        else if (p.kc == 64) {
            if (p.msub == 2) mma_role<4, 2>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
            else mma_role<4, 1>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
        } else {
            if (p.msub == 2) mma_role<2, 2>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
            else mma_role<2, 1>(p, sA, sB, full_bar, empty_bar, tfull_bar, tempty_bar, w_bar, tmem_base, total_tiles);
        }
    } else {
        // =================== epilogue warps (2..9) ===================
        // warp w may only touch TMEM lanes 32*(w%4)..+31; two warps share a lane quadrant and split the columns
        const int q = warp & 3;
        const int part = (warp - 2) >> 2;                      // 0 .. TC_EPI_WARPS/4 - 1
        const int row = q * 32 + lane;                         // tile row == TMEM lane
        int nparts = TC_EPI_WARPS / 4;
        while (nparts > 1 && p.block_n % (16 * nparts)) nparts >>= 1;
        // narrow layers (one 16-column chunk): the two warps of a lane quadrant split the two sub-tiles instead of the columns
        const bool sub_split = nparts == 1 && p.msub == 2 && p.ksplit == 1;
        const int ncols = sub_split ? p.block_n : (part < nparts ? p.block_n / nparts : 0);
        const int c_begin = sub_split ? 0 : part * ncols;
        int acc = 0;
        uint32_t acc_phase = 0;
        constexpr bool pair = PAIR;
        const int prank = pair ? (int)cluster_ctarank() : 0;
        // CTA pair: the leader's MMA warp waits for the epilogues of BOTH CTAs; the peer arrives on the leader's barrier
        const uint32_t tempty_lead0 = pair ? dsmem_addr(s_addr(&tempty_bar[0]), 0) : 0u, tempty_lead1 = pair ? dsmem_addr(s_addr(&tempty_bar[1]), 0) : 0u;
        const int e_step = pair ? (int)gridDim.x >> 1 : (int)gridDim.x / p.ksplit, e_count = pair ? total_tiles >> 1 : total_tiles;
        for (int it = pair ? (int)blockIdx.x >> 1 : (int)blockIdx.x / p.ksplit; it < e_count; it += e_step) {
            const int tile = pair ? 2 * it + prank : it;
            const int mt = p.n_tiles == 1 ? tile : tile / p.n_tiles, nt = tile - mt * p.n_tiles;
            const int tx = mt & (p.tiles_x - 1), ty = (mt >> p.txs) & (p.tiles_y - 1), tb = mt >> (p.txs + p.tys);
            if (p.ksplit > 1) {
                // ---- split-K: push this CTA's partial accumulator, 16-column chunk by chunk, into the receive buffer of
                // the cluster CTA that owns the chunk (remote stores are fire-and-forget; the cluster barrier after the
                // role code publishes them).  One tile per cluster.
                mbar_wait(&tfull_bar[0], 0);
                tc_fence_after();
                const int S = p.ksplit, cpc = (p.block_n >> 4) / S;    // chunks per owner
                const uint32_t me = cluster_ctarank();
                const uint32_t recv = s_addr(s_recv);                 // [S sources][128 rows][cpc*16 floats]
                const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c_begin;
                asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
                for (int c = 0; c < ncols; c += 16) {
                    uint32_t r[16];
                    tmem_ld16(t_base + (uint32_t)c, r);
                    tmem_ld_wait();
                    const int ch = (c_begin + c) >> 4, owner = ch / cpc, jc = ch - owner * cpc;
                    const uint32_t dst = dsmem_addr(recv + (uint32_t)((((int)me * TC_BLOCK_M + row) * cpc + jc) * 64), (uint32_t)owner);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 16u * i), "r"(r[4 * i]), "r"(r[4 * i + 1]),
                                     "r"(r[4 * i + 2]), "r"(r[4 * i + 3]) : "memory");
                }
                tc_fence_before();
                split_tile = tile;
                break;
            }
            if (p.fast_epi == 2 && ncols > 0) {
                // ---- warp-staged epilogue.  A warp owns 32 consecutive pixels of one image row (Wt >= 32) x ncols
                // channels per sub-tile; residual in and results out go through a 4 KB swizzled staging block so that
                // each global instruction of the warp moves whole 128-byte lines (the direct path touches 32 lines
                // per instruction and saturates the L1TEX data pipe: 74 % lsu wavefronts in r1_ncu_conv_res128raw_B64.csv)
                const int ppr_shift = 31 - __clz(ncols >> 3);      // 16-byte pieces per row: 2, 4 or 8
                const int ppr = 1 << ppr_shift;
                const int rp_shift = 3 - ppr_shift;                // log2(rows per 128 bytes)
                const uint32_t stg = s_addr(s_stage) + (uint32_t)(warp - 2) * (uint32_t)TC_STAGE_BYTES;
                const int n_base = nt * p.block_n + c_begin;
                const FastEpi &fe = p.fe;
                const int sw = (lane >> rp_shift) & (ppr - 1);
                // read-back role of this lane: piece jr of rows rw0, rw0 + rw_step, ...
                const int jr = lane & (ppr - 1), rw0 = lane >> ppr_shift, rw_step = 32 >> ppr_shift;
                bool waited = false;
                // pull the residual rows of this warp's NEXT tile towards L2 now: a prefetch issued at the start of the tile it is
                // for has no lead when the epilogue is the critical path (the accumulator is already complete), and the first
                // use of every residual piece then waits for DRAM (25 % of the samples of the 32-channel 3x3 layers at 256^2)
                if (fe.res && it + e_step < e_count) {
                    const int tile2 = pair ? 2 * (it + e_step) + prank : it + e_step;
                    const int mt2 = p.n_tiles == 1 ? tile2 : tile2 / p.n_tiles, nt2 = tile2 - mt2 * p.n_tiles;
                    const int tx2 = mt2 & (p.tiles_x - 1), ty2 = (mt2 >> p.txs) & (p.tiles_y - 1), tb2 = mt2 >> (p.txs + p.tys);
                    for (int sub = 0; sub < p.msub; ++sub) {
                        const int trow = row + sub * TC_BLOCK_M;
                        const int wt = trow & (p.Wt - 1), ht = (trow >> p.wt_shift) & (p.Ht - 1), bt = trow >> (p.wt_shift + p.ht_shift);
                        const int b2 = tb2 * p.Bt + bt;
                        if (b2 < d.B) {
                            const size_t opix2 = ((size_t)b2 * p.Ho + ty2 * p.Ht + ht) * p.Wo + tx2 * p.Wt + wt;
                            const __nv_bfloat16 *rp2 = fe.res + opix2 * d.cout + nt2 * p.block_n + c_begin;
                            for (int c = 0; c < ncols; c += 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp2 + c));
                        }
                    }
                }
                for (int sub = 0; sub < p.msub; ++sub) {
                    const int trow = row + sub * TC_BLOCK_M;
                    const int wt = trow & (p.Wt - 1), ht = (trow >> p.wt_shift) & (p.Ht - 1), bt = trow >> (p.wt_shift + p.ht_shift);
                    const int ox = tx * p.Wt + wt, oy = ty * p.Ht + ht, b = tb * p.Bt + bt;
                    const size_t opix = ((size_t)b * p.Ho + oy) * p.Wo + ox;
                    const bool valid = b < d.B;                    // uniform across the warp
                    const __nv_bfloat16 *rp = fe.res + opix * d.cout + n_base;
                    if (fe.res && valid) {                         // pull this thread's residual row towards L2 while the MMAs run
                        for (int c = 0; c < ncols; c += 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + c));
                    }
                    // output offset of this lane's read-back piece in the warp's first pixel (x0 = ox - lane, a multiple of 32)
                    const size_t off0 = fast_out_offset(fe, d.cout, p.Ho, p.Wo, b, oy, ox - lane, n_base + 8 * jr);
                    if (!waited) { mbar_wait(&tfull_bar[acc], acc_phase); tc_fence_after(); waited = true; }
                    const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((acc * p.msub + sub) * p.block_n + c_begin);
                    uint32_t r[16];
                    tmem_ld16(t_base, r);
                    for (int c = 0; c < ncols; c += 16) {
                        tmem_ld_wait();
                        float v[16];
                        const float4 *b4 = reinterpret_cast<const float4 *>(s_bias + n_base + c);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 bb = b4[i];
                            v[4 * i] = __uint_as_float(r[4 * i]) + bb.x;
                            v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + bb.y;
                            v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + bb.z;
                            v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + bb.w;
                        }
                        if (c + 16 < ncols) tmem_ld16(t_base + (uint32_t)(c + 16), r);  // prefetch the next chunk
                        const int j0 = c >> 3;
                        const uint32_t s0 = stg + (uint32_t)(((lane << ppr_shift) + (j0 ^ sw)) << 4);
                        const uint32_t s1 = stg + (uint32_t)(((lane << ppr_shift) + ((j0 + 1) ^ sw)) << 4);
                        if (fe.res && valid) {
                            const uint4 *rq = reinterpret_cast<const uint4 *>(rp + c);
                            const uint4 q0 = __ldg(rq), q1 = __ldg(rq + 1);
                            const uint32_t w[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
                            for (int i = 0; i < 8; ++i) { v[2 * i] += bf16lo_to_f(w[i]); v[2 * i + 1] += bf16hi_to_f(w[i]); }
                        }
                        if (fe.f16) {
                            sts128(s0, make_uint4(pack_f16x2(v[0], v[1]), pack_f16x2(v[2], v[3]), pack_f16x2(v[4], v[5]), pack_f16x2(v[6], v[7])));
                            sts128(s1, make_uint4(pack_f16x2(v[8], v[9]), pack_f16x2(v[10], v[11]), pack_f16x2(v[12], v[13]), pack_f16x2(v[14], v[15])));
                        } else {
                            sts128(s0, make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7])));
                            sts128(s1, make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15])));
                        }
                    }
                    __syncwarp();
                    if (sub == p.msub - 1) {                       // all TMEM reads of this tile are done: release the buffer early
                        tc_fence_before();
                        if (lane == 0) {
                            if constexpr (PAIR) mbar_arrive_cluster(acc ? tempty_lead1 : tempty_lead0);
                            else mbar_arrive(&tempty_bar[acc]);
                        }
                    }
                    if (valid) {                                   // transposed read-back: 8 lanes cover one pixel's 128 bytes
                        for (int rw = rw0; rw < 32; rw += rw_step) {
                            const uint4 val = lds128(stg + (uint32_t)(((rw << ppr_shift) + (jr ^ ((rw >> rp_shift) & (ppr - 1)))) << 4));
                            const size_t off = off0 + (size_t)((rw >> 1) * fe.stride_a + (rw & 1) * fe.stride_b);
                            if (fe.raw) *reinterpret_cast<uint4 *>(fe.raw + off) = val;
                            if (fe.elu) *reinterpret_cast<uint4 *>(fe.elu + off) = elu_piece(val);
                        }
                    }
                    __syncwarp();
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                continue;
            }
            if (p.fast_epi && p.fe.res && ncols > 0) {
                // the residual rows this thread will add: pull them into L2 while the MMAs of this tile run
                for (int sub = 0; sub < p.msub; ++sub) {
                    if (sub_split && sub != part) continue;
                    const int trow = row + sub * TC_BLOCK_M;
                    const int wt = trow & (p.Wt - 1), ht = (trow >> p.wt_shift) & (p.Ht - 1), bt = trow >> (p.wt_shift + p.ht_shift);
                    const int b = tb * p.Bt + bt;
                    if (b < d.B) {
                        const size_t opix = ((size_t)b * p.Ho + ty * p.Ht + ht) * p.Wo + tx * p.Wt + wt;
                        const __nv_bfloat16 *rp = p.fe.res + opix * d.cout + nt * p.block_n + c_begin;
                        for (int c = 0; c < ncols; c += 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + c));
                    }
                }
            }
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            for (int sub = 0; sub < p.msub && ncols > 0; ++sub) {
                if (sub_split && sub != part) continue;
                const int trow = row + sub * TC_BLOCK_M;               // row of the CTA tile
                const int wt = trow & (p.Wt - 1), ht = (trow >> p.wt_shift) & (p.Ht - 1), bt = trow >> (p.wt_shift + p.ht_shift);
                const int ox = tx * p.Wt + wt, oy = ty * p.Ht + ht, b = tb * p.Bt + bt;
                const size_t opix = ((size_t)b * p.Ho + oy) * p.Wo + ox;
                const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((acc * p.msub + sub) * p.block_n + c_begin);
                uint32_t r[16];
                tmem_ld16(t_base, r);
                for (int c = 0; c < ncols; c += 16) {
                    tmem_ld_wait();
                    uint32_t rr[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) rr[i] = r[i];
                    if (c + 16 < ncols) tmem_ld16(t_base + (uint32_t)(c + 16), r);      // prefetch the next chunk
                    if (b < d.B) {
                        const int n = nt * p.block_n + c_begin + c;
                        if (p.fast_epi == 3) unpair_chunk(reinterpret_cast<float *>(p.fe.raw), s_bias, d.cout >> 1, p.Ho, p.Wo, b, oy, ox, rr);
                        else if (p.fast_epi) fast_chunk16(p.fe, s_bias, d.cout, p.Ho, p.Wo, opix, b, oy, ox, n, rr);
                        else {
                            float v[16];
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rr[i]);
                            epilogue16<__nv_bfloat16>(d, s_bias, p.Ho, p.Wo, b, oy, ox, n, v);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (PAIR) mbar_arrive_cluster(acc ? tempty_lead1 : tempty_lead0);
                else mbar_arrive(&tempty_bar[acc]);
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    if (p.ksplit > 1) {
        // split-K reduction: CTA r of the cluster owns the 16-column chunks [r*cpc, (r+1)*cpc) of the tile; every CTA
        // has pushed its partials of those chunks into this CTA's receive buffer.  Sum them in rank order
        // (deterministic) and run the normal epilogue.
        __syncwarp();
        if (warp < 2) asm volatile("barrier.cluster.wait.aligned;" ::: "memory");   // pairs with the arrive of the prologue
        cluster_sync_all();
        if (warp >= 2 && split_tile >= 0) {
            const int q = warp & 3, part = (warp - 2) >> 2, row = q * 32 + lane;
            const int S = p.ksplit, cpc = (p.block_n >> 4) / S;
            const int crank = (int)cluster_ctarank();
            const int mt = p.n_tiles == 1 ? split_tile : split_tile / p.n_tiles, nt = split_tile - mt * p.n_tiles;
            const int tx = mt & (p.tiles_x - 1), ty = (mt >> p.txs) & (p.tiles_y - 1), tb = mt >> (p.txs + p.tys);
            const int wt = row & (p.Wt - 1), ht = (row >> p.wt_shift) & (p.Ht - 1), bt = row >> (p.wt_shift + p.ht_shift);
            const int ox = tx * p.Wt + wt, oy = ty * p.Ht + ht, b = tb * p.Bt + bt;
            const size_t opix = ((size_t)b * p.Ho + oy) * p.Wo + ox;
            const float4 *recv = reinterpret_cast<const float4 *>(s_recv);
            for (int j = part; j < cpc; j += TC_EPI_WARPS / 4) {
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = 0.f;
                for (int src = 0; src < S; ++src) {
                    const float4 *pr = recv + ((size_t)(src * TC_BLOCK_M + row) * cpc + j) * 4;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 t = pr[i];
                        v[4 * i] += t.x; v[4 * i + 1] += t.y; v[4 * i + 2] += t.z; v[4 * i + 3] += t.w;
                    }
                }
                if (b < d.B) {
                    const int n = nt * p.block_n + (crank * cpc + j) * 16;
                    if (p.fast_epi) {
                        uint32_t rr[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) rr[i] = __float_as_uint(v[i]);
                        fast_chunk16(p.fe, s_bias, d.cout, p.Ho, p.Wo, opix, b, oy, ox, n, rr);
                    } else {
                        epilogue16<__nv_bfloat16>(d, s_bias, p.Ho, p.Wo, b, oy, ox, n, v);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();    // the peer may still be signalling this CTA's barriers / reading its operands
    if (warp == 1) {
        tc_fence_after();
        if constexpr (PAIR) tmem_dealloc2(tmem_base, (uint32_t)p.tmem_cols);
        else tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
    }
}

// ------------------------------------------------------------------------------------------------
// layout / weight helpers
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_fold_weightnorm(const float *__restrict__ v, const float *__restrict__ g, T *__restrict__ w, int cout, int cin, int ks,
                                  int cout_pad, int cin_pad) {
    // one CTA per (padded) output channel
    const int n = blockIdx.x;
    const int taps = ks * ks, len = cin * taps;
    __shared__ float red[32];
    float ss = 0.f;
    if (n < cout) for (int i = threadIdx.x; i < len; i += blockDim.x) { const float a = v[(size_t)n * len + i]; ss += a * a; }
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (threadIdx.x == 0) red[0] = t;
    }
    __syncthreads();
    const float scale = n < cout ? g[n] / sqrtf(red[0]) : 0.f;
    for (int i = threadIdx.x; i < taps * cin_pad; i += blockDim.x) {
        const int tap = i / cin_pad, c = i - tap * cin_pad;
        float val = 0.f;
        if (n < cout && c < cin) val = v[((size_t)n * cin + c) * taps + tap] * scale;
        w[((size_t)n * taps + tap) * cin_pad + c] = from_f<T>(val);
    }
}

// weight_norm fold for pixel-pair packed execution (see fusg.h).  One CTA per padded output channel
// n' = dx*cout + co; K index = tap' * 2*(c0+c1) + [in0: h*c0 + ci | in1: 2*c0 + h*c1 + ci].
template <typename T>
__global__ void k_fold_weightnorm_paired(const float *__restrict__ v, const float *__restrict__ g, const float *__restrict__ bias,
                                         T *__restrict__ w, float *__restrict__ bias_out, int cout, int c0, int c1, int ks, int cout_pad) {
    const int np = blockIdx.x;
    const int cin = c0 + c1, taps = ks * ks, len = cin * taps, kp = 2 * cin;
    const int dx = np / cout, co = np - dx * cout;
    const bool real = np < 2 * cout;
    __shared__ float red[32];
    float ss = 0.f;
    if (real) for (int i = threadIdx.x; i < len; i += blockDim.x) { const float a = v[(size_t)co * len + i]; ss += a * a; }
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (threadIdx.x == 0) red[0] = t;
    }
    __syncthreads();
    const float scale = real ? g[co] / sqrtf(red[0]) : 0.f;
    if (threadIdx.x == 0) bias_out[np] = real ? bias[co] : 0.f;
    for (int i = threadIdx.x; i < taps * kp; i += blockDim.x) {
        const int tap = i / kp, k = i - tap * kp;
        int src_c, h;                                   // original input channel and input half
        if (k < 2 * c0) { h = k / c0; src_c = k - h * c0; }
        else { const int kk = k - 2 * c0; h = kk / c1; src_c = c0 + (kk - h * c1); }
        float val = 0.f;
        if (real) {
            if (ks == 1) {
                if (h == dx) val = v[(size_t)co * cin + src_c] * scale;
            } else {
                const int ky = tap / 3, s = tap - ky * 3 - 1;          // pair shift -1, 0, +1
                const int kx = 2 * s + h - dx + 1;
                if (kx >= 0 && kx < 3) val = v[((size_t)co * cin + src_c) * 9 + ky * 3 + kx] * scale;
            }
        }
        w[((size_t)np * taps + tap) * kp + k] = from_f<T>(val);
    }
}

// NCHW fp32 -> NHWC (zero-padded channels, optional ELU).  One thread per pixel: the per-channel reads
// are coalesced across the warp, the writes are 16-byte pieces of the thread's own contiguous pixel row.
// gridDim.y > 1: one thread per (pixel, 8-channel group) instead -- the Sampler noise tensors are a few hundred pixels of
// 128 channels, and a thread that walks all 16 groups of its pixel is one long chain of strided loads (20-40 us per
// launch, ten launches at the head of every step).
template <typename T>
__global__ void k_nchw_to_nhwc(const float *__restrict__ in, T *__restrict__ out, int C, int HW, int cpad, int elu, size_t npix) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // over B*HW
    if (i >= npix) return;
    const size_t b = i / HW, pix = i - b * HW;
    const float *src = in + b * C * HW + pix;
    T *dst = out + i * cpad;
    const int c_lo = gridDim.y > 1 ? (int)blockIdx.y * 8 : 0, c_hi = gridDim.y > 1 ? c_lo + 8 : cpad;
    for (int c0 = c_lo; c0 < c_hi; c0 += 8) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float a = 0.f;
            if (c0 + k < C) { a = __ldg(src + (size_t)(c0 + k) * HW); if (elu) a = elu1(a); }
            v[k] = a;
        }
        if constexpr (std::is_same_v<T, __nv_bfloat16>) {
            *reinterpret_cast<uint4 *>(dst + c0) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        } else if constexpr (std::is_same_v<T, __half>) {
            __half2 h[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) h[k] = __floats2half2_rn(v[2 * k], v[2 * k + 1]);
            *reinterpret_cast<uint4 *>(dst + c0) = *reinterpret_cast<const uint4 *>(h);
        } else {
            *reinterpret_cast<float4 *>(dst + c0) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4 *>(dst + c0 + 4) = make_float4(v[4], v[5], v[6], v[7]);
        }
    }
}

template <typename T>
__global__ void k_nhwc_to_nchw(const T *__restrict__ in, float *__restrict__ out, int C, int HW, int pitch, size_t total) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // over B*C*HW (output order)
    if (i >= total) return;
    const size_t pix = i % HW;
    const size_t bc = i / HW;
    const size_t b = bc / C, c = bc % C;
    out[i] = to_f<T>(in[(b * HW + pix) * pitch + c]);
}

template <typename T>
__global__ void k_elu(const T *__restrict__ in, T *__restrict__ out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = from_f<T>(elu1(to_f<T>(in[i])));
}

__global__ void k_to_image(const float *__restrict__ in, uint8_t *__restrict__ out, int HW, size_t total) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // over B*HW*3 (output order)
    if (i >= total) return;
    const int c = (int)(i % 3);
    const size_t bp = i / 3;
    const size_t b = bp / HW, pix = bp % HW;
    // numpy evaluates (x + 1.) / 2 * 255 in fp32 for a float32 array
    float v = (in[(b * 3 + c) * HW + pix] + 1.f) / 2.f * 255.f;
    v = fminf(fmaxf(v, 0.f), 255.f);
    out[i] = (uint8_t)v;                                               // astype(np.uint8): truncation
}

}  // namespace fusg

// ================================================================================================
// host side
// ================================================================================================
using namespace fusg;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

static int conv_out_size(int in, int ks, int stride, int pad) { return (in + 2 * pad - ks) / stride + 1; }
static int desc_pad(const fusg_conv_desc &d) { return d.pad_mode ? d.pad : d.ksize / 2; }

static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

static bool tc_supported(const fusg_conv_desc &d, int Ho, int Wo) {
    if (d.dtype != FUSG_DTYPE_BF16 && d.dtype != FUSG_DTYPE_F16) return false;
    if (d.dtype == FUSG_DTYPE_F16) {
        // fp16 activations (the ICN row): raw NHWC outputs or NCHW fp32 slots only -- no residual, noise or ELU copy
        // A raw NHWC fp16 slot is written by the lean epilogue only, so it must be the launch's one output: the general
        // epilogue (epilogue16<__nv_bfloat16>) would store it as bf16.
        if (d.residual || d.noise) return false;
        int nouts = 0, nhwc = 0;
        for (int s = 0; s < FUSG_CONV_MAX_OUTS; ++s) {
            if (!d.outs[s].ptr) continue;
            ++nouts;
            if (d.outs[s].layout == 0) {
                ++nhwc;
                if (d.outs[s].elu || d.outs[s].mode != FUSG_OUT_PLAIN || d.outs[s].source || d.cout % 16) return false;
            }
        }
        if (nhwc && nouts > 1) return false;
    }
    if (d.c0 % 32 != 0 || (d.in1 && d.c1 % 32 != 0)) return false;
    if (d.cout_pad % 16 != 0) return false;
    if (!is_pow2(Ho) || !is_pow2(Wo)) return false;
    if (d.cout_pad > 128 && d.cout_pad % 128 != 0) return false;
    if (d.pitch0 % 8 != 0 || (d.in1 && d.pitch1 % 8 != 0)) return false;   // 16-byte global strides for TMA
    return get_encode() != nullptr;
}

// SMs the persistent conv grids leave free for kernels of other streams (fusg_conv2d_set_sm_reserve)
static int g_sm_reserve = 0;

extern "C" int fusg_conv2d_set_sm_reserve(int n) {
    const int prev = g_sm_reserve;
    if (n >= 0) g_sm_reserve = n;
    return prev;
}

// tiling plan of this host thread's last tcgen05 launch (fusg_conv2d_last_plan)
static thread_local int32_t g_last_plan[8];

extern "C" void fusg_conv2d_last_plan(int32_t *plan8) {
    for (int i = 0; i < 8; ++i) plan8[i] = g_last_plan[i];
}

// Tiling policy of k_conv_tc: fills every field of p except the three tensor maps, the grid size and the dynamic
// shared-memory size.  Reads nothing but its arguments and g_sm_reserve.
static int plan_tc(const fusg_conv_desc &d, int Ho, int Wo, int num_sms, ConvTcParams &p, int &grid, size_t &smem) {
    memset(&p, 0, sizeof(p));
    p.d = d;
    p.Ho = Ho; p.Wo = Wo;
    p.block_n = d.cout_pad < 128 ? d.cout_pad : 128;
    p.n_tiles = d.cout_pad / p.block_n;
    // 256-row CTA tiles (two 128-row MMA sub-tiles sharing each weight k-block) once there is enough work for
    // at least ~4 tiles per SM; halves the weight traffic per output pixel
    const long long rows = (long long)d.B * Ho * Wo;
    // (1x1 layers too: half as many barrier round trips per output row -- 0.51 -> 0.46 ms on the 6->128 NiN)
    p.msub = (rows / 256 * p.n_tiles >= 4LL * num_sms && rows % 256 == 0) ? 2 : 1;
    const int trows = TC_BLOCK_M * p.msub;
    p.Wt = Wo < 128 ? Wo : 128;
    p.Ht = (trows / p.Wt) < Ho ? (trows / p.Wt) : Ho;
    p.Bt = trows / (p.Wt * p.Ht);
    p.tiles_x = Wo / p.Wt; p.tiles_y = Ho / p.Ht; p.tiles_b = (d.B + p.Bt - 1) / p.Bt;
    const int total_tiles = p.tiles_x * p.tiles_y * p.tiles_b * p.n_tiles;
    auto ilog2 = [](int v) { int sh = 0; while ((1 << sh) < v) ++sh; return sh; };
    p.wt_shift = ilog2(p.Wt); p.ht_shift = ilog2(p.Ht); p.txs = ilog2(p.tiles_x); p.tys = ilog2(p.tiles_y);
    const bool k64 = (d.c0 % 64 == 0) && (!d.in1 || d.c1 % 64 == 0);
    p.kc = k64 ? 64 : 32;
    p.chunks0 = d.c0 / p.kc;
    p.chunks1 = d.in1 ? d.c1 / p.kc : 0;
    const int taps = d.ksize * d.ksize;
    p.num_kblocks = taps * (p.chunks0 + p.chunks1);
    p.a_bytes = TC_BLOCK_M * p.msub * p.kc * 2;
    p.b_bytes = p.block_n * p.kc * 2;
    // B k-blocks must start 1024-aligned too (swizzle atom): round the size up
    p.b_bytes = (p.b_bytes + 1023) & ~1023;
    // few-tile layers (the coarse scales and the auto-regressive tail): a cluster of `ksplit` CTAs per tile, each
    // streaming 1/ksplit of the K range (at least 36 k-blocks in all), then a DSMEM reduce-scatter -- a single SM pulls
    // ~50-80 GB/s through TMA, so a 128 x 4608 weight slab per CTA costs ~45 us however few tiles there are
    p.ksplit = 1;
    if (p.msub == 1 && p.block_n % 16 == 0) {
        for (int sk = 8; sk >= 2; sk >>= 1) {
            if (total_tiles * sk > 128) continue;
            if (p.num_kblocks % sk || p.num_kblocks < 36) continue;
            if ((p.block_n / 16) % sk) continue;
            p.ksplit = sk;
            break;
        }
    }
    p.kb_local = p.num_kblocks / p.ksplit;
    // warp-staged epilogue for the big layers (needs 32 KB): applies to the lean-epilogue case with Wt >= 32
    // (1x1 layers too: their direct epilogue touches 32 lines per store instruction -- 64 % LSU wavefronts, 236 -> 169 us on the 32->32 skip NiN at 256^2)
    bool want_staged = p.ksplit == 1 && p.Wt >= 32 && p.block_n >= 32 && is_pow2(p.block_n) && d.noise == nullptr && d.cout % 16 == 0;
    const int smem_budget = (want_staged ? 168 : 200) * 1024 - (p.ksplit > 1 ? p.block_n * TC_BLOCK_M * 4 : 0);
    // weights resident when the whole (single) N tile fits next to a useful pipeline
    p.w_resident = (p.ksplit == 1 && p.n_tiles == 1 && p.num_kblocks * p.b_bytes <= 72 * 1024) ? 1 : 0;
    const int avail = smem_budget - (p.w_resident ? p.num_kblocks * p.b_bytes : 0);
    const int kb_bytes = p.a_bytes + (p.w_resident ? 0 : p.b_bytes);
    // group = k-blocks per barrier round trip: the largest divisor of num_kblocks that keeps the
    // stage <= 64 KB and leaves >= 3 stages
    int group = 1;
    for (int g = 1; g <= p.kb_local; ++g) {
        if (p.kb_local % g) continue;
        if (g * kb_bytes > 64 * 1024) break;
        if (avail / (g * kb_bytes) >= 3) group = g;
    }
    p.group = group;
    int stages = avail / (group * kb_bytes);
    if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
    if (stages < 2) stages = 2;
    p.stages = stages;
    // sliding-window (halo) A tiles for the wide-frame 3x3 layers: one row-segment load serves the three horizontal taps
    p.hks = d.ksize;
    const bool halo_ks = d.pad_mode ? (d.ksize == 3 || d.ksize == 5 || d.ksize == 7) : d.ksize == 3;
    if (p.ksplit == 1 && halo_ks && d.stride == 1 && p.kc == 64 && p.msub == 2 && p.Wt == 128 && p.Ht == 2 && p.Bt == 1) {
        // CTA pairs (cta_group::2) for the 128-wide layers: each CTA keeps half of the weight rows, which makes room for
        // a third pipeline stage, and every MMA reads a quarter less shared memory
        p.pair = (d.ksize == 3 && p.block_n == 128 && p.n_tiles == 1 && !p.w_resident && total_tiles % 2 == 0 && total_tiles >= 4 * num_sms) ? 1 : 0;
        if (p.pair) p.b_bytes = (p.block_n / 2) * p.kc * 2;                 // half of the weight rows per CTA and k-block
        const int stage_bytes = 2 * TC_HALO_BYTES + (p.w_resident ? 0 : d.ksize * p.b_bytes);
        // wide kernels (5x5 / 7x7): a third pipeline stage is worth more than the staged epilogue's 32 KB
        if (d.ksize > 3 && want_staged && (192 * 1024) / stage_bytes < 3 && (222 * 1024) / stage_bytes >= 3) want_staged = false;
        const int budget = (want_staged ? 192 : 222) * 1024 - (p.w_resident ? p.num_kblocks * p.b_bytes : 0);
        int st = budget / stage_bytes;
        if (st > TC_MAX_STAGES) st = TC_MAX_STAGES;
        if (st >= 2) { p.halo = 1; p.stages = st; p.group = 1; }
        else if (p.pair) return FUSG_ERR_UNSUPPORTED;
    }
    if (p.halo && d.zero_kblocks && d.ksize == 3) {
        const int cpt = p.chunks0 + p.chunks1;
        for (int ky = 0; ky < 3 && 9 * cpt <= 64; ++ky)
            for (int c = 0; c < cpt; ++c) {
                bool all = true;
                for (int kx = 0; kx < 3; ++kx) all = all && ((d.zero_kblocks >> ((ky * 3 + kx) * cpt + c)) & 1ull);
                if (all) p.halo_skip |= 1u << (ky * cpt + c);
            }
        if (p.halo_skip == (1u << (3 * cpt)) - 1u) p.halo_skip = 0;          // (a layer of zeros: keep the plain schedule)
    }
    int cols = 2 * p.msub * p.block_n;
    p.tmem_cols = cols < 32 ? 32 : cols;
    p.epi_smem = want_staged ? TC_STAGING_BYTES : (p.ksplit > 1 ? p.block_n * TC_BLOCK_M * 4 : 0);

    // lean epilogue: no noise, only NHWC bf16 outputs (<= one raw, <= one ELU) with one addressing mode
    {
        bool ok = d.noise == nullptr && d.cout % 16 == 0;
        FastEpi fe;
        memset(&fe, 0, sizeof(fe));
        fe.res = reinterpret_cast<const __nv_bfloat16 *>(d.residual);
        int mode = -1;
        for (int sidx = 0; sidx < FUSG_CONV_MAX_OUTS && ok; ++sidx) {
            const fusg_conv_out &o = d.outs[sidx];
            if (!o.ptr) continue;
            if (o.layout != 0 || o.source != 0 || o.elu > 1) { ok = false; break; }
            if (mode == -1) { mode = o.mode; fe.blk = o.blk; }
            else if (mode != o.mode || fe.blk != o.blk) { ok = false; break; }
            if (o.elu) { if (fe.elu) ok = false; fe.elu = reinterpret_cast<__nv_bfloat16 *>(o.ptr); }
            else { if (fe.raw) ok = false; fe.raw = reinterpret_cast<__nv_bfloat16 *>(o.ptr); }
        }
        if (ok && mode == FUSG_OUT_D2S) {
            const int cq = d.cout / 4;
            if (!is_pow2(cq) || cq < 16) ok = false;
            else { int sh = 0; while ((1 << sh) < cq) ++sh; fe.cq_shift = sh; }
        }
        fe.mode = mode < 0 ? 0 : mode;
        fe.f16 = d.dtype == FUSG_DTYPE_F16 ? 1 : 0;
        switch (fe.mode) {
            default: fe.stride_a = 2 * d.cout; fe.stride_b = d.cout; break;
            case FUSG_OUT_D2S: fe.stride_a = d.cout; fe.stride_b = d.cout / 2; break;          // 4*cq, 2*cq with cq = cout/4
            case FUSG_OUT_S2D: fe.stride_a = 4 * d.cout; fe.stride_b = d.cout; break;
            case FUSG_OUT_D2S_BLOCK: fe.stride_a = 4 * d.cout; fe.stride_b = 2 * d.cout; break;
        }
        p.fast_epi = ok ? (want_staged ? 2 : 1) : 0;
        // pixel-pair packed layer -> NCHW fp32, nothing else (the network's last convolution)
        if (!ok && p.ksplit == 1 && d.noise == nullptr && d.residual == nullptr && d.dtype == FUSG_DTYPE_BF16 && d.cout <= 16 && d.cout % 2 == 0 && p.block_n == 16) {
            int nouts = 0;
            const fusg_conv_out *only = nullptr;
            for (int sidx = 0; sidx < FUSG_CONV_MAX_OUTS; ++sidx)
                if (d.outs[sidx].ptr) { ++nouts; only = &d.outs[sidx]; }
            if (nouts == 1 && only->layout == 1 && only->mode == FUSG_OUT_UNPAIR && only->source == 0 && only->elu == 0 &&
                (reinterpret_cast<uintptr_t>(only->ptr) & 7) == 0) {
                memset(&fe, 0, sizeof(fe));
                fe.raw = reinterpret_cast<__nv_bfloat16 *>(only->ptr);        // (an fp32 NCHW tensor on this path)
                p.fast_epi = 3;
            }
        }
        p.fe = fe;
    }
    const unsigned long long wbytes = (unsigned long long)d.cout_pad * taps * (d.c0 + d.c1) * 2ull;
    p.w_prefetch_bytes = (total_tiles * p.ksplit <= 64 && wbytes >= 65536ull && (reinterpret_cast<uintptr_t>(d.weight) & 15) == 0) ? wbytes : 0ull;
    // persistent CTAs own a STATIC share of the tiles, and one CTA fills an SM: if a co-tenant (the solver warps of the warp
    // stage that runs next to the VUNet in a pipeline step) holds even one SM, the CTA meant for it starts only when another
    // CTA has finished its whole share -- the layer takes twice as long.  g_sm_reserve SMs are therefore left to co-tenants.
    const int usable = num_sms - g_sm_reserve > 8 ? num_sms - g_sm_reserve : num_sms;
    grid = p.ksplit > 1 ? total_tiles * p.ksplit /* one cluster per tile */ : (total_tiles < usable ? total_tiles : usable);
    if (p.pair) grid &= ~1;                                                  // whole CTA pairs
    smem = tc_smem(p).total;
    return FUSG_OK;
}

static int launch_tc(const fusg_conv_desc &d, int Ho, int Wo, cudaStream_t st) {
    ConvTcParams p;
    int grid;
    size_t smem;
    const int rc = plan_tc(d, Ho, Wo, fusg_num_sms(), p, grid, smem);
    if (rc != FUSG_OK) return rc;
    PFN_encodeTiled enc = get_encode();
    const CUtensorMapSwizzle sw = p.kc == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    // c = channels the tensor really holds: a k-block box that reaches beyond them is zero-filled by TMA
    auto encodeA = [&](CUtensorMap *tm, const void *ptr, int c, int pitch) -> bool {
        const int bd = d.pad_mode ? d.border : 0;
        const cuuint64_t Wp = (cuuint64_t)(d.W + 2 * bd), Hp = (cuuint64_t)(d.H + 2 * bd);
        cuuint64_t dims[4] = {(cuuint64_t)c, Wp, Hp, (cuuint64_t)d.B};
        cuuint64_t strides[3] = {(cuuint64_t)pitch * 2, Wp * pitch * 2, Hp * Wp * pitch * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.kc, (cuuint32_t)(p.Wt * d.stride), (cuuint32_t)(p.Ht * d.stride), (cuuint32_t)p.Bt};
        if (p.halo) { box[1] = (cuuint32_t)(TC_BLOCK_M + d.ksize - 1); box[2] = 1; box[3] = 1; }
        cuuint32_t estr[4] = {1, (cuuint32_t)d.stride, (cuuint32_t)d.stride, 1};
        return enc(tm, d.dtype == FUSG_DTYPE_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    };
    if (!encodeA(&p.tmA0, d.in0, d.cphys0 ? d.cphys0 : d.c0, d.pitch0)) return FUSG_ERR_UNSUPPORTED;
    if (d.in1 && !encodeA(&p.tmA1, d.in1, d.cphys1 ? d.cphys1 : d.c1, d.pitch1)) return FUSG_ERR_UNSUPPORTED;
    {
        const int ktot = d.ksize * d.ksize * (d.c0 + d.c1);
        cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)d.cout_pad};
        cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
        cuuint32_t box[2] = {(cuuint32_t)p.kc, (cuuint32_t)(p.pair ? p.block_n / 2 : p.block_n)};
        cuuint32_t estr[2] = {1, 1};
        if (enc(&p.tmW, d.dtype == FUSG_DTYPE_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(d.weight), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return FUSG_ERR_UNSUPPORTED;
    }
    if (fusg_once_per_device(0, 0, [] {
            cudaError_t e = cudaFuncSetAttribute(k_conv_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
            return e != cudaSuccess ? e : cudaFuncSetAttribute(k_conv_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        }) != cudaSuccess)
        return fusg_check_launch();
    g_last_plan[0] = p.msub; g_last_plan[1] = p.pair; g_last_plan[2] = p.halo; g_last_plan[3] = p.ksplit;
    g_last_plan[4] = p.stages; g_last_plan[5] = p.group; g_last_plan[6] = p.w_resident; g_last_plan[7] = p.fast_epi;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3(TC_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    // programmatic stream serialization: the kernel's prologue overlaps the previous kernel (griddepcontrol in k_conv_tc)
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    int na = 1;
    if (p.ksplit > 1 || p.pair) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = p.pair ? 2u : (unsigned)p.ksplit;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = (unsigned)na;
    if ((p.pair ? cudaLaunchKernelEx(&cfg, k_conv_tc<true>, p) : cudaLaunchKernelEx(&cfg, k_conv_tc<false>, p)) != cudaSuccess) return fusg_check_launch();
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" size_t fusg_sizeof_conv_desc(void) { return sizeof(fusg_conv_desc); }

// ------------------------------------------------------------------------------------------------
// FUSG_IMPL_SMALLCIN: 1x1 convolution of a network INPUT (NiN of the 6- / 3-channel images, vunet/models.py:141-150,
// stored 16 channels wide, of which at most 8 are real) -- K is so small that the layer is a pure stream: read 32 bytes per pixel, write cout bf16 raw
// and/or ELU values per pixel.  On the tensor-core kernel its epilogue warps (8 of 12) are the bottleneck (0.50 ms for the
// 6->128 layer at 64 crops, 2.2 TB/s); here EVERY thread is an "epilogue" thread: a thread owns 8 output channels, keeps
// their 8 x 8 weights in registers and walks over pixels, four in flight; 16-byte coalesced stores.
// ------------------------------------------------------------------------------------------------
constexpr int SC_THREADS = 256;
constexpr int SC_CIN = 8;                                  // real input channels served (the images have 6 and 3)
constexpr int SC_PIX = 4;                                  // pixels in flight per thread: their loads are issued before any math

__global__ void __launch_bounds__(SC_THREADS, 2) k_conv1x1_smallcin(const __nv_bfloat16 *__restrict__ in, int pitch_in, const __nv_bfloat16 *__restrict__ w,
                                                                    int cin_pad, const float *__restrict__ bias, __nv_bfloat16 *__restrict__ raw,
                                                                    __nv_bfloat16 *__restrict__ elu, int cout, long long npix) {
    const int chunks = cout >> 3;                          // 16-byte output chunks per pixel
    const int chunk = threadIdx.x % chunks, pl = threadIdx.x / chunks, ppc = SC_THREADS / chunks;
    float wr[8][SC_CIN], bs[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) {
        bs[o] = bias[chunk * 8 + o];
        const uint4 a = *reinterpret_cast<const uint4 *>(w + (size_t)(chunk * 8 + o) * cin_pad);
        const uint32_t ww[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) { wr[o][2 * c] = bf16lo_to_f(ww[c]); wr[o][2 * c + 1] = bf16hi_to_f(ww[c]); }
    }
    if (pl >= ppc) return;                                 // (cout/8 not a divisor of 256: idle tail threads)
    const long long step = (long long)gridDim.x * ppc;
    for (long long p0 = (long long)blockIdx.x * ppc + pl; p0 < npix; p0 += step * SC_PIX) {
        uint4 xin[SC_PIX];
#pragma unroll
        for (int j = 0; j < SC_PIX; ++j) {
            const long long p = p0 + j * step;
            xin[j] = p < npix ? __ldg(reinterpret_cast<const uint4 *>(in + (size_t)p * pitch_in)) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int j = 0; j < SC_PIX; ++j) {
            const long long p = p0 + j * step;
            if (p >= npix) break;
            const uint32_t xw[4] = {xin[j].x, xin[j].y, xin[j].z, xin[j].w};
            float x[SC_CIN];
#pragma unroll
            for (int c = 0; c < 4; ++c) { x[2 * c] = bf16lo_to_f(xw[c]); x[2 * c + 1] = bf16hi_to_f(xw[c]); }
            uint32_t pk[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float s0 = bs[2 * i], s1 = bs[2 * i + 1];
#pragma unroll
                for (int c = 0; c < SC_CIN; ++c) { s0 = fmaf(wr[2 * i][c], x[c], s0); s1 = fmaf(wr[2 * i + 1][c], x[c], s1); }
                pk[i] = pack_bf16x2(s0, s1);
            }
            const size_t off = (size_t)p * cout + chunk * 8;
            if (raw) *reinterpret_cast<uint4 *>(raw + off) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            if (elu) {
                uint32_t ek[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) ek[i] = pack_bf16x2(elu1(bf16lo_to_f(pk[i])), elu1(bf16hi_to_f(pk[i])));   // ELU of the rounded value, like the tensor-core epilogue
                *reinterpret_cast<uint4 *>(elu + off) = make_uint4(ek[0], ek[1], ek[2], ek[3]);
            }
        }
    }
}

// the layers FUSG_IMPL_SMALLCIN serves: one bf16 input stored 16 channels wide of which <= 8 are real (cin_real), 1x1, stride 1,
// plain NHWC bf16 outputs
static bool smallcin_supported(const fusg_conv_desc &d, __nv_bfloat16 **raw, __nv_bfloat16 **elu) {
    if (d.dtype != FUSG_DTYPE_BF16 || d.ksize != 1 || d.stride != 1 || d.pad_mode != 0 || d.in1 || d.residual || d.noise) return false;
    if (d.cphys0 != 16 || d.pitch0 != 16 || d.cin_real <= 0 || d.cin_real > SC_CIN || d.cout % 8 || d.cout > 256 || SC_THREADS % (d.cout / 8)) return false;
    if ((reinterpret_cast<uintptr_t>(d.in0) & 15) || (reinterpret_cast<uintptr_t>(d.weight) & 15)) return false;
    __nv_bfloat16 *r = nullptr, *e = nullptr;
    for (int s = 0; s < FUSG_CONV_MAX_OUTS; ++s) {
        const fusg_conv_out &o = d.outs[s];
        if (!o.ptr) continue;
        if (o.layout != 0 || o.source != 0 || o.mode != FUSG_OUT_PLAIN || o.elu > 1 || (reinterpret_cast<uintptr_t>(o.ptr) & 15)) return false;
        if (o.elu) { if (e) return false; e = reinterpret_cast<__nv_bfloat16 *>(o.ptr); }
        else { if (r) return false; r = reinterpret_cast<__nv_bfloat16 *>(o.ptr); }
    }
    if (raw) *raw = r;
    if (elu) *elu = e;
    return r || e;
}

extern "C" int fusg_conv2d_select(const fusg_conv_desc *desc) {
    if (!desc) return FUSG_ERR_ARG;
    const int Ho = conv_out_size(desc->H, desc->ksize, desc->stride, desc_pad(*desc)), Wo = conv_out_size(desc->W, desc->ksize, desc->stride, desc_pad(*desc));
    if (smallcin_supported(*desc, nullptr, nullptr)) return FUSG_IMPL_SMALLCIN;
    return tc_supported(*desc, Ho, Wo) ? FUSG_IMPL_TCGEN05 : FUSG_IMPL_DIRECT;
}

extern "C" int fusg_conv2d(const fusg_conv_desc *desc, void *stream) {
    if (!desc || !desc->in0 || !desc->weight || !desc->bias) return FUSG_ERR_ARG;
    const fusg_conv_desc &d = *desc;
    if (d.B <= 0 || d.H <= 0 || d.W <= 0 || d.c0 <= 0 || d.cout <= 0 || d.cout_pad < d.cout) return FUSG_ERR_ARG;
    if (d.stride != 1 && d.stride != 2) return FUSG_ERR_UNSUPPORTED;
    if (d.pad_mode == 0) {
        if (d.ksize != 1 && d.ksize != 3) return FUSG_ERR_UNSUPPORTED;
    } else {
        if (d.pad_mode != 1 || d.ksize < 1 || d.ksize > 7 || d.pad < 0 || d.border < d.pad) return FUSG_ERR_UNSUPPORTED;
    }
    if (d.in1 == nullptr && d.c1 != 0) return FUSG_ERR_ARG;
    if (d.cphys0 < 0 || d.cphys0 > d.c0 || d.cphys0 % 8 || d.cphys1 < 0 || d.cphys1 > d.c1 || d.cphys1 % 8) return FUSG_ERR_ARG;
    if ((d.cphys0 && d.pitch0 < d.cphys0) || (d.cphys1 && d.pitch1 < d.cphys1)) return FUSG_ERR_ARG;
    if (d.dtype != FUSG_DTYPE_BF16 && d.dtype != FUSG_DTYPE_F32 && d.dtype != FUSG_DTYPE_F16) return FUSG_ERR_ARG;
    bool any_out = false, need_noise = false;
    for (int s = 0; s < FUSG_CONV_MAX_OUTS; ++s) {
        if (!d.outs[s].ptr) continue;
        any_out = true;
        if (d.outs[s].source == 1) need_noise = true;
        if (d.outs[s].mode == FUSG_OUT_D2S && (d.cout % 4 != 0 || (d.cout / 4) % 16 != 0)) return FUSG_ERR_UNSUPPORTED;
    }
    if (!any_out || (need_noise && !d.noise)) return FUSG_ERR_ARG;
    const int Ho = conv_out_size(d.H, d.ksize, d.stride, desc_pad(d)), Wo = conv_out_size(d.W, d.ksize, d.stride, desc_pad(d));
    if (Ho <= 0 || Wo <= 0) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int impl = d.impl;
    __nv_bfloat16 *sc_raw = nullptr, *sc_elu = nullptr;
    if (impl == FUSG_IMPL_AUTO) impl = smallcin_supported(d, &sc_raw, &sc_elu) ? FUSG_IMPL_SMALLCIN : (tc_supported(d, Ho, Wo) ? FUSG_IMPL_TCGEN05 : FUSG_IMPL_DIRECT);
    if (impl == FUSG_IMPL_SMALLCIN) {
        if (!smallcin_supported(d, &sc_raw, &sc_elu)) return FUSG_ERR_UNSUPPORTED;
        const long long npix = (long long)d.B * d.H * d.W;
        const int ppc = SC_THREADS / (d.cout / 8);
        const long long want = (npix + ppc - 1) / ppc;
        const int grid = (int)(want < (long long)fusg_num_sms() * 2 ? want : (long long)fusg_num_sms() * 2);
        // weights: [cout_pad][1][cin_pad] bf16, the first 8 input channels of every row (the rest is the zero padding of K)
        k_conv1x1_smallcin<<<grid, SC_THREADS, 0, st>>>(reinterpret_cast<const __nv_bfloat16 *>(d.in0), d.pitch0, reinterpret_cast<const __nv_bfloat16 *>(d.weight),
                                                      d.c0, d.bias, sc_raw, sc_elu, d.cout, npix);
        fusg_count_launch(1);
        return fusg_check_launch();
    }
    if (impl == FUSG_IMPL_TCGEN05) {
        if (!tc_supported(d, Ho, Wo)) return FUSG_ERR_UNSUPPORTED;
        return launch_tc(d, Ho, Wo, st);
    }
    const long long total = (long long)d.B * Ho * Wo;
    dim3 grid((unsigned)((total + 127) / 128), (unsigned)((d.cout_pad + 15) / 16));
    if (d.dtype == FUSG_DTYPE_BF16) k_conv_direct<__nv_bfloat16><<<grid, 128, 0, st>>>(d, Ho, Wo);
    else if (d.dtype == FUSG_DTYPE_F16) k_conv_direct<__half><<<grid, 128, 0, st>>>(d, Ho, Wo);
    else k_conv_direct<float><<<grid, 128, 0, st>>>(d, Ho, Wo);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_fold_weightnorm(const float *v, const float *g, void *w_out, int cout, int cin, int ksize, int cout_pad, int cin_pad,
                                    int dtype, void *stream) {
    if (!v || !g || !w_out || cout <= 0 || cin <= 0 || cout_pad < cout || cin_pad < cin) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == FUSG_DTYPE_BF16) k_fold_weightnorm<__nv_bfloat16><<<cout_pad, 256, 0, st>>>(v, g, (__nv_bfloat16 *)w_out, cout, cin, ksize, cout_pad, cin_pad);
    else if (dtype == FUSG_DTYPE_F16) k_fold_weightnorm<__half><<<cout_pad, 256, 0, st>>>(v, g, (__half *)w_out, cout, cin, ksize, cout_pad, cin_pad);
    else if (dtype == FUSG_DTYPE_F32) k_fold_weightnorm<float><<<cout_pad, 256, 0, st>>>(v, g, (float *)w_out, cout, cin, ksize, cout_pad, cin_pad);
    else return FUSG_ERR_ARG;
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_fold_weightnorm_paired(const float *v, const float *g, const float *bias, void *w_out, float *bias_out, int cout,
                                           int cin0, int cin1, int ksize, int cout_pad, int dtype, void *stream) {
    if (!v || !g || !bias || !w_out || !bias_out || cout <= 0 || cin0 <= 0 || cin1 < 0 || cout_pad < 2 * cout) return FUSG_ERR_ARG;
    if (ksize != 1 && ksize != 3) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == FUSG_DTYPE_BF16) k_fold_weightnorm_paired<__nv_bfloat16><<<cout_pad, 256, 0, st>>>(v, g, bias, (__nv_bfloat16 *)w_out, bias_out, cout, cin0, cin1, ksize, cout_pad);
    else if (dtype == FUSG_DTYPE_F16) k_fold_weightnorm_paired<__half><<<cout_pad, 256, 0, st>>>(v, g, bias, (__half *)w_out, bias_out, cout, cin0, cin1, ksize, cout_pad);
    else if (dtype == FUSG_DTYPE_F32) k_fold_weightnorm_paired<float><<<cout_pad, 256, 0, st>>>(v, g, bias, (float *)w_out, bias_out, cout, cin0, cin1, ksize, cout_pad);
    else return FUSG_ERR_ARG;
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_nchw_to_nhwc(const float *in, void *out, int B, int C, int H, int W, int cpad, int elu, int dtype, void *stream) {
    if (!in || !out || B <= 0 || C <= 0 || cpad < C) return FUSG_ERR_ARG;
    if (cpad % 8 != 0) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t npix = (size_t)B * H * W;
    // small tensors (the Sampler noise): a thread per (pixel, 8-channel group), 64-thread blocks
    const bool split = npix < 16384 && cpad > 8;
    const dim3 grid((unsigned)((npix + (split ? 63 : 255)) / (split ? 64 : 256)), split ? (unsigned)(cpad / 8) : 1u);
    const unsigned threads = split ? 64 : 256;
    if (dtype == FUSG_DTYPE_BF16) k_nchw_to_nhwc<__nv_bfloat16><<<grid, threads, 0, st>>>(in, (__nv_bfloat16 *)out, C, H * W, cpad, elu, npix);
    else if (dtype == FUSG_DTYPE_F16) k_nchw_to_nhwc<__half><<<grid, threads, 0, st>>>(in, (__half *)out, C, H * W, cpad, elu, npix);
    else if (dtype == FUSG_DTYPE_F32) k_nchw_to_nhwc<float><<<grid, threads, 0, st>>>(in, (float *)out, C, H * W, cpad, elu, npix);
    else return FUSG_ERR_ARG;
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_nhwc_to_nchw(const void *in, float *out, int B, int C, int H, int W, int pitch, int dtype, void *stream) {
    if (!in || !out || B <= 0 || C <= 0 || pitch < C) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t total = (size_t)B * C * H * W;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (dtype == FUSG_DTYPE_BF16) k_nhwc_to_nchw<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16 *)in, out, C, H * W, pitch, total);
    else if (dtype == FUSG_DTYPE_F16) k_nhwc_to_nchw<__half><<<grid, 256, 0, st>>>((const __half *)in, out, C, H * W, pitch, total);
    else if (dtype == FUSG_DTYPE_F32) k_nhwc_to_nchw<float><<<grid, 256, 0, st>>>((const float *)in, out, C, H * W, pitch, total);
    else return FUSG_ERR_ARG;
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_to_image(const float *in, uint8_t *out, int B, int H, int W, void *stream) {
    if (!in || !out || B <= 0 || H <= 0 || W <= 0) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t total = (size_t)B * H * W * 3;
    k_to_image<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, out, H * W, total);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_elu(const void *in, void *out, size_t n, int dtype, void *stream) {
    if (!in || !out || n == 0) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (dtype == FUSG_DTYPE_BF16) k_elu<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16 *)in, (__nv_bfloat16 *)out, n);
    else if (dtype == FUSG_DTYPE_F16) k_elu<__half><<<grid, 256, 0, st>>>((const __half *)in, (__half *)out, n);
    else if (dtype == FUSG_DTYPE_F32) k_elu<float><<<grid, 256, 0, st>>>((const float *)in, (float *)out, n);
    else return FUSG_ERR_ARG;
    fusg_count_launch(1);
    return fusg_check_launch();
}
