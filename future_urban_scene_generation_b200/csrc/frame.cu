// frame.cu -- paste-back of completed vehicle crops into video frames (include/fusg.h: fusg_resize_u8, fusg_paste_back).
//
// Reference semantics: trajectory_inference.py:236-250 (also :184-198, :393-407, :428-442), per vehicle
//     crop_inv = cv2.resize(net_image, crop_size_orig[::-1]);  crop_inv = crop_inv[pad_before : -pad_after]
//     out_frame = zeros;  out_frame[crop_xy_min ...] = crop_inv;  img_output[dst_sketch_mask] = out_frame[dst_sketch_mask]
// with crop_info from warp_learn/models.py:334-342.  Vehicles are pasted in sequence, so where masks overlap the last
// vehicle wins.  Here the whole batch is two launches: k_paste_owner resolves "last writer" per frame pixel with an
// atomicMax over the item index, k_paste_apply evaluates cv2.resize (INTER_LINEAR, 8-bit) pointwise for exactly the
// pixels that survive -- no intermediate resized crop, no per-vehicle frame-sized temporaries.
//
// cv2.resize is restated from its observable behaviour (OpenCV 4.13; oracle/frame_oracle.py holds the same
// statement in numpy, pinned to cv2 by tests/golden/frame_golden.json): double scale = 1/(dst/src), float coordinate,
// 11-bit coefficients rounded half-to-even, int32 horizontal pass, (((b0*(S0>>4))>>16) + ((b1*(S1>>4))>>16) + 2) >> 2
// vertically; an exact halving in both axes is a 2x2 box average.  Compiled with -fmad=false: the coordinate
// arithmetic must round like the host code it mirrors.
#include <cstdint>

#include "../../include/fusg.h"
#include "fusg_common.h"

namespace fusg {

struct Tap { int i0, i1, a0, a1; };

// coefficient pair of destination index d on an axis of sn source and dn destination samples
__device__ __forceinline__ Tap resize_tap(int dn, int sn, int d, bool horizontal) {
    const double scale = 1.0 / ((double)dn / (double)sn);
    float f = (float)(((double)d + 0.5) * scale - 0.5);
    int s = (int)floorf(f);
    f = f - (float)s;
    Tap t;
    if (horizontal) {
        if (s < 0) { s = 0; f = 0.f; }
        if (s >= sn - 1) { s = sn - 1; f = 0.f; }
        t.i0 = s;
        t.i1 = min(s + 1, sn - 1);
    } else {
        t.i0 = min(max(s, 0), sn - 1);
        t.i1 = min(max(s + 1, 0), sn - 1);
    }
    t.a0 = __float2int_rn((1.f - f) * 2048.f);
    t.a1 = __float2int_rn(f * 2048.f);
    return t;
}

// pixel (y, x) of cv2.resize(src[sh, sw, 3], (dw, dh)); three channels
__device__ __forceinline__ void resize_pixel(const uint8_t *__restrict__ src, int sh, int sw, int dh, int dw, int y, int x, uint8_t out[3]) {
    if (sw == 2 * dw && sh == 2 * dh) {
        const uint8_t *p = src + ((size_t)(2 * y) * sw + 2 * x) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) out[c] = (uint8_t)((p[c] + p[3 + c] + p[(size_t)sw * 3 + c] + p[(size_t)sw * 3 + 3 + c] + 2) >> 2);
        return;
    }
    const Tap tx = resize_tap(dw, sw, x, true), ty = resize_tap(dh, sh, y, false);
    const uint8_t *r0 = src + (size_t)ty.i0 * sw * 3, *r1 = src + (size_t)ty.i1 * sw * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int s0 = r0[tx.i0 * 3 + c] * tx.a0 + r0[tx.i1 * 3 + c] * tx.a1;
        const int s1 = r1[tx.i0 * 3 + c] * tx.a0 + r1[tx.i1 * 3 + c] * tx.a1;
        const int v = (((ty.a0 * (s0 >> 4)) >> 16) + ((ty.a1 * (s1 >> 4)) >> 16) + 2) >> 2;
        out[c] = (uint8_t)min(max(v, 0), 255);
    }
}

// one thread per destination pixel; blockIdx.y = item
__global__ void __launch_bounds__(256) k_resize_u8(const uint8_t *__restrict__ src, const long long *__restrict__ src_off,
                                                   const int *__restrict__ src_hw, uint8_t *__restrict__ dst,
                                                   const long long *__restrict__ dst_off, const int *__restrict__ dst_hw) {
    const int b = blockIdx.y;
    const int sh = src_hw[2 * b], sw = src_hw[2 * b + 1], dh = dst_hw[2 * b], dw = dst_hw[2 * b + 1];
    const uint8_t *s = src + src_off[b];
    uint8_t *d = dst + dst_off[b];
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < (long long)dh * dw; p += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(p / dw), x = (int)(p - (long long)y * dw);
        uint8_t o[3];
        resize_pixel(s, sh, sw, dh, dw, y, x, o);
        d[p * 3] = o[0]; d[p * 3 + 1] = o[1]; d[p * 3 + 2] = o[2];
    }
}

constexpr int PASTE_INFO = 9;   // frame, h_orig, w_orig, pad_x0, pad_y0, pad_x1, pad_y1, x_min, y_min

// owner[frame][y][x] = highest item index whose mask covers the pixel (-1: nobody).  An item whose frame index is outside [0, F) --
// possible when the info comes from device data (fusg_crop_geometry's frame_index) that the host never range-checked -- pastes nothing.
__global__ void __launch_bounds__(256) k_paste_owner(const uint8_t *__restrict__ masks, const long long *__restrict__ mask_off,
                                                     const int *__restrict__ mask_rect, const int *__restrict__ info,
                                                     int *__restrict__ owner, int F, int Hf, int Wf) {
    const int b = blockIdx.y;
    const int x0 = mask_rect[4 * b], y0 = mask_rect[4 * b + 1], w = mask_rect[4 * b + 2], h = mask_rect[4 * b + 3];
    const int frame = info[PASTE_INFO * b];
    if (frame < 0 || frame >= F) return;
    const uint8_t *m = masks + mask_off[b];
    int *own = owner + (size_t)frame * Hf * Wf;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < (long long)w * h; p += (long long)gridDim.x * blockDim.x) {
        if (!m[p]) continue;
        const int yy = (int)(p / w), xx = (int)(p - (long long)yy * w);
        const int fy = y0 + yy, fx = x0 + xx;
        if (fy >= 0 && fy < Hf && fx >= 0 && fx < Wf) atomicMax(&own[(size_t)fy * Wf + fx], b);
    }
}

__global__ void __launch_bounds__(256) k_paste_apply(uint8_t *__restrict__ frames, const uint8_t *__restrict__ crops,
                                                     const int *__restrict__ info, const int *__restrict__ owner, int Hf, int Wf, int S) {
    const int frame = blockIdx.y;
    const size_t fbase = (size_t)frame * Hf * Wf;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < (long long)Hf * Wf; p += (long long)gridDim.x * blockDim.x) {
        const int o = owner[fbase + p];
        if (o < 0) continue;
        const int *in = info + PASTE_INFO * o;
        const int h = in[1], w = in[2], px0 = in[3], py0 = in[4], px1 = in[5], py1 = in[6], xmin = in[7], ymin = in[8];
        const int y = (int)(p / Wf), x = (int)(p - (long long)y * Wf);
        const int ry = y - ymin, rx = x - xmin;
        uint8_t v[3] = {0, 0, 0};                              // out_frame is zero outside the pasted rectangle
        if (ry >= 0 && ry < h - py0 - py1 && rx >= 0 && rx < w - px0 - px1)
            resize_pixel(crops + (size_t)o * S * S * 3, S, S, h, w, ry + py0, rx + px0, v);
        uint8_t *d = frames + (fbase + p) * 3;
        d[0] = v[0]; d[1] = v[1]; d[2] = v[2];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// VUNet input packing (trajectory_inference.py:205-227): bbox of the vehicle mask -> square crop (utils/crop_utils.py:
// 4-52) of the masked frame and of the two normal sketches -> cv2.resize to res x res -> background fill ->
// to_tensor (utils/misc_utils.py:35-50) -> channel flip / concat.  Everything is pointwise in the output pixel once the
// bbox is known, so it is one reduction kernel (k_mask_bbox) and one gather kernel (k_pack_inputs).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mask_bbox(const uint8_t *__restrict__ masks, const long long *__restrict__ off,
                                                   const int *__restrict__ rect, int *__restrict__ bbox) {
    const int b = blockIdx.y;
    const int x0 = rect[4 * b], y0 = rect[4 * b + 1], w = rect[4 * b + 2], h = rect[4 * b + 3];
    const uint8_t *m = masks + off[b];
    int xmin = 0x7fffffff, ymin = 0x7fffffff, xmax = -1, ymax = -1;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < (long long)w * h; p += (long long)gridDim.x * blockDim.x) {
        if (!m[p]) continue;
        const int yy = (int)(p / w), xx = (int)(p - (long long)yy * w);
        xmin = min(xmin, x0 + xx); xmax = max(xmax, x0 + xx);
        ymin = min(ymin, y0 + yy); ymax = max(ymax, y0 + yy);
    }
    for (int o = 16; o > 0; o >>= 1) {
        xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, o)); ymin = min(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
        xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o)); ymax = max(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
    }
    if ((threadIdx.x & 31) == 0 && xmax >= 0) {
        atomicMin(&bbox[4 * b], xmin); atomicMin(&bbox[4 * b + 1], ymin);
        atomicMax(&bbox[4 * b + 2], xmax); atomicMax(&bbox[4 * b + 3], ymax);
    }
}

__global__ void k_bbox_init(int *__restrict__ bbox, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) { bbox[4 * b] = 0x7fffffff; bbox[4 * b + 1] = 0x7fffffff; bbox[4 * b + 2] = -1; bbox[4 * b + 3] = -1; }
}

struct CropGeom { int nx0, ny0, pxb, pyb, pxa, pya, cw, ch; };

// utils/crop_utils.py:14-50 for dataset='pascal' (Python float = double, int() truncates toward zero -- also for the values in
// (-1, 0), which give 0).  Each fp64 operation rounds on its own, as in the interpreter.
__device__ __forceinline__ CropGeom crop_geometry(const int *bb, int image_h, int image_w) {
    const int x_min = bb[0], y_min = bb[1], side_x = bb[2] - bb[0], side_y = bb[3] - bb[1];
    const double major = __dmul_rn((double)max(side_x, side_y), 1.1), half = __ddiv_rn(major, 2.0);
    const double cx = __dadd_rn((double)x_min, __ddiv_rn((double)side_x, 2.0)), cy = __dadd_rn((double)y_min, __ddiv_rn((double)side_y, 2.0));
    CropGeom g;
    g.pxb = g.pyb = g.pxa = g.pya = 0;
    g.nx0 = (int)__dsub_rn(cx, half);
    if (g.nx0 < 0) { g.pxb = -g.nx0; g.nx0 = 0; }
    int nx1 = (int)__dadd_rn(cx, half) + g.pxb;
    if (nx1 > image_w) { g.pxa = nx1 - image_w; nx1 = image_w + g.pxa; }
    g.ny0 = (int)__dsub_rn(cy, half);
    if (g.ny0 < 0) { g.pyb = -g.ny0; g.ny0 = 0; }
    int ny1 = (int)__dadd_rn(cy, half) + g.pyb;
    if (ny1 > image_h) { g.pya = ny1 - image_h; ny1 = image_h + g.pya; }
    g.cw = min(nx1, image_w + g.pxb + g.pxa) - g.nx0;
    g.ch = min(ny1, image_h + g.pyb + g.pya) - g.ny0;
    return g;
}

// ---------------------------------------------------------------------------------------------------------------
// Crop geometry of a batch of sketch masks on the device (fusg_crop_geometry): from fusg_mask_bbox's output, what the kernels
// downstream read -- paste info (frame_ops.pack_crop_info of square_crop_info), the ICN window (icn_window_rect) and its byte
// offset (window_layout: exclusive scan of 16-byte-aligned five-plane blocks, in item order) -- plus a status per item.
// B is a few thousand at most, so one CTA walks the items in chunks with a block-wide scan and a running carry.
// ---------------------------------------------------------------------------------------------------------------
constexpr int GEOM_THREADS = 1024;

// icn_window_rect along one axis: the frame span [a, a+n) the resize taps of a crop side of `size` read (size 0 reads index -1)
__device__ __forceinline__ void window_span(int n0, int pad, int size, int limit, int &a, int &n) {
    const int lo = size > 0 ? n0 - pad : n0 - pad - 1;
    a = max(lo, 0);
    int e = min(lo + max(size, 1), limit);
    if (e <= a) { a = min(max(lo, 0), limit - 1); e = a + 1; }
    n = e - a;
}

__global__ void __launch_bounds__(GEOM_THREADS) k_crop_geometry(const int32_t *__restrict__ bbox, const int32_t *__restrict__ frame_index, int B,
                                                                int Hf, int Wf, long long capacity, int max_win_h, int32_t *__restrict__ info,
                                                                int32_t *__restrict__ win, long long *__restrict__ win_off,
                                                                int8_t *__restrict__ status) {
    __shared__ long long s_warp[GEOM_THREADS / 32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    for (int base = 0; base < B; base += GEOM_THREADS) {
        const int b = base + threadIdx.x;
        int st = 0, in[PASTE_INFO] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, wx = 0, wy = 0, ww = 0, wh = 0;
        long long bytes = 0;
        if (b < B) {
            in[0] = frame_index ? frame_index[b] : 0;
            if (bbox[4 * b + 2] < 0) {
                st = 1;                                                      // empty mask: fusg_mask_bbox's (INT_MAX, INT_MAX, -1, -1)
            } else {
                const CropGeom g = crop_geometry(bbox + 4 * b, Hf, Wf);
                in[1] = g.ch; in[2] = g.cw; in[3] = g.pxb; in[4] = g.pyb; in[5] = g.pxa; in[6] = g.pya; in[7] = g.nx0; in[8] = g.ny0;
                window_span(g.nx0, g.pxb, g.cw, Wf, wx, ww);
                window_span(g.ny0, g.pyb, g.ch, Hf, wy, wh);
                bytes = ((5LL * ww * wh * 3) + 15) & ~15LL;
            }
        }
        long long v = bytes;                                                 // inclusive scan of the block sizes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long n = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += n;
        }
        __syncthreads();                                                     // s_warp / s_carry of the previous chunk consumed
        if (lane == 31) s_warp[wid] = v;
        __syncthreads();
        if (wid == 0) {
            long long w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long n = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += n;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const long long end = s_carry + (wid ? s_warp[wid - 1] : 0) + v, off = end - bytes;
        if (b < B) {
            // the offsets only grow: the first block that ends past the capacity refuses itself and every later item
            if (st == 0 && capacity > 0 && (end > capacity || wh > max_win_h)) st = 2;
            int32_t *io = info + (size_t)PASTE_INFO * b;
#pragma unroll
            for (int k = 0; k < PASTE_INFO; ++k) io[k] = in[k];
            if (win) {
                const bool ok = st == 0;
                win[4 * b] = ok ? wx : 0; win[4 * b + 1] = ok ? wy : 0; win[4 * b + 2] = ok ? ww : 0; win[4 * b + 3] = ok ? wh : 0;
            }
            if (win_off) win_off[b] = off;
            status[b] = (int8_t)st;
        }
        __syncthreads();
        if (threadIdx.x == GEOM_THREADS - 1) s_carry = end;
    }
}

struct Px9 { uint8_t m[3], ns[3], nd[3]; };

// pixel (cy, cx) of the three square crops: masked frame, source normals, destination normals (zero in the padding)
__device__ __forceinline__ Px9 pack_fetch(const uint8_t *__restrict__ frame, const uint8_t *__restrict__ mask, const uint8_t *__restrict__ nsrc,
                                          const uint8_t *__restrict__ ndst, const CropGeom &g, int rx0, int ry0, int rw, int rh, int Hf, int Wf,
                                          int cy, int cx) {
    Px9 p;
#pragma unroll
    for (int c = 0; c < 3; ++c) p.m[c] = p.ns[c] = p.nd[c] = 0;
    const int fy = g.ny0 + cy - g.pyb, fx = g.nx0 + cx - g.pxb;
    if (fy < 0 || fy >= Hf || fx < 0 || fx >= Wf) return p;
    const int yy = fy - ry0, xx = fx - rx0;
    if (yy < 0 || yy >= rh || xx < 0 || xx >= rw) return p;          // outside the item's rectangle everything is background
    const size_t q = (size_t)yy * rw + xx;
    const bool veh = mask[q] != 0;
    const uint8_t *fp = frame + ((size_t)fy * Wf + fx) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) { p.m[c] = veh ? fp[c] : 0; p.ns[c] = nsrc[q * 3 + c]; p.nd[c] = ndst[q * 3 + c]; }
    return p;
}

__device__ __forceinline__ float to_tensor1(int v) { return ((float)v / 255.f) * 2.f - 1.f; }

__global__ void __launch_bounds__(256) k_pack_inputs(const uint8_t *__restrict__ frames, const int *__restrict__ frame_idx,
                                                     const uint8_t *__restrict__ masks, const uint8_t *__restrict__ nsrc,
                                                     const uint8_t *__restrict__ ndst, const long long *__restrict__ off,
                                                     const int *__restrict__ rect, const int *__restrict__ bbox, float *__restrict__ x,
                                                     float *__restrict__ y, int Hf, int Wf, int res) {
    const int b = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= res * res) return;
    const size_t plane = (size_t)res * res;
    float *xb = x + (size_t)b * 6 * plane + p, *yb = y + (size_t)b * 3 * plane + p;
    if (frame_idx[b] < 0) {                                                     // a refused item: zero rows
#pragma unroll
        for (int ch = 0; ch < 6; ++ch) xb[ch * plane] = 0.f;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) yb[ch * plane] = 0.f;
        return;
    }
    const int oy = p / res, ox = p - oy * res;
    const CropGeom g = crop_geometry(bbox + 4 * b, Hf, Wf);
    const uint8_t *frame = frames + (size_t)frame_idx[b] * Hf * Wf * 3;
    const uint8_t *mk = masks + off[b], *ns = nsrc + off[b] * 3, *nd = ndst + off[b] * 3;
    const int rx0 = rect[4 * b], ry0 = rect[4 * b + 1], rw = rect[4 * b + 2], rh = rect[4 * b + 3];
    int vm[3], vs[3], vd[3];
    if (g.cw == 2 * res && g.ch == 2 * res) {                                  // exact halving -> 2x2 box average
        const Px9 a = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, 2 * oy, 2 * ox);
        const Px9 bq = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, 2 * oy, 2 * ox + 1);
        const Px9 c = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, 2 * oy + 1, 2 * ox);
        const Px9 d = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, 2 * oy + 1, 2 * ox + 1);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            vm[ch] = (a.m[ch] + bq.m[ch] + c.m[ch] + d.m[ch] + 2) >> 2;
            vs[ch] = (a.ns[ch] + bq.ns[ch] + c.ns[ch] + d.ns[ch] + 2) >> 2;
            vd[ch] = (a.nd[ch] + bq.nd[ch] + c.nd[ch] + d.nd[ch] + 2) >> 2;
        }
    } else {
        const Tap tx = resize_tap(res, g.cw, ox, true), ty = resize_tap(res, g.ch, oy, false);
        const Px9 p00 = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, ty.i0, tx.i0);
        const Px9 p01 = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, ty.i0, tx.i1);
        const Px9 p10 = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, ty.i1, tx.i0);
        const Px9 p11 = pack_fetch(frame, mk, ns, nd, g, rx0, ry0, rw, rh, Hf, Wf, ty.i1, tx.i1);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            int s0 = p00.m[ch] * tx.a0 + p01.m[ch] * tx.a1, s1 = p10.m[ch] * tx.a0 + p11.m[ch] * tx.a1;
            vm[ch] = min(max((((ty.a0 * (s0 >> 4)) >> 16) + ((ty.a1 * (s1 >> 4)) >> 16) + 2) >> 2, 0), 255);
            s0 = p00.ns[ch] * tx.a0 + p01.ns[ch] * tx.a1; s1 = p10.ns[ch] * tx.a0 + p11.ns[ch] * tx.a1;
            vs[ch] = min(max((((ty.a0 * (s0 >> 4)) >> 16) + ((ty.a1 * (s1 >> 4)) >> 16) + 2) >> 2, 0), 255);
            s0 = p00.nd[ch] * tx.a0 + p01.nd[ch] * tx.a1; s1 = p10.nd[ch] * tx.a0 + p11.nd[ch] * tx.a1;
            vd[ch] = min(max((((ty.a0 * (s0 >> 4)) >> 16) + ((ty.a1 * (s1 >> 4)) >> 16) + 2) >> 2, 0), 255);
        }
    }
    if (vs[0] == 0 && vs[1] == 0 && vs[2] == 0) vm[0] = vm[1] = vm[2] = 255;      // trajectory_inference.py:219-220
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        xb[ch * plane] = to_tensor1(vm[ch]);                  // x_1: masked frame crop, channel order kept
        xb[(3 + ch) * plane] = to_tensor1(vs[2 - ch]);        // x_2: source normals, [..., ::-1]
        yb[ch * plane] = to_tensor1(vd[2 - ch]);              // y_tilde: destination normals, [..., ::-1]
    }
}

// to_tensor + channel flip + concat of the three already-resized uint8 images of trajectory_inference.py:215-227
__global__ void __launch_bounds__(256) k_u8_to_inputs(const uint8_t *__restrict__ m, const uint8_t *__restrict__ ns, const uint8_t *__restrict__ nd,
                                                      float *__restrict__ x, float *__restrict__ y, int res) {
    const int b = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= res * res) return;
    const size_t plane = (size_t)res * res, q = ((size_t)b * plane + p) * 3;
    float *xb = x + (size_t)b * 6 * plane + p, *yb = y + (size_t)b * 3 * plane + p;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        xb[ch * plane] = to_tensor1(m[q + ch]);
        xb[(3 + ch) * plane] = to_tensor1(ns[q + 2 - ch]);
        yb[ch * plane] = to_tensor1(nd[q + 2 - ch]);
    }
}

// y alone (the trajectory step: the appearance image x is encoded once per vehicle, not per item) -- the same arithmetic
__global__ void __launch_bounds__(256) k_u8_to_y(const uint8_t *__restrict__ nd, float *__restrict__ y, int res) {
    const int b = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= res * res) return;
    const size_t plane = (size_t)res * res, q = ((size_t)b * plane + p) * 3;
    float *yb = y + (size_t)b * 3 * plane + p;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) yb[ch * plane] = to_tensor1(nd[q + 2 - ch]);
}

// ---------------------------------------------------------------------------------------------------------------
// Per-item gather of per-vehicle rows: dst row b of every segment = src row index[b] (zeros for an index out of range).  The
// segment table travels in the kernel's parameter space, so a captured graph holds it by value.  grid (segment, item, split):
// a CTA copies a 1/split share of one row with 16-byte vectors.
// ---------------------------------------------------------------------------------------------------------------
struct GatherTable { fusg_gather_seg s[FUSG_GATHER_MAX_SEGS]; };

constexpr int GATHER_THREADS = 256;

__global__ void __launch_bounds__(GATHER_THREADS) k_gather_rows(const GatherTable tab, const int32_t *__restrict__ index) {
    const fusg_gather_seg &sg = tab.s[blockIdx.x];
    const int b = blockIdx.y;
    const long long n16 = sg.row_bytes / 16;
    const long long per = (n16 + gridDim.z - 1) / gridDim.z, k0 = per * blockIdx.z, k1 = min(n16, k0 + per);
    if (k0 >= n16) return;
    const int r = index[b];
    int4 *d = reinterpret_cast<int4 *>(static_cast<uint8_t *>(sg.dst) + (size_t)b * sg.row_bytes);
    if (r < 0 || r >= sg.n_src) {
        for (long long k = k0 + threadIdx.x; k < k1; k += GATHER_THREADS) d[k] = make_int4(0, 0, 0, 0);
        return;
    }
    const int4 *s4 = reinterpret_cast<const int4 *>(static_cast<const uint8_t *>(sg.src) + (size_t)r * sg.row_bytes);
    for (long long k = k0 + threadIdx.x; k < k1; k += GATHER_THREADS) d[k] = __ldg(s4 + k);
}

// ---------------------------------------------------------------------------------------------------------------
// ICN input packing (warp_learn/models.py:323-366 get_icn_inputs): square crop (bbox of the sketch mask) + cv2.resize of the
// destination normal sketch and of the five warped planes, cv2's 8-bit RGB/BGR -> Lab, ToTensor + Normalize(0.5, 0.5),
// concat with the Lab central crop into 21 channels.  Pointwise in the output pixel like k_pack_inputs.
// OpenCV's uint8 Lab is the integer pipeline below PLUS a sorted list of 1671 colours where its interpolated table deviates
// by one in a or b (scripts/make_lab_tables.py: verified against cv2 on all 2^24 colours).
// ---------------------------------------------------------------------------------------------------------------
struct LabTables { const uint16_t *gamma_tab, *cbrt_tab; const uint32_t *exc_keys; const uint16_t *exc_vals; int n_exc; const uint32_t *exc_bitmap; };

__device__ __forceinline__ void rgb2lab_u8(const LabTables &T, int r, int g, int b, int *lab) {
    const int R = __ldg(T.gamma_tab + r), G = __ldg(T.gamma_tab + g), B = __ldg(T.gamma_tab + b);
    const int fX = __ldg(T.cbrt_tab + ((R * 1777 + G * 1541 + B * 778 + 2048) >> 12));
    const int fY = __ldg(T.cbrt_tab + ((R * 871 + G * 2929 + B * 296 + 2048) >> 12));
    const int fZ = __ldg(T.cbrt_tab + ((R * 73 + G * 448 + B * 3575 + 2048) >> 12));
    lab[0] = min(max((296 * fY - 1336934 + 16384) >> 15, 0), 255);
    lab[1] = min(max((500 * (fX - fY) + (128 << 15) + 16384) >> 15, 0), 255);
    lab[2] = min(max((200 * (fY - fZ) + (128 << 15) + 16384) >> 15, 0), 255);
    const uint32_t key = ((uint32_t)r << 16) | ((uint32_t)g << 8) | (uint32_t)b;
    // one bit per colour (2 MB, L2 resident) says whether the colour is an exception at all: 1 in 10,000 pixels searches the list
    if (T.exc_bitmap && !((__ldg(T.exc_bitmap + (key >> 5)) >> (key & 31u)) & 1u)) return;
    int lo = 0, hi = T.n_exc;                           // first index with exc_keys[i] >= key
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(T.exc_keys + mid) < key) lo = mid + 1; else hi = mid;
    }
    if (lo < T.n_exc && __ldg(T.exc_keys + lo) == key) {
        const int v = __ldg(T.exc_vals + lo);
        lab[1] = v >> 8;
        lab[2] = v & 0xff;
    }
}

// pixel (cy, cx) of the square crop of an image that holds the frame rectangle (rx0, ry0, rw, rh) -- the whole frame, or a
// window of it -- zero outside it (the crop's padding, and for a window that covers the crop square clipped to the frame, only that)
__device__ __forceinline__ void crop_fetch3(const uint8_t *__restrict__ img, const CropGeom &g, int rx0, int ry0, int rw, int rh, int cy, int cx,
                                            int *v) {
    const int fy = g.ny0 + cy - g.pyb - ry0, fx = g.nx0 + cx - g.pxb - rx0;
    if (fy < 0 || fy >= rh || fx < 0 || fx >= rw) { v[0] = v[1] = v[2] = 0; return; }
    const uint8_t *p = img + ((size_t)fy * rw + fx) * 3;
    v[0] = p[0]; v[1] = p[1]; v[2] = p[2];
}

// WINDOW: the warped planes of item b are the window win[b] = (x0, y0, w, h) of the frame, five [h,w,3] planes at planes + win_off[b]
// (fusg_warp_fused_window's layout); otherwise planes is [B,5,Hf,Wf,3].
template <bool WINDOW>
__global__ void __launch_bounds__(256) k_pack_icn(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ normals,
                                                  const uint8_t *__restrict__ central, const int *__restrict__ bbox, LabTables T,
                                                  float *__restrict__ out, int Hf, int Wf, int res, const int32_t *__restrict__ win,
                                                  const long long *__restrict__ win_off) {
    const int b = blockIdx.z, q = blockIdx.y;            // q: 0 normal sketch, 1 central crop, 2..6 warped plane q-2
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= res * res) return;
    const size_t plane = (size_t)res * res;
    float *o = out + ((size_t)b * 21 + q * 3) * plane + p;
    if (WINDOW && (win[4 * b + 2] < 1 || win[4 * b + 3] < 1)) {     // no window (an item fusg_crop_geometry refused): a zero row
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) o[ch * plane] = 0.f;
        return;
    }
    const int oy = p / res, ox = p - oy * res;
    int v[3];
    if (q == 1) {
        const uint8_t *c = central + ((size_t)b * res * res + p) * 3;
        v[0] = c[0]; v[1] = c[1]; v[2] = c[2];
    } else {
        const uint8_t *img;
        int rx0 = 0, ry0 = 0, rw = Wf, rh = Hf;
        if (q == 0) img = normals + (size_t)b * Hf * Wf * 3;
        else if (!WINDOW) img = planes + ((size_t)b * 5 + (q - 2)) * Hf * Wf * 3;
        else {
            rx0 = win[4 * b]; ry0 = win[4 * b + 1]; rw = win[4 * b + 2]; rh = win[4 * b + 3];
            img = planes + win_off[b] + (size_t)(q - 2) * rh * rw * 3;
        }
        const CropGeom g = crop_geometry(bbox + 4 * b, Hf, Wf);
        if (g.cw == 2 * res && g.ch == 2 * res) {                              // exact halving -> 2x2 box average
            int a[3], bq[3], c[3], d[3];
            crop_fetch3(img, g, rx0, ry0, rw, rh, 2 * oy, 2 * ox, a); crop_fetch3(img, g, rx0, ry0, rw, rh, 2 * oy, 2 * ox + 1, bq);
            crop_fetch3(img, g, rx0, ry0, rw, rh, 2 * oy + 1, 2 * ox, c); crop_fetch3(img, g, rx0, ry0, rw, rh, 2 * oy + 1, 2 * ox + 1, d);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) v[ch] = (a[ch] + bq[ch] + c[ch] + d[ch] + 2) >> 2;
        } else {
            const Tap tx = resize_tap(res, g.cw, ox, true), ty = resize_tap(res, g.ch, oy, false);
            int p00[3], p01[3], p10[3], p11[3];
            crop_fetch3(img, g, rx0, ry0, rw, rh, ty.i0, tx.i0, p00); crop_fetch3(img, g, rx0, ry0, rw, rh, ty.i0, tx.i1, p01);
            crop_fetch3(img, g, rx0, ry0, rw, rh, ty.i1, tx.i0, p10); crop_fetch3(img, g, rx0, ry0, rw, rh, ty.i1, tx.i1, p11);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const int s0 = p00[ch] * tx.a0 + p01[ch] * tx.a1, s1 = p10[ch] * tx.a0 + p11[ch] * tx.a1;
                v[ch] = min(max((((ty.a0 * (s0 >> 4)) >> 16) + ((ty.a1 * (s1 >> 4)) >> 16) + 2) >> 2, 0), 255);
            }
        }
    }
    int lab[3];
    if (q >= 2) rgb2lab_u8(T, v[2], v[1], v[0], lab);    // planes are BGR (COLOR_BGR2LAB, planes_utils.py:88)
    else rgb2lab_u8(T, v[0], v[1], v[2], lab);           // sketches are RGB (COLOR_RGB2LAB, models.py:355,358)
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) o[ch * plane] = ((float)lab[ch] / 255.f - 0.5f) / 0.5f;
}

// ---------------------------------------------------------------------------------------------------------------
// to_image(x, from_LAB=True) (warp_learn/planes_utils.py:96-118), the ICN's output side: (x + 1) / 2 * 255, clip, truncating
// uint8 cast, then cv2.cvtColor(COLOR_LAB2BGR) on uint8 -- OpenCV's integer pipeline (Lab2RGBinteger), bit-exact on all 2^24
// (L, a, b) triples with the tables of data/lab8.npz (scripts/make_lab_tables.py).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int ab_to_xz(int i) {                 // OpenCV's abToXZ_b table as the integer formula it is filled with
    constexpr int BASE = 1 << 14;
    if (i <= 3390) return i * 108 / 841 - BASE * 16 / 116 * 108 / 841;          // C division: truncation toward zero
    return i * i / BASE * i / BASE;
}

__global__ void __launch_bounds__(256) k_to_image_lab(const float *__restrict__ in, uint8_t *__restrict__ out, const uint16_t *__restrict__ lab_to_yf,
                                                      const uint8_t *__restrict__ inv_gamma, int HW, size_t npix) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;      // over B*HW
    if (i >= npix) return;
    const size_t b = i / HW, pix = i - b * HW;
    int lab[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float v = (in[(b * 3 + c) * HW + pix] + 1.f) / 2.f * 255.f;      // numpy float32 arithmetic of to_image
        v = fminf(fmaxf(v, 0.f), 255.f);
        lab[c] = (int)v;                                                  // astype(np.uint8): truncation
    }
    constexpr int BASE = 1 << 14;
    const int y = __ldg(lab_to_yf + 2 * lab[0]), ify = __ldg(lab_to_yf + 2 * lab[0] + 1);
    const int adiv = ((5 * lab[1] * 53687 + (1 << 7)) >> 13) - 128 * BASE / 500;
    const int bdiv = ((lab[2] * 41943 + (1 << 4)) >> 9) - 128 * BASE / 200 + 1;
    const int x = ab_to_xz(ify + adiv), z = ab_to_xz(ify - bdiv);
    const int r = min(max((12615 * x - 6296 * y - 2223 * z + (1 << 13)) >> 14, 0), 4095);
    const int g = min(max((-3773 * x + 7684 * y + 185 * z + (1 << 13)) >> 14, 0), 4095);
    const int bl = min(max((217 * x - 836 * y + 4715 * z + (1 << 13)) >> 14, 0), 4095);
    uint8_t *o = out + i * 3;                                             // BGR
    o[0] = __ldg(inv_gamma + bl); o[1] = __ldg(inv_gamma + g); o[2] = __ldg(inv_gamma + r);
}

}  // namespace fusg

using namespace fusg;

extern "C" int fusg_u8_to_vunet_inputs(const uint8_t *mask_bbox, const uint8_t *normal_src, const uint8_t *normal_dst, float *x, float *y, int B,
                                       int res, void *stream) {
    if (!mask_bbox || !normal_src || !normal_dst || !x || !y || B <= 0 || res <= 0) return FUSG_ERR_ARG;
    if (B > 65535 || res > 4096) return FUSG_ERR_UNSUPPORTED;
    k_u8_to_inputs<<<dim3((res * res + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(mask_bbox, normal_src, normal_dst, x, y, res);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_u8_to_vunet_y(const uint8_t *normal_dst, float *y, int B, int res, void *stream) {
    if (!normal_dst || !y || B <= 0 || res <= 0) return FUSG_ERR_ARG;
    if (B > 65535 || res > 4096) return FUSG_ERR_UNSUPPORTED;
    k_u8_to_y<<<dim3((res * res + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(normal_dst, y, res);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" size_t fusg_sizeof_gather_seg(void) { return sizeof(fusg_gather_seg); }

extern "C" int fusg_gather_rows(const fusg_gather_seg *segs, int nseg, const int32_t *index, int B, void *stream) {
    if (!segs || nseg <= 0 || nseg > FUSG_GATHER_MAX_SEGS || !index || B <= 0) return FUSG_ERR_ARG;
    GatherTable tab = {};
    long long max16 = 0;
    for (int i = 0; i < nseg; ++i) {
        const fusg_gather_seg &sg = segs[i];
        if (!sg.src || !sg.dst || sg.n_src <= 0 || sg.row_bytes <= 0 || sg.row_bytes % 16 != 0) return FUSG_ERR_ARG;
        if ((reinterpret_cast<uintptr_t>(sg.src) | reinterpret_cast<uintptr_t>(sg.dst)) & 15) return FUSG_ERR_ARG;
        tab.s[i] = sg;
        max16 = sg.row_bytes / 16 > max16 ? sg.row_bytes / 16 : max16;
    }
    if (B > 65535) return FUSG_ERR_UNSUPPORTED;
    // a CTA moves at least 4 vectors per thread; rows of a few KB (the cached appearance tensors) take one CTA each
    long long split = (max16 + 4 * GATHER_THREADS - 1) / (4 * GATHER_THREADS);
    if (split > 1024) split = 1024;
    k_gather_rows<<<dim3(nseg, B, (unsigned)split), GATHER_THREADS, 0, (cudaStream_t)stream>>>(tab, index);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_mask_bbox(const uint8_t *masks, const long long *mask_off, const int32_t *mask_rect, int32_t *bbox, int B, int max_mask_pixels,
                              void *stream) {
    if (!masks || !mask_off || !mask_rect || !bbox || B <= 0 || max_mask_pixels <= 0) return FUSG_ERR_ARG;
    if (B > 65535) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    k_bbox_init<<<(B + 255) / 256, 256, 0, st>>>(bbox, B);      // rows start as (INT_MAX, INT_MAX, -1, -1): an empty mask stays that way
    int gx = (max_mask_pixels + 255) / 256;
    if (gx > 1024) gx = 1024;
    k_mask_bbox<<<dim3(gx, B), 256, 0, st>>>(masks, mask_off, mask_rect, bbox);
    fusg_count_launch(2);
    return fusg_check_launch();
}

extern "C" int fusg_crop_geometry(const int32_t *bbox, const int32_t *frame_index, int B, int Hf, int Wf, long long window_capacity_bytes,
                                  int max_win_h, int32_t *info, int32_t *win, long long *win_off, int8_t *status, void *stream) {
    if (!bbox || !info || !status || B <= 0 || Hf <= 0 || Wf <= 0 || window_capacity_bytes < 0) return FUSG_ERR_ARG;
    if (window_capacity_bytes > 0 && (!win || !win_off || max_win_h <= 0)) return FUSG_ERR_ARG;
    k_crop_geometry<<<1, GEOM_THREADS, 0, (cudaStream_t)stream>>>(bbox, frame_index, B, Hf, Wf, window_capacity_bytes, max_win_h, info, win,
                                                                win_off, status);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_pack_vunet_inputs(const uint8_t *frames, const int32_t *frame_idx, const uint8_t *masks, const uint8_t *normal_src,
                                      const uint8_t *normal_dst, const long long *off, const int32_t *rect, const int32_t *bbox, float *x,
                                      float *y, int B, int Hf, int Wf, int res, void *stream) {
    if (!frames || !frame_idx || !masks || !normal_src || !normal_dst || !off || !rect || !bbox || !x || !y) return FUSG_ERR_ARG;
    if (B <= 0 || Hf <= 0 || Wf <= 0 || res <= 0) return FUSG_ERR_ARG;
    if (B > 65535 || res > 4096) return FUSG_ERR_UNSUPPORTED;
    k_pack_inputs<<<dim3((res * res + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(frames, frame_idx, masks, normal_src, normal_dst, off, rect, bbox,
                                                                                      x, y, Hf, Wf, res);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_resize_u8(const uint8_t *src, const long long *src_off, const int32_t *src_hw, uint8_t *dst, const long long *dst_off,
                              const int32_t *dst_hw, int B, int max_dst_pixels, void *stream) {
    if (!src || !src_off || !src_hw || !dst || !dst_off || !dst_hw || B <= 0 || max_dst_pixels <= 0) return FUSG_ERR_ARG;
    if (B > 65535) return FUSG_ERR_UNSUPPORTED;
    int gx = (max_dst_pixels + 255) / 256;
    if (gx > 4096) gx = 4096;
    k_resize_u8<<<dim3(gx, B), 256, 0, (cudaStream_t)stream>>>(src, src_off, src_hw, dst, dst_off, dst_hw);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" size_t fusg_paste_workspace_bytes(int F, int Hf, int Wf) {
    return F <= 0 || Hf <= 0 || Wf <= 0 ? 0 : (size_t)F * Hf * Wf * sizeof(int);
}

extern "C" int fusg_paste_back(uint8_t *frames, const uint8_t *crops, const uint8_t *masks, const long long *mask_off, const int32_t *mask_rect,
                               const int32_t *info, void *workspace, size_t workspace_bytes, int B, int F, int Hf, int Wf, int S,
                               int max_mask_pixels, void *stream) {
    if (!frames || !crops || !masks || !mask_off || !mask_rect || !info || !workspace) return FUSG_ERR_ARG;
    if (B <= 0 || F <= 0 || Hf <= 0 || Wf <= 0 || S <= 0 || max_mask_pixels <= 0) return FUSG_ERR_ARG;
    if (B > 65535 || F > 65535) return FUSG_ERR_UNSUPPORTED;
    if (workspace_bytes < fusg_paste_workspace_bytes(F, Hf, Wf)) return FUSG_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    int *owner = reinterpret_cast<int *>(workspace);
    if (fusg_record_cuda(cudaMemsetAsync(owner, 0xFF, (size_t)F * Hf * Wf * sizeof(int), st)) != FUSG_OK) return FUSG_ERR_CUDA;
    int gx = (max_mask_pixels + 255) / 256;
    if (gx > 8192) gx = 8192;
    k_paste_owner<<<dim3(gx, B), 256, 0, st>>>(masks, mask_off, mask_rect, info, owner, F, Hf, Wf);
    int gf = (int)(((long long)Hf * Wf + 255) / 256);
    if (gf > 16384) gf = 16384;
    k_paste_apply<<<dim3(gf, F), 256, 0, st>>>(frames, crops, info, owner, Hf, Wf, S);
    fusg_count_launch(2);
    return fusg_check_launch();
}

// ================================================================================================
// Per-step keypoint kinematics of the trajectory loop (SURVEY.md section 8f-4): for item n = (vehicle, future step)
//   moved = v @ z_rot(theta) + tr            trajectory_inference.py:359-361 (z_rot is a float32 matrix, utils/geometry.py:80-113)
//   kp2d  = cv2.projectPoints(moved, rvec, tvec, K, 0)                        trajectory_inference.py:363-367
//   verts = np.int32((kp2d / (w,h)) * (w,h))      warp_learn/vehicle_utils.py:24-26, warp_learn/planes_utils.py:22-27
// i.e. exactly the kp3d / dst_kp inputs fusg_warp_fused_traj takes for that item.  Bit-exact restatement (oracle/
// kinematics_oracle.py): numpy's BLAS evaluates v @ M as the FMA chain fma(v2, M2c, fma(v1, M1c, v0*M0c)); projectPoints
// with zero distortion is R X + t left to right, z -> 1/z, x*fx + cx.  This file is compiled with -fmad=false, so only the
// explicit fma() calls fuse.
// ================================================================================================
__global__ void __launch_bounds__(128) k_step_keypoints(const double *__restrict__ kp3d, const int32_t *__restrict__ vehicle,
                                                        const float *__restrict__ rot, const double *__restrict__ tr, const double *__restrict__ R,
                                                        const double *__restrict__ t, const double *__restrict__ K, double *__restrict__ kp3d_out,
                                                        double *__restrict__ kp2d_out, int32_t *__restrict__ verts, int N, int H, int W) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;           // over N * 12
    if (i >= N * 12) return;
    const int n = i / 12, k = i - n * 12, v = vehicle[n];
    const double *p = kp3d + ((size_t)v * 12 + k) * 3;
    const float *M = rot + (size_t)n * 9;
    double m[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) m[c] = fma(p[2], (double)M[6 + c], fma(p[1], (double)M[3 + c], p[0] * (double)M[c])) + tr[(size_t)n * 3 + c];
    const double *Rv = R + (size_t)v * 9, *tv = t + (size_t)v * 3, *Kv = K + (size_t)v * 9;
    double x = Rv[0] * m[0] + Rv[1] * m[1] + Rv[2] * m[2] + tv[0];
    double y = Rv[3] * m[0] + Rv[4] * m[1] + Rv[5] * m[2] + tv[1];
    double z = Rv[6] * m[0] + Rv[7] * m[1] + Rv[8] * m[2] + tv[2];
    z = z != 0.0 ? 1. / z : 1.;
    x *= z;
    y *= z;
    const double u = x * Kv[0] + Kv[2], w = y * Kv[4] + Kv[5];
    kp3d_out[(size_t)i * 3] = m[0]; kp3d_out[(size_t)i * 3 + 1] = m[1]; kp3d_out[(size_t)i * 3 + 2] = m[2];
    kp2d_out[(size_t)i * 2] = u; kp2d_out[(size_t)i * 2 + 1] = w;
    // normalise by the frame size, scale back, truncate (far-out values are clamped; the warp stage rejects them anyway)
    double px = (u / (double)W) * (double)W, py = (w / (double)H) * (double)H;
    px = fmin(fmax(px, -1.0e9), 1.0e9);
    py = fmin(fmax(py, -1.0e9), 1.0e9);
    verts[(size_t)i * 2] = (int)px;
    verts[(size_t)i * 2 + 1] = (int)py;
}

extern "C" int fusg_step_keypoints(const double *kp3d, const int32_t *vehicle, const float *rot, const double *tr, const double *R,
                                   const double *t, const double *K, double *kp3d_out, double *kp2d_out, int32_t *verts, int N, int H, int W,
                                   void *stream) {
    if (!kp3d || !vehicle || !rot || !tr || !R || !t || !K || !kp3d_out || !kp2d_out || !verts || N <= 0 || H <= 0 || W <= 0) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    k_step_keypoints<<<(N * 12 + 127) / 128, 128, 0, st>>>(kp3d, vehicle, rot, tr, R, t, K, kp3d_out, kp2d_out, verts, N, H, W);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_pack_icn_inputs(const uint8_t *planes, const uint8_t *normals, const uint8_t *central, const int32_t *bbox,
                                    const uint16_t *gamma_tab, const uint16_t *cbrt_tab, const uint32_t *exc_keys, const uint16_t *exc_vals, int n_exc,
                                    const uint32_t *exc_bitmap, float *out, int B, int Hf, int Wf, int res, void *stream) {
    if (!planes || !normals || !central || !bbox || !gamma_tab || !cbrt_tab || !out || B <= 0 || Hf <= 0 || Wf <= 0 || res <= 0 || n_exc < 0) return FUSG_ERR_ARG;
    if (n_exc > 0 && (!exc_keys || !exc_vals)) return FUSG_ERR_ARG;
    if (B > 65535) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    LabTables T{gamma_tab, cbrt_tab, exc_keys, exc_vals, n_exc, exc_bitmap};
    k_pack_icn<false><<<dim3((res * res + 255) / 256, 7, B), 256, 0, st>>>(planes, normals, central, bbox, T, out, Hf, Wf, res, nullptr, nullptr);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_pack_icn_inputs_window(const uint8_t *planes, const int32_t *win, const long long *win_off, const uint8_t *normals,
                                           const uint8_t *central, const int32_t *bbox, const uint16_t *gamma_tab, const uint16_t *cbrt_tab,
                                           const uint32_t *exc_keys, const uint16_t *exc_vals, int n_exc, const uint32_t *exc_bitmap, float *out,
                                           int B, int Hf, int Wf, int res, void *stream) {
    if (!planes || !win || !win_off || !normals || !central || !bbox || !gamma_tab || !cbrt_tab || !out) return FUSG_ERR_ARG;
    if (B <= 0 || Hf <= 0 || Wf <= 0 || res <= 0 || n_exc < 0) return FUSG_ERR_ARG;
    if (n_exc > 0 && (!exc_keys || !exc_vals)) return FUSG_ERR_ARG;
    if (B > 65535) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    LabTables T{gamma_tab, cbrt_tab, exc_keys, exc_vals, n_exc, exc_bitmap};
    k_pack_icn<true><<<dim3((res * res + 255) / 256, 7, B), 256, 0, st>>>(planes, normals, central, bbox, T, out, Hf, Wf, res, win, win_off);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_to_image_lab(const float *in, uint8_t *out, const uint16_t *lab_to_yf, const uint8_t *inv_gamma, int B, int H, int W, void *stream) {
    if (!in || !out || !lab_to_yf || !inv_gamma || B <= 0 || H <= 0 || W <= 0) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t npix = (size_t)B * H * W;
    k_to_image_lab<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(in, out, lab_to_yf, inv_gamma, H * W, npix);
    fusg_count_launch(1);
    return fusg_check_launch();
}
