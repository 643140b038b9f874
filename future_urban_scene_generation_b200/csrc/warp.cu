// warp.cu -- fused planar-warp stage for sm_100a: visibility, per-plane homographies and the
// masked fixed-point bilinear gather, behind the C ABI of include/fusg.h.
//
// Reference path (file:line in the reference repo): trajectory_inference.py:165-174 =
//   compute_visibility (warp_learn/online_visibility.py:105-150) for both poses,
//   get_planes        (warp_learn/planes_utils.py:11-37),
//   warp_unwarp_planes(warp_learn/planes_utils.py:40-82), first return value.
//
// Three launches per batch, one C call:
//   k_visibility   one CTA per (crop, pose): polygon scanline coverage as 32-pixel bit words,
//                  painter's-order occlusion, area ratio test -> 7 flags.
//   k_homography   one warp per (crop, plane): gating, DLT (OpenCV Jacobi) + LM, inverse map.
//   k_warp         one CTA per crop: source crop staged in shared memory by TMA bulk copies,
//                  per-plane polygon bit mask in shared memory, per-row conservative active
//                  span, cv2-exact 1/32-px fixed-point bilinear gather, rows written back with
//                  128-bit coalesced stores.  HBM traffic = read crop once + write 5 planes.
//
// Compiled with -fmad=false (see warp_geom.cuh).
#include <cuda_runtime.h>
#include <climits>
#include <cstdlib>
#include <cstdint>
#include <cstdio>
#include "../../include/fusg.h"
#include "fusg_common.h"
#include "warp_geom.cuh"
#include "warp_solver.cuh"

namespace fusg {

// ============================================================================================
// k_visibility
// ============================================================================================
struct VisShared {
    int vx[N_KP], vy[N_KP];
    double dist[N_VIS];
    PolyEdge edge[32];            // the 6 + 6 + 5 x 4 = 32 edges of the seven polygons, polygon after polygon
};
// first edge record of polygon p
__device__ __forceinline__ int vis_edge_base(int p) { return p < 2 ? 6 * p : 12 + 4 * (p - 2); }

constexpr int VIS_WARPS = 4;     // poses per CTA (one warp each; no block-level barriers)

// grid.x = ceil(poses / VIS_WARPS).  Pose g reads K[b], kp3d[b], and E0/E1[b] (fused src/dst layout, b = g/2)
// when E1 != nullptr, else K[g], E0[g], kp3d[g].  kp3d1 (fused layout only, may be NULL): the destination pose's own
// keypoints -- the trajectory loop moves the CAD keypoints instead of the camera (trajectory_inference.py:359-376).
__global__ void __launch_bounds__(VIS_WARPS * 32) k_visibility(const double *__restrict__ K, const double *__restrict__ E0,
                                                               const double *__restrict__ E1, const double *__restrict__ kp3d,
                                                               const double *__restrict__ kp3d1, uint8_t *__restrict__ vis, int32_t *__restrict__ pts,
                                                               int32_t *__restrict__ areas, int n_poses, int H, int W) {
    __shared__ VisShared sm_all[VIS_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * VIS_WARPS + warp;
    if (g >= n_poses) return;
    VisShared &sm = sm_all[warp];
    const double *Kp, *Ep, *Xp;
    if (E1) {
        const int b = g >> 1;
        Kp = K + 9 * b; Xp = (((g & 1) && kp3d1) ? kp3d1 : kp3d) + 36 * b;
        Ep = ((g & 1) ? E1 : E0) + 12 * b;
    } else {
        Kp = K + 9 * g; Xp = kp3d + 36 * g; Ep = E0 + 12 * g;
    }
    // 12 projections (lanes 0..11) and 7 plane distances (lanes 12..18)
    if (lane < N_KP) {
        double u, v;
        project_point(Kp, Ep, Xp + 3 * lane, &u, &v);
        // int(): truncation toward zero; far-out values are clamped (and refused below: POLY_COORD_MAX)
        u = fmin(fmax(u, -1.0e9), 1.0e9);
        v = fmin(fmax(v, -1.0e9), 1.0e9);
        sm.vx[lane] = (int)u;
        sm.vy[lane] = (int)v;
    } else if (lane < N_KP + N_VIS) {
        sm.dist[lane - N_KP] = plane_distance(Ep, Xp, lane - N_KP);
    }
    __syncwarp();
    // Vertices outside the frame are fine (cv2.fillPoly clips, poly_row_ranges follows it); only absurd
    // magnitudes (a keypoint on the camera plane) are refused.
    bool oob = false;
    if (lane < N_KP) oob = abs(sm.vx[lane]) > POLY_COORD_MAX || abs(sm.vy[lane]) > POLY_COORD_MAX;
    oob = __any_sync(0xffffffffu, oob);
    int cnt_abs[N_VIS], cnt_occ[N_VIS];
#pragma unroll
    for (int p = 0; p < N_VIS; ++p) cnt_abs[p] = cnt_occ[p] = 0;
    if (!oob) {
        // occluder sets: planes strictly nearer to the camera
        unsigned nearer[N_VIS];
#pragma unroll
        for (int p = 0; p < N_VIS; ++p) {
            unsigned mk = 0;
#pragma unroll
            for (int q = 0; q < N_VIS; ++q)
                if (sm.dist[q] < sm.dist[p]) mk |= 1u << q;
            nearer[p] = mk;
        }
        // every polygon lies inside the bounding box of the 12 projected keypoints
        int bx0 = sm.vx[0], bx1 = sm.vx[0], by0 = sm.vy[0], by1 = sm.vy[0];
        for (int k = 1; k < N_KP; ++k) {
            bx0 = min(bx0, sm.vx[k]); bx1 = max(bx1, sm.vx[k]);
            by0 = min(by0, sm.vy[k]); by1 = max(by1, sm.vy[k]);
        }
        bx0 = max(bx0, 0); bx1 = min(bx1, W - 1);
        by0 = max(by0, 0); by1 = min(by1, H - 1);
        const int w0 = bx0 >> 5, w1 = bx1 >> 5;
        // row-independent part of the 32 polygon edges, one lane each (edge i of a polygon runs from vertex i-1 to vertex i)
        {
            const int p = lane < 12 ? lane / 6 : 2 + (lane - 12) / 4;
            const int i = lane - vis_edge_base(p), n = c_plane_n[p];
            const int ka = c_plane_kp[p][i == 0 ? n - 1 : i - 1], kb = c_plane_kp[p][i];
            PolyEdge e;
            poly_edge_setup(sm.vx[ka], sm.vy[ka], sm.vx[kb], sm.vy[kb], H, W, e);
            sm.edge[lane] = e;
        }
        __syncwarp();
        for (int y = by0 + lane; y <= by1; y += 32) {
            int lo[N_VIS][MAX_RANGES], hi[N_VIS][MAX_RANGES], rc[N_VIS];
#pragma unroll 1
            for (int p = 0; p < N_VIS; ++p) rc[p] = poly_row_ranges_edges(sm.edge + vis_edge_base(p), c_plane_n[p], y, W, lo[p], hi[p]);
            for (int w = w0; w <= w1; ++w) {
                unsigned bits[N_VIS];
#pragma unroll
                for (int p = 0; p < N_VIS; ++p) bits[p] = ranges_word(lo[p], hi[p], rc[p], w);
#pragma unroll
                for (int p = 0; p < N_VIS; ++p) {
                    unsigned occl = 0;
#pragma unroll
                    for (int q = 0; q < N_VIS; ++q)
                        if ((nearer[p] >> q) & 1u) occl |= bits[q];
                    cnt_abs[p] += __popc(bits[p]);
                    cnt_occ[p] += __popc(bits[p] & ~occl);
                }
            }
        }
#pragma unroll
        for (int p = 0; p < N_VIS; ++p) {
            for (int off = 16; off > 0; off >>= 1) {
                cnt_abs[p] += __shfl_xor_sync(0xffffffffu, cnt_abs[p], off);
                cnt_occ[p] += __shfl_xor_sync(0xffffffffu, cnt_occ[p], off);
            }
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int p = 0; p < N_VIS; ++p) {
            vis[N_VIS * g + p] = oob ? 0xff : ((double)cnt_occ[p] > 0.9 * (double)cnt_abs[p] ? 1 : 0);   // 0xff: refused (see above)
            if (areas) { areas[2 * N_VIS * g + 2 * p] = oob ? -1 : cnt_abs[p]; areas[2 * N_VIS * g + 2 * p + 1] = oob ? -1 : cnt_occ[p]; }
        }
    }
    if (pts && lane < N_KP) { pts[(N_KP * g + lane) * 2] = sm.vx[lane]; pts[(N_KP * g + lane) * 2 + 1] = sm.vy[lane]; }
}

// ============================================================================================
// Homographies: k_plane_gate applies the gating / symmetry remap of planes_utils.py:57-68 and appends the
// surviving (crop, plane) tasks to a 6-point list (left / right, LM-refined: ~10 Jacobi runs) or a 4-point
// list (one Jacobi run); skipped planes get their outputs written there.  k_solve then runs the thread-per-
// point-set solver of warp_solver.cuh over the lists, `lanes` tasks per warp (1 for small batches: the
// latency of one solve; 32 for large ones: throughput), 6-point and 4-point tasks in separate warps so that the
// lanes of a warp run jobs of the same length.  Outputs are indexed by task id, so the (non-deterministic)
// list order does not affect results.
// workspace layout per crop: Minv[5][9] f64 (inverse maps indexed by SOURCE plane i)
// ============================================================================================
// What the gather needs to bound the destination region of a solved (crop, source plane): the forward image of the source
// polygon under H12 and how far a 2-px source step can move in the destination.  Written by k_solve, whose lane holds the
// point set and H12 in registers anyway (in the gather this was a serial section of one thread per plane).
struct PlaneRec {
    float fwdx[6], fwdy[6];       // destination pixels of the source polygon's vertices
    float pad;                    // 1.5 * sqrt(2) * (reach of a 2-px source step, worst vertex) + 1
    int ok;                       // 0: horizon through the polygon / absurd magnification -> bbox spans only
};

// Output window (x0, y0, w, h) of an item of fusg_warp_fused_window: non-empty, inside the H x W frame, at most max_h rows.
__device__ __forceinline__ bool window_ok(const int32_t *win, int max_h, int H, int W) {
    const int x0 = win[0], y0 = win[1], w = win[2], h = win[3];
    return x0 >= 0 && y0 >= 0 && w >= 1 && h >= 1 && h <= max_h && x0 <= W - w && y0 <= H - h;
}

// WINDOW: the items also carry an output window (win [B,4]); an item whose window is not window_ok is refused.
template <bool WINDOW>
__global__ void __launch_bounds__(256) k_plane_gate(const int32_t *__restrict__ src_kp, const int32_t *__restrict__ dst_kp,
                                                    const uint8_t *__restrict__ vis, int8_t *__restrict__ plane_j, double *__restrict__ H12,
                                                    double *__restrict__ Minv, int *__restrict__ counters, int *__restrict__ list6,
                                                    int *__restrict__ list4, const int32_t *__restrict__ src_index, int n_src,
                                                    const int32_t *__restrict__ win, int max_win_h, int B, int H, int W) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * N_TEX) return;
    const int b = t / N_TEX, i = t % N_TEX;
    const uint8_t *sv = vis + 2 * N_VIS * b, *dv = sv + N_VIS;
    bool bad = sv[0] == 0xff || dv[0] == 0xff;
    if (src_index && (src_index[b] < 0 || src_index[b] >= n_src)) bad = true;     // no source image: refused like an absurd vertex
    if (WINDOW && !window_ok(win + 4 * b, max_win_h, H, W)) bad = true;
    const int32_t *sk = src_kp + 2 * N_KP * b, *dk = dst_kp + 2 * N_KP * b;
    for (int k = 0; k < 2 * N_KP && !bad; ++k)
        if (abs(sk[k]) > POLY_COORD_MAX || abs(dk[k]) > POLY_COORD_MAX) bad = true;
    const int j = bad ? -2 : plane_target(i, sv, dv);
    plane_j[t] = (int8_t)j;
    if (j >= 0) {
        if (i < 2) list6[atomicAdd(&counters[0], 1)] = t;
        else list4[atomicAdd(&counters[1], 1)] = t;
    } else {
        for (int k = 0; k < 9; ++k) Minv[9 * t + k] = 0;
        if (H12) for (int k = 0; k < 9; ++k) H12[9 * t + k] = 0;
    }
}

// grid = blocks6 + blocks4 one-warp blocks; block b < blocks6 serves 6-point tasks [b*lanes, (b+1)*lanes)
__global__ void __launch_bounds__(32) k_solve(const int32_t *__restrict__ src_kp, const int32_t *__restrict__ dst_kp,
                                              int8_t *__restrict__ plane_j, double *__restrict__ H12, double *__restrict__ Minv,
                                              const int *__restrict__ counters, const int *__restrict__ list6,
                                              const int *__restrict__ list4, PlaneRec *__restrict__ recs, int blocks6, int lanes) {
    extern __shared__ double solver_smem[];
    const int lane = threadIdx.x;
    const bool six = (int)blockIdx.x < blocks6;
    const int blk = six ? blockIdx.x : blockIdx.x - blocks6;
    const int count = six ? counters[0] : counters[1];
    if (blk * lanes >= count) return;                       // whole warp without work
    const int idx = blk * lanes + lane;
    const bool has = lane < lanes && idx < count;
    PointSet ps;
    ps.count = 0;
    int t = 0;
    if (has) {
        t = six ? list6[idx] : list4[idx];
        const int b = t / N_TEX, i = t % N_TEX, j = plane_j[t];
        const int32_t *sk = src_kp + 2 * N_KP * b, *dk = dst_kp + 2 * N_KP * b;
        ps.count = c_plane_n[i];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            if (k < ps.count) {
                ps.Mx[k] = (float)sk[2 * c_plane_kp[i][k]]; ps.My[k] = (float)sk[2 * c_plane_kp[i][k] + 1];
                ps.mx[k] = (float)dk[2 * c_plane_kp[j][k]]; ps.my[k] = (float)dk[2 * c_plane_kp[j][k] + 1];
            }
        }
    }
    double Hm[9], Mi[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) Hm[k] = Mi[k] = 0;
    // H21 is only ever used through its "is None" test, the same (symmetric) degeneracy test as H12's -- planes_utils.py:72-74
    const bool good = sv_find_homography(LaneMem{solver_smem + lane}, ps, Hm);
    if (!has) return;
    if (good) invert3(Hm, Mi);
    else plane_j[t] = -1;
#pragma unroll
    for (int k = 0; k < 9; ++k) Minv[9 * t + k] = Mi[k];
    if (H12) {
#pragma unroll
        for (int k = 0; k < 9; ++k) H12[9 * t + k] = good ? Hm[k] : 0.0;
    }
    if (recs && good) {
        // forward image of the vertices and of 2-px steps away from them (any accuracy better than a pixel will do)
        // (the vertices are re-read from global memory: a run-time index into ps.Mx / ps.My would move the point set of the
        // whole solve from registers to local memory)
        PlaneRec &r = recs[t];
        int ok = 1;
        double reach = 0;
        const int pi = t % N_TEX, pn = c_plane_n[pi];
        const int32_t *pk = src_kp + 2 * N_KP * (t / N_TEX);
        const double w0 = Hm[6] * (double)pk[2 * c_plane_kp[pi][0]] + Hm[7] * (double)pk[2 * c_plane_kp[pi][0] + 1] + Hm[8];
#pragma unroll 1
        for (int k = 0; k < pn; ++k) {
            const double vx = (double)pk[2 * c_plane_kp[pi][k]], vy = (double)pk[2 * c_plane_kp[pi][k] + 1];
            const double wv = Hm[6] * vx + Hm[7] * vy + Hm[8];
            const double px = (Hm[0] * vx + Hm[1] * vy + Hm[2]) / wv, py = (Hm[3] * vx + Hm[4] * vy + Hm[5]) / wv;
            if (!(fabs(px) < 1e6) || !(fabs(py) < 1e6)) ok = 0;
            if (!(wv * w0 > 0)) ok = 0;                     // the projective denominator must keep its sign over the polygon
            r.fwdx[k] = (float)px; r.fwdy[k] = (float)py;
#pragma unroll 1
            for (int d = 0; d < 4; ++d) {                   // where does a 2-px step away from the vertex land?
                const double ux = vx + (d == 0 ? 2. : d == 1 ? -2. : 0.), uy = vy + (d == 2 ? 2. : d == 3 ? -2. : 0.);
                const double wu = Hm[6] * ux + Hm[7] * uy + Hm[8];
                if (!(wu * wv > 0)) { ok = 0; continue; }
                const double qx = (Hm[0] * ux + Hm[1] * uy + Hm[2]) / wu, qy = (Hm[3] * ux + Hm[4] * uy + Hm[5]) / wu;
                reach = fmax(reach, fmax(fabs(qx - px), fabs(qy - py)));
            }
        }
        if (!(reach < 64.)) ok = 0;                         // absurd magnification: keep the bbox spans
        r.pad = (float)(1.5 * 1.4143 * reach + 1.0);        // diagonal source steps, then slack
        r.ok = ok;
    }
}

// cv2.findHomography drop-in on N explicit point sets of n points each
__global__ void __launch_bounds__(32) k_find_homography(const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int n,
                                                        double *__restrict__ H, uint8_t *__restrict__ ok, int N, int lanes) {
    extern __shared__ double solver_smem[];
    const int lane = threadIdx.x;
    const int t = blockIdx.x * lanes + lane;
    const bool has = lane < lanes && t < N;
    PointSet ps;
    ps.count = 0;
    if (has) {
        ps.count = n;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            if (k < n) {
                ps.Mx[k] = (float)src[(t * n + k) * 2]; ps.My[k] = (float)src[(t * n + k) * 2 + 1];
                ps.mx[k] = (float)dst[(t * n + k) * 2]; ps.my[k] = (float)dst[(t * n + k) * 2 + 1];
            }
        }
    }
    double Hm[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) Hm[k] = 0;
    const bool good = sv_find_homography(LaneMem{solver_smem + lane}, ps, Hm);
    if (!has) return;
#pragma unroll
    for (int k = 0; k < 9; ++k) H[9 * t + k] = good ? Hm[k] : 0.0;
    ok[t] = good ? 1 : 0;
}

// ============================================================================================
// The gather: cv2.warpPerspective INTER_LINEAR / BORDER_CONSTANT(0) for one destination pixel.
// M is the inverse map; (bx,y) the start of OpenCV's 64-wide processing block containing x.
// ============================================================================================
struct RowBase { double X0, Y0, W0; };

__device__ __forceinline__ RowBase row_base(const double *M, int bx, int y) {
    RowBase r;
    r.X0 = M[0] * bx + M[1] * y + M[2];
    r.Y0 = M[3] * bx + M[4] * y + M[5];
    r.W0 = M[6] * bx + M[7] * y + M[8];
    return r;
}

__device__ __forceinline__ void src_coord(const double *M, const RowBase &rb, int x1, int &X, int &Y) {
    double Wv = rb.W0 + M[6] * x1;
    Wv = Wv ? 32. / Wv : 0;
    const double fX = fmax((double)INT_MIN, fmin((double)INT_MAX, (rb.X0 + M[0] * x1) * Wv));
    const double fY = fmax((double)INT_MIN, fmin((double)INT_MAX, (rb.Y0 + M[3] * x1) * Wv));
    X = __double2int_rn(fX);      // cvRound: round half to even
    Y = __double2int_rn(fY);
}

// OpenCV's block width for warpPerspective (BLOCK_SZ = 32)
__host__ __device__ inline int warp_block_w(int H, int W) {
    const int bh0 = 16 < H ? 16 : H;
    const int bw0 = 32 * 32 / bh0;
    return bw0 < W ? bw0 : W;
}

// `src` / `mask` may be row WINDOWS: they are addressed with absolute row numbers (the caller passes pointers already
// offset by -ylo rows) and only rows ylo..yhi exist; a tap outside them is a tap outside the plane's polygon, i.e. zero.
template <bool MASKED, typename SrcPtr>
__device__ __forceinline__ uchar3 bilinear_tap4(SrcPtr src, const uint32_t *mask, int mask_words, int ylo, int yhi, int W, int X, int Y) {
    int sx = X >> 5, sy = Y >> 5;
    const int a = X & 31, b = Y & 31;
    sx = max(-32768, min(32767, sx));
    sy = max(-32768, min(32767, sy));
    const int w00 = (32 - a) * (32 - b) * 32, w01 = a * (32 - b) * 32, w10 = (32 - a) * b * 32, w11 = a * b * 32;
    const bool xin0 = (unsigned)sx < (unsigned)W, xin1 = (unsigned)(sx + 1) < (unsigned)W;
    const bool yin0 = sy >= ylo && sy <= yhi, yin1 = sy + 1 >= ylo && sy + 1 <= yhi;
    bool t00 = xin0 && yin0, t01 = xin1 && yin0, t10 = xin0 && yin1, t11 = xin1 && yin1;
    if (MASKED) {
        if (t00) t00 = (mask[sy * mask_words + (sx >> 5)] >> (sx & 31)) & 1u;
        if (t01) t01 = (mask[sy * mask_words + ((sx + 1) >> 5)] >> ((sx + 1) & 31)) & 1u;
        if (t10) t10 = (mask[(sy + 1) * mask_words + (sx >> 5)] >> (sx & 31)) & 1u;
        if (t11) t11 = (mask[(sy + 1) * mask_words + ((sx + 1) >> 5)] >> ((sx + 1) & 31)) & 1u;
    }
    int acc0 = 1 << 14, acc1 = 1 << 14, acc2 = 1 << 14;
    if (t00) { const auto *p = src + (sy * W + sx) * 3;           acc0 += p[0] * w00; acc1 += p[1] * w00; acc2 += p[2] * w00; }
    if (t01) { const auto *p = src + (sy * W + sx + 1) * 3;       acc0 += p[0] * w01; acc1 += p[1] * w01; acc2 += p[2] * w01; }
    if (t10) { const auto *p = src + ((sy + 1) * W + sx) * 3;     acc0 += p[0] * w10; acc1 += p[1] * w10; acc2 += p[2] * w10; }
    if (t11) { const auto *p = src + ((sy + 1) * W + sx + 1) * 3; acc0 += p[0] * w11; acc1 += p[1] * w11; acc2 += p[2] * w11; }
    return make_uchar3((unsigned char)(acc0 >> 15), (unsigned char)(acc1 >> 15), (unsigned char)(acc2 >> 15));
}

// ============================================================================================
// The gather stage for crops up to 256 x 256.
//
// 97 % of the 5 output planes of a crop is zero: a written plane is non-zero only inside the destination polygon, and
// ~3 of the 5 planes have no writer at all.  So the bytes are written by the TMA engine -- bulk stores from a block of
// zeros in shared memory, issued by k_warp_rows two crops ahead of its gather, so that the HBM write stream runs underneath
// the per-pixel arithmetic -- and the gather itself only visits the rows of each written plane
// whose active span is not empty: it stages just the source rows the crop's polygons cover (TMA bulk copy of one
// contiguous row range into a WIN-row window of shared memory), builds the polygon bit masks of those rows, gathers
// with cv2's 1/32-px fixed-point bilinear rule and overwrites the rows with 16-byte coalesced stores.
// Crops whose polygons span more than WIN source rows are queued for a second launch with a full-height window.
// ============================================================================================
constexpr int WARP_THREADS = 512;
constexpr int WARP_NWARPS = WARP_THREADS / 32;
constexpr int MAX_HW = 256;
constexpr int ROW_BYTES_MAX = MAX_HW * 3;          // 768
constexpr int MASK_WORDS = MAX_HW / 32;            // 8 words per row
constexpr int WIN_SMALL = 120;                     // source rows of the common-case window (2 CTAs per SM)

struct WarpSmemHeader {
    unsigned long long mbar;
    unsigned wait_start, pad0;                     // kernel start time; must directly follow mbar (mbar_wait)
    double Minv[N_TEX][9];
    int sel[N_TEX];                                // source plane feeding output plane j, or -1
    int polyx[6], polyy[6], polyn;
    unsigned row_bits[MAX_HW / 32];                // output rows of the current plane with a non-empty span (bit r of word w: row 32w + r)
    PolyEdge edge[6];                              // row-independent part of the source polygon's edges (poly_edge_setup)
    float fwdx[6], fwdy[6];                        // forward image of the source polygon under H12 (destination pixels)
    int fwd_ok;                                    // 0: a vertex is on / behind the horizon of H12 -> bbox spans only
    float fwd_pad;                                 // how far (destination px) a 2-px step in the source can move, worst vertex, with slack
    int bbox[4];                                   // xmin,xmax,ymin,ymax of the source polygon
    int win_lo, win_hi;                            // source rows held in the window (absolute row numbers)
    int skip;                                      // this crop does not fit the window: queued for the big-window launch
    short span_lo[MAX_HW], span_hi[MAX_HW];        // conservative active span per output row
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t phase) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
        if (!done) fusg_wait_failed(smem_u32(bar) + 8);      // WarpSmemHeader::wait_start follows mbar
    }
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// shared -> global bulk copy (TMA), tracked by the issuing thread's bulk async-groups
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all but the `pending` most recent groups of this thread have completed, writes included
__device__ __forceinline__ void bulk_wait(int pending) {
    switch (pending) {
        case 0: asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); break;
        case 1: asm volatile("cp.async.bulk.wait_group 1;" ::: "memory"); break;
        case 2: asm volatile("cp.async.bulk.wait_group 2;" ::: "memory"); break;
        case 3: asm volatile("cp.async.bulk.wait_group 3;" ::: "memory"); break;
        default: asm volatile("cp.async.bulk.wait_group 4;" ::: "memory"); break;
    }
}
constexpr int ZERO_BYTES = 4096;
constexpr int ZERO_PER_ROW = 1;        // blocks a filler lane issues after each row its warp gathers
constexpr int ZERO_AHEAD = 2;          // crops the fill runs ahead of the gather (per CTA)
// bulk zero fill of `bytes` (a multiple of 16) at `dst` (16-byte aligned): one bulk async-group of the calling thread,
// which takes every nsh-th block (share `sh`)
__device__ __forceinline__ void zero_crop(uint8_t *dst, const uint8_t *s_zero, size_t bytes, int sh, int nsh) {
    for (size_t off = (size_t)sh * ZERO_BYTES; off < bytes; off += (size_t)nsh * ZERO_BYTES)
        bulk_s2g(dst + off, s_zero, (uint32_t)(bytes - off < (size_t)ZERO_BYTES ? bytes - off : (size_t)ZERO_BYTES));
    bulk_commit();
}

// conservative x-span of output row y whose source footprint can touch the polygon bbox
__device__ __forceinline__ void row_active_span(const double *M, int y, int W, const int *bbox, int &xlo, int &xhi) {
    // u = (M0 x + cu) / (M6 x + cd), v = (M3 x + cv) / (M6 x + cd);  need u in [ulo,uhi], v in [vlo,vhi]
    const double cu = M[1] * y + M[2], cv = M[4] * y + M[5], cd = M[7] * y + M[8];
    const double d0 = cd, d1 = M[6] * (W - 1) + cd;
    xlo = 0; xhi = W - 1;
    if (!(d0 > 0 && d1 > 0) && !(d0 < 0 && d1 < 0)) return;         // sign change / zero / NaN: keep full row
    const double sgn = d0 > 0 ? 1.0 : -1.0;
    const double ulo = bbox[0] - 2.0, uhi = bbox[1] + 2.0, vlo = bbox[2] - 2.0, vhi = bbox[3] + 2.0;
    double l = 0.0, h = (double)(W - 1);
    // each constraint: sgn * (a x + c) >= 0
    const double ca[4] = {sgn * (M[0] - ulo * M[6]), -sgn * (M[0] - uhi * M[6]), sgn * (M[3] - vlo * M[6]), -sgn * (M[3] - vhi * M[6])};
    const double cc[4] = {sgn * (cu - ulo * cd), -sgn * (cu - uhi * cd), sgn * (cv - vlo * cd), -sgn * (cv - vhi * cd)};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double a = ca[k], c = cc[k];
        if (!(a == a) || !(c == c)) return;                        // NaN: full row
        if (fabs(a) < 1e-300) {
            if (c < 0) { l = 1; h = 0; }                            // infeasible (up to rounding: c<0 strictly)
        } else {
            const double r = -c / a;
            if (!(fabs(r) < 1e15)) { if (a > 0 ? r > 0 : r < 0) { l = 1; h = 0; } continue; }
            if (a > 0) l = fmax(l, r - 1.5); else h = fmin(h, r + 1.5);
        }
    }
    if (l > h) { xlo = 1; xhi = 0; return; }
    xlo = max(0, (int)floor(l) - 1);
    xhi = min(W - 1, (int)ceil(h) + 1);
}

// Row span of the destination region: every non-zero pixel of warped[j] has a bilinear tap inside the source polygon, so it
// has a source point within 2 px of that polygon (mask outline + tap footprint + 1/32-px rounding).  With P' the forward
// image of the polygon under H12 and PAD the distance a 2-px source step can move in the destination (measured at the
// vertices, where the projective magnification ~ 1/w^2 of a polygon peaks, times 1.5, plus 1), the pixel lies within PAD of
// P'.  For output row y the span is the x-range of the parts of the boundary of P' (a closed polyline through
// fwd[0..n-1]) inside the band [y - PAD, y + PAD], widened by PAD -- the boundary of a closed polygon crosses every row
// that P' reaches, so the range between its extreme crossings covers the interior too.  fp32 is ample for a bound.
__device__ __forceinline__ void row_polygon_span(const float *fx, const float *fy, int n, float PAD, int y, int W, int &xlo, int &xhi) {
    const float y0 = (float)y - PAD, y1 = (float)y + PAD;
    float lo = 1e30f, hi = -1e30f;
    float ax = fx[n - 1], ay = fy[n - 1];
    for (int k = 0; k < n; ++k) {
        const float bx = fx[k], by = fy[k];
        const float emin = fminf(ay, by), emax = fmaxf(ay, by);
        if (emax >= y0 && emin <= y1) {
            // clip the edge to the band and take the x-range of the clipped piece
            float t0 = 0.f, t1 = 1.f;
            const float dy = by - ay;
            if (fabsf(dy) > 1e-6f) {
                const float ta = (y0 - ay) / dy, tb = (y1 - ay) / dy;
                t0 = fmaxf(t0, fminf(ta, tb)); t1 = fminf(t1, fmaxf(ta, tb));
            }
            if (t0 <= t1) {
                const float xa = ax + (bx - ax) * t0, xb = ax + (bx - ax) * t1;
                lo = fminf(lo, fminf(xa, xb)); hi = fmaxf(hi, fmaxf(xa, xb));
            }
        }
        ax = bx; ay = by;
    }
    if (lo > hi) { xlo = 1; xhi = 0; return; }     // no boundary in the band: the row is outside P' (+ PAD)
    xlo = max(0, (int)floorf(lo - PAD));
    xhi = min(W - 1, (int)ceilf(hi + PAD));
}

// WIN = rows of the source window.  First launch: a persistent grid strides over the crops; oversize crops are appended to big_list.
// Second launch (big_list != nullptr as INPUT, `from_list`): a fixed grid strides over the queued crops.
// src_index (may be NULL): crop b reads source image src_index[b] (k_plane_gate has refused every crop whose index is out of
// range, so such a crop selects no plane and never reaches the source read).
template <int WIN>
__global__ void __launch_bounds__(WARP_THREADS, WIN == WIN_SMALL ? 2 : 1)
k_warp_rows(const uint8_t *__restrict__ src, const int32_t *__restrict__ src_index, const int32_t *__restrict__ src_kp, const int8_t *__restrict__ plane_j,
            const double *__restrict__ Minv, const PlaneRec *__restrict__ recs, uint8_t *__restrict__ warped, int H, int W, int *__restrict__ big_count,
            int *__restrict__ big_list, int from_list, int n_crops, int zero_ahead) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int crop_bytes = H * W * 3;
    const int row_bytes = W * 3;
    // smem carve-up
    uint8_t *s_win = smem;                                                            // WIN * 768 bytes
    uint32_t *s_mask = reinterpret_cast<uint32_t *>(smem + WIN * ROW_BYTES_MAX);       // WIN * MASK_WORDS words
    uint8_t *s_rows = reinterpret_cast<uint8_t *>(s_mask + WIN * MASK_WORDS);          // WARP_NWARPS * 768
    uint8_t *s_zero = s_rows + WARP_NWARPS * ROW_BYTES_MAX;                            // ZERO_BYTES of zeros: source of the bulk zero fill
    WarpSmemHeader *hd = reinterpret_cast<WarpSmemHeader *>(s_zero + ZERO_BYTES);
    if (tid == 0) {
        mbar_init(&hd->mbar, 1);
        fusg_wait_guard_start(&hd->wait_start);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // Zero fill of the five output planes (97 % of the output bytes): the TMA engine streams it from a small block of zeros,
    // `zero_ahead` crops AHEAD of the gather -- the fills of this CTA's next crops are in flight while the current crop is
    // computed, so most of the HBM write stream (the roofline term of the call) runs underneath the exact per-pixel arithmetic
    // instead of in a kernel of its own.  Lane 0 of warps 1..7 each issue a seventh of a crop's 240 bulk stores and own those
    // bulk groups; before the first row of a crop is stored each waits for its share of that crop's fill and the block barrier
    // orders everyone's stores behind it.  Warp 0 is left out: it runs the crop's prologue meanwhile.
    const bool filler = zero_ahead > 0 && lane == 0 && warp >= 1;
    if (zero_ahead > 0) {
        for (int k = tid; k < ZERO_BYTES / 16; k += WARP_THREADS) reinterpret_cast<int4 *>(s_zero)[k] = make_int4(0, 0, 0, 0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (filler) {
            for (int a = 0; a < zero_ahead; ++a) {
                const int it = (int)blockIdx.x + a * (int)gridDim.x;
                if (it < n_crops) zero_crop(warped + (size_t)it * N_TEX * crop_bytes, s_zero, (size_t)N_TEX * crop_bytes, warp - 1, WARP_NWARPS - 1);
                else bulk_commit();
            }
        }
    }
    uint32_t phase = 0;
    const int n_items = from_list ? *big_count : n_crops;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int b = from_list ? big_list[item] : item;
        uint8_t *gout = warped + (size_t)b * N_TEX * crop_bytes;
        __syncthreads();                                      // previous item done with the header / window
        // (filler lanes) this lane's blocks of the crop `zero_ahead` crops on are issued a block at a time between the rows of
        // the current crop -- a burst of bulk stores clogs the SM's memory-instruction queue for everybody -- and committed as
        // one group at the end of the crop
        bool zero_pending = filler;
        size_t zoff = 0, zend = 0;
        uint8_t *zdst = nullptr;
        if (filler) {
            const int nxt = item + zero_ahead * (int)gridDim.x;
            if (nxt < n_items) { zdst = warped + (size_t)nxt * N_TEX * crop_bytes; zoff = (size_t)(warp - 1) * ZERO_BYTES; zend = (size_t)N_TEX * crop_bytes; }
        }
        auto zero_step = [&](int n) {
            for (; n > 0 && zoff < zend; --n, zoff += (size_t)(WARP_NWARPS - 1) * ZERO_BYTES)
                bulk_s2g(zdst + zoff, s_zero, (uint32_t)(zend - zoff < (size_t)ZERO_BYTES ? zend - zoff : (size_t)ZERO_BYTES));
        };
        if (!from_list && warp == 2 && lane < 8) {
            // pull the next crop's few hundred bytes of per-crop inputs towards L2: its prologue is a chain of dependent loads
            // that otherwise waits behind the zero-fill traffic
            const size_t nb = (size_t)item + gridDim.x;
            if (nb < (size_t)n_items) {
                const void *pp = lane == 0 ? (const void *)(plane_j + nb * N_TEX)
                               : lane == 1 ? (const void *)(src_kp + nb * N_KP * 2)
                               : lane < 5  ? (const void *)(reinterpret_cast<const uint8_t *>(Minv + nb * N_TEX * 9) + (lane - 2) * 128)
                                           : (const void *)(reinterpret_cast<const uint8_t *>(recs + nb * N_TEX) + (lane - 5) * 128);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(pp));
            }
        }
        if (warp == 0) {
            // which source plane feeds output plane j -- last writer wins (planes_utils.py:79): the largest i with plane_j[i] == j --
            // and the source rows the selected polygons cover (only there can a mask bit be set); lane = output plane
            const int pj = lane < N_TEX ? (int)plane_j[b * N_TEX + lane] : -1;
            int sel = -1;
#pragma unroll
            for (int i = 0; i < N_TEX; ++i)
                if (__shfl_sync(0xffffffffu, pj, i) == lane) sel = i;
            int lo = INT_MAX, hi = INT_MIN;
            if (lane < N_TEX && sel >= 0) {
                for (int k = 0; k < c_plane_n[sel]; ++k) {
                    const int vy = src_kp[(b * N_KP + c_plane_kp[sel][k]) * 2 + 1];
                    lo = min(lo, vy); hi = max(hi, vy);
                }
            }
#pragma unroll
            for (int off = 4; off > 0; off >>= 1) {
                lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off));
                hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, off));
            }
            if (lane < N_TEX) hd->sel[lane] = sel;
            if (lane == 0) {
                lo = max(lo, 0); hi = min(hi, H - 1);
                hd->win_lo = lo; hd->win_hi = hi;
                hd->skip = 0;
                if (lo <= hi && hi - lo + 1 > WIN) {
                    hd->skip = 1;
                    big_list[atomicAdd(big_count, 1)] = b;    // (only reachable with WIN == WIN_SMALL: the big window holds any crop)
                }
            }
        }
        if (tid >= 32 && tid < 32 + N_TEX * 9) hd->Minv[0][tid - 32] = Minv[(size_t)b * N_TEX * 9 + (tid - 32)];
        __syncthreads();
        const int win_lo = hd->win_lo, win_hi = hd->win_hi;
        if (hd->skip || win_lo > win_hi) {                    // nothing to warp here: the planes stay zero
            if (filler) { zero_step(1 << 30); bulk_commit(); }
            continue;
        }
        const int win_rows = win_hi - win_lo + 1;
        const uint8_t *gwin = src + (size_t)(src_index ? src_index[b] : b) * crop_bytes + (size_t)win_lo * row_bytes;
        const uint32_t win_bytes = (uint32_t)win_rows * row_bytes;
        const bool use_tma = (win_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(gwin) & 15) == 0);
        if (use_tma) {
            if (tid == 0) {
                mbar_expect_tx(&hd->mbar, win_bytes);
                const uint32_t CH = 32768;
                for (uint32_t off = 0; off < win_bytes; off += CH) bulk_g2s(s_win + off, gwin + off, min(CH, win_bytes - off), &hd->mbar);
            }
        } else {
            for (uint32_t i = tid; i < win_bytes; i += WARP_THREADS) s_win[i] = gwin[i];
        }
        const uint8_t *s_src = s_win - (size_t)win_lo * row_bytes;                    // absolute-row addressing
        const uint32_t *mask_abs = s_mask - (size_t)win_lo * MASK_WORDS;
        const int bw = warp_block_w(H, W);
        const bool vec_rows = (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(gout) & 15) == 0);
        uint8_t *my_row = s_rows + warp * ROW_BYTES_MAX;
        const int4 z4 = make_int4(0, 0, 0, 0);
        bool src_ready = !use_tma;
        for (int j = 0; j < N_TEX; ++j) {
            const int i = hd->sel[j];
            if (i < 0) continue;
            __syncthreads();                                  // previous plane done with mask / spans
            {
                // polygon of source plane i: vertices and the row-independent part of its edges (one lane per edge), bounding
                // box, and the destination-side bounds k_solve left in recs
                const int n = c_plane_n[i];
                const int32_t *kp = src_kp + (size_t)b * N_KP * 2;
                if (tid < n) {
                    const int ka = c_plane_kp[i][tid == 0 ? n - 1 : tid - 1], kb = c_plane_kp[i][tid];
                    const int bx = kp[2 * kb], by = kp[2 * kb + 1];
                    hd->polyx[tid] = bx; hd->polyy[tid] = by;
                    PolyEdge e;
                    poly_edge_setup(kp[2 * ka], kp[2 * ka + 1], bx, by, H, W, e);
                    hd->edge[tid] = e;
                } else if (tid == 32) {
                    int x0 = INT_MAX, x1 = INT_MIN, y0 = INT_MAX, y1 = INT_MIN;
                    for (int k = 0; k < n; ++k) {
                        const int vx = kp[2 * c_plane_kp[i][k]], vy = kp[2 * c_plane_kp[i][k] + 1];
                        x0 = min(x0, vx); x1 = max(x1, vx); y0 = min(y0, vy); y1 = max(y1, vy);
                    }
                    hd->polyn = n;
                    hd->bbox[0] = x0; hd->bbox[1] = x1; hd->bbox[2] = y0; hd->bbox[3] = y1;
                    // A polygon that leaves the frame is rasterised with cv2's clipped-edge rules, whose mask can set pixels well
                    // away from the ideal polygon (e.g. a run along the border column): only in-frame polygons get the tight spans.
                    const bool inframe = x0 >= 0 && x1 < W && y0 >= 0 && y1 < H;
                    const PlaneRec &r = recs[(size_t)b * N_TEX + i];
                    hd->fwd_ok = r.ok && inframe;
                    hd->fwd_pad = r.pad;
                } else if (tid >= 64 && tid < 64 + n) {
                    const PlaneRec &r = recs[(size_t)b * N_TEX + i];
                    hd->fwdx[tid - 64] = r.fwdx[tid - 64]; hd->fwdy[tid - 64] = r.fwdy[tid - 64];
                }
            }
            __syncthreads();
            const double *M = hd->Minv[i];
            const int pl_lo = max(hd->bbox[2], 0), pl_hi = min(hd->bbox[3], H - 1);   // rows of THIS plane's polygon (inside the window)
            // polygon bit mask of the plane's source rows + active span of every output row
            for (int y = pl_lo + tid; y <= pl_hi; y += WARP_THREADS) {
                int lo[MAX_RANGES], hi[MAX_RANGES];
                const int rc = poly_row_ranges_edges(hd->edge, hd->polyn, y, W, lo, hi);
#pragma unroll
                for (int w = 0; w < MASK_WORDS; ++w) s_mask[(y - win_lo) * MASK_WORDS + w] = ranges_word(lo, hi, rc, w);
            }
            {   // the upper half of the CTA: thread = output row (H <= 256); the rows with a non-empty span as one bit word per warp
                // (the lower half is busy with the mask rows above: the two loops run side by side instead of one after the other)
                const int y = tid - MAX_HW;
                int xlo = 1, xhi = 0;
                if (y >= 0 && y < H) {
                    row_active_span(M, y, W, hd->bbox, xlo, xhi);
                    if (hd->fwd_ok && xlo <= xhi) {
                        int plo, phi;
                        row_polygon_span(hd->fwdx, hd->fwdy, hd->polyn, hd->fwd_pad, y, W, plo, phi);
                        xlo = max(xlo, plo); xhi = min(xhi, phi);
                    }
                    hd->span_lo[y] = (short)xlo; hd->span_hi[y] = (short)xhi;
                }
                const unsigned act = __ballot_sync(0xffffffffu, xlo <= xhi);
                if (lane == 0 && warp >= MAX_HW / 32) hd->row_bits[warp - MAX_HW / 32] = act;
            }
            if (!src_ready) { mbar_wait(&hd->mbar, phase); phase ^= 1; src_ready = true; }
            if (zero_pending) { bulk_wait(zero_ahead - 1); zero_pending = false; }     // groups are committed at the END of a crop: one fewer may be pending
            __syncthreads();
            uint8_t *oplane = gout + (size_t)j * crop_bytes;
            // the ACTIVE rows are dealt round-robin to the warps (neighbouring rows have similar spans; a static share of all rows
            // left warps idle at the barrier below, a shared-memory ticket per row cost more than it balanced)
            // active row k of the plane = the k-th set bit of row_bits (a find-n-th-set over the eight words)
            int n_active = 0;
#pragma unroll
            for (int ww = 0; ww < MAX_HW / 32; ++ww) n_active += __popc(hd->row_bits[ww]);
            for (int k = warp; k < n_active; k += WARP_NWARPS) {
                int y = -1, rem = k;
#pragma unroll
                for (int ww = 0; ww < MAX_HW / 32; ++ww) {
                    const unsigned m = hd->row_bits[ww];
                    const int c = __popc(m);
                    if (y < 0) { if (rem < c) y = ww * 32 + (int)__fns(m, 0, rem + 1); else rem -= c; }
                }
                const int xlo = hd->span_lo[y], xhi = hd->span_hi[y];
                uint8_t *orow = oplane + (size_t)y * row_bytes;
                // zero the staging row, then fill the active 32-pixel groups
                for (int k = lane; k < (row_bytes + 15) / 16; k += 32) reinterpret_cast<int4 *>(my_row)[k] = z4;
                __syncwarp();
                for (int g = xlo >> 5; g <= (xhi >> 5); ++g) {
                    const int x = g * 32 + lane;
                    if (x < W) {
                        const int bx = (x / bw) * bw;
                        const RowBase rb = row_base(M, bx, y);
                        int X, Y;
                        src_coord(M, rb, x - bx, X, Y);
                        const uchar3 v = bilinear_tap4<true>(s_src, mask_abs, MASK_WORDS, pl_lo, pl_hi, W, X, Y);
                        my_row[3 * x] = v.x; my_row[3 * x + 1] = v.y; my_row[3 * x + 2] = v.z;
                    }
                }
                __syncwarp();
                if (vec_rows) {
                    int4 *o4 = reinterpret_cast<int4 *>(orow);
                    for (int k = lane; k < row_bytes / 16; k += 32) o4[k] = reinterpret_cast<const int4 *>(my_row)[k];
                } else {
                    for (int k = lane; k < row_bytes; k += 32) orow[k] = my_row[k];
                }
                if (filler) zero_step(ZERO_PER_ROW);
                __syncwarp();
            }
        }
        if (!src_ready) { mbar_wait(&hd->mbar, phase); phase ^= 1; }          // never leave a bulk copy in flight into the window
        if (filler) { zero_step(1 << 30); bulk_commit(); }                    // what the rows did not cover
    }
    if (filler) bulk_wait(0);
}

// ============================================================================================
// Stand-alone kernels for the per-function drop-ins
// ============================================================================================
__global__ void __launch_bounds__(256) k_get_planes(const uint8_t *__restrict__ img, const int32_t *__restrict__ kp,
                                                    uint8_t *__restrict__ planes, int H, int W) {
    // grid: (rows, 5 planes, B).  One CTA per image row.
    const int y = blockIdx.x, p = blockIdx.y, b = blockIdx.z;
    __shared__ int lo[MAX_RANGES], hi[MAX_RANGES], rc;
    if (threadIdx.x == 0) {
        int px[6], py[6];
        const int n = c_plane_n[p];
        for (int k = 0; k < n; ++k) { px[k] = kp[(b * N_KP + c_plane_kp[p][k]) * 2]; py[k] = kp[(b * N_KP + c_plane_kp[p][k]) * 2 + 1]; }
        int l[MAX_RANGES], h[MAX_RANGES];
        const int c = poly_row_ranges(px, py, n, y, H, W, l, h);
        for (int k = 0; k < c; ++k) { lo[k] = l[k]; hi[k] = h[k]; }
        rc = c;
    }
    __syncthreads();
    const uint8_t *irow = img + ((size_t)b * H + y) * W * 3;
    uint8_t *orow = planes + (((size_t)b * N_TEX + p) * H + y) * W * 3;
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        bool in = false;
        for (int k = 0; k < rc; ++k) in = in || (x >= lo[k] && x <= hi[k]);
        orow[3 * x] = in ? irow[3 * x] : 0;
        orow[3 * x + 1] = in ? irow[3 * x + 1] : 0;
        orow[3 * x + 2] = in ? irow[3 * x + 2] : 0;
    }
}

__global__ void __launch_bounds__(256) k_warp_perspective(const uint8_t *__restrict__ img, const double *__restrict__ Hm,
                                                          uint8_t *__restrict__ out, int H, int W) {
    const int n = blockIdx.z;
    const int y = blockIdx.y;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ double M[9];
    if (threadIdx.x == 0) { double T[9]; invert3(Hm + 9 * n, T); for (int k = 0; k < 9; ++k) M[k] = T[k]; }
    __syncthreads();
    if (x >= W) return;
    const int bw = warp_block_w(H, W);
    const int bx = (x / bw) * bw;
    const RowBase rb = row_base(M, bx, y);
    int X, Y;
    src_coord(M, rb, x - bx, X, Y);
    const uint8_t *s = img + (size_t)n * H * W * 3;
    const uchar3 v = bilinear_tap4<false>(s, nullptr, 0, 0, H - 1, W, X, Y);
    uint8_t *o = out + (((size_t)n * H + y) * W + x) * 3;
    o[0] = v.x; o[1] = v.y; o[2] = v.z;
}


// ============================================================================================
// Frames larger than the shared-memory path (the reference runs the stage on whole 1280x720 frames,
// GUI/app_interface.py:181): same arithmetic, source and polygon bit masks read from global memory / L2.
// ============================================================================================
constexpr int PM_ROWS = 8;         // mask rows per CTA of k_plane_masks: one per warp

__global__ void __launch_bounds__(32 * PM_ROWS) k_plane_masks(const int32_t *__restrict__ src_kp, const int8_t *__restrict__ plane_j,
                                                             uint32_t *__restrict__ masks, int H, int W, int words) {
    // grid (ceil(H / PM_ROWS), 5, B): bit mask of PM_ROWS rows of SOURCE plane i (only for planes that are warped), a warp per row
    const int i = blockIdx.y, b = blockIdx.z;
    if (plane_j[b * N_TEX + i] < 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int y = blockIdx.x * PM_ROWS + warp;
    if (y >= H) return;
    __shared__ int s_lo[PM_ROWS][MAX_RANGES], s_hi[PM_ROWS][MAX_RANGES], s_rc[PM_ROWS];
    if (lane == 0) {
        int px[6], py[6], l[MAX_RANGES], h[MAX_RANGES];
        const int n = c_plane_n[i];
        for (int k = 0; k < n; ++k) { px[k] = src_kp[(b * N_KP + c_plane_kp[i][k]) * 2]; py[k] = src_kp[(b * N_KP + c_plane_kp[i][k]) * 2 + 1]; }
        const int c = poly_row_ranges(px, py, n, y, H, W, l, h);
        for (int k = 0; k < c; ++k) { s_lo[warp][k] = l[k]; s_hi[warp][k] = h[k]; }
        s_rc[warp] = c;
    }
    __syncwarp();
    uint32_t *row = masks + (((size_t)b * N_TEX + i) * H + y) * words;
    for (int w = lane; w < words; w += 32) row[w] = ranges_word(s_lo[warp], s_hi[warp], s_rc[warp], w);
}

constexpr int WF_ROWS = 8;        // output rows per CTA of k_warp_frame: one per warp

// WINDOW: only the window win[b] = (x0, y0, w, h) of every output plane is produced, written window-relative at warped + win_off[b]
// (plane j = [h, w, 3] at byte j*h*w*3): output row r is frame row y0 + r, pixel (r, c) equals frame pixel (y0 + r, x0 + c) of the
// whole-frame output bit for bit.  The grid then covers max_win_h rows; an item whose window is not window_ok (k_plane_gate has
// refused it) is not written at all.
template <bool WINDOW>
__global__ void __launch_bounds__(32 * WF_ROWS) k_warp_frame(const uint8_t *__restrict__ src, const int32_t *__restrict__ src_index,
                                                            const int32_t *__restrict__ src_kp,
                                                            const int8_t *__restrict__ plane_j, const double *__restrict__ Minv,
                                                            const uint32_t *__restrict__ masks, uint8_t *__restrict__ warped, int H, int W, int words,
                                                            int row_smem, const int32_t *__restrict__ win, const long long *__restrict__ win_off,
                                                            int max_win_h) {
    // grid (ceil(H / WF_ROWS), 5, B): WF_ROWS output rows of output plane j, one warp per row (a CTA per row meant 3.2 million CTAs
    // for the 600-item 1080p clip).  Rows are assembled in shared memory and leave with 16-byte stores.
    extern __shared__ __align__(16) uint8_t s_rows[];
    const int j = blockIdx.y, b = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int x0 = 0, y0 = 0, ww = W, wh = H;                  // the output rectangle in frame coordinates
    if (WINDOW) {
        if (!window_ok(win + 4 * b, max_win_h, H, W)) return;
        x0 = win[4 * b]; y0 = win[4 * b + 1]; ww = win[4 * b + 2]; wh = win[4 * b + 3];
    }
    __shared__ double M[9];
    __shared__ int s_i, s_bbox[4];
    if (threadIdx.x == 0) {
        int i = -1;
        for (int k = 0; k < N_TEX; ++k) if (plane_j[b * N_TEX + k] == j) i = k;      // last writer wins
        s_i = i;
        if (i >= 0) {
            for (int k = 0; k < 9; ++k) M[k] = Minv[((size_t)b * N_TEX + i) * 9 + k];
            int bbox[4] = {INT_MAX, INT_MIN, INT_MAX, INT_MIN};
            for (int k = 0; k < c_plane_n[i]; ++k) {
                const int vx = src_kp[(b * N_KP + c_plane_kp[i][k]) * 2], vy = src_kp[(b * N_KP + c_plane_kp[i][k]) * 2 + 1];
                bbox[0] = min(bbox[0], vx); bbox[1] = max(bbox[1], vx); bbox[2] = min(bbox[2], vy); bbox[3] = max(bbox[3], vy);
            }
            for (int k = 0; k < 4; ++k) s_bbox[k] = bbox[k];
        }
    }
    __syncthreads();
    const int r = blockIdx.x * WF_ROWS + warp;
    if (r >= wh) return;
    const int y = y0 + r;
    uint8_t *orow = WINDOW ? warped + win_off[b] + ((size_t)j * wh + r) * ww * 3 : warped + ((((size_t)b * N_TEX + j) * H + y) * W) * 3;
    const int i = s_i;
    const int row_bytes = ww * 3;
    const bool vec = (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(orow) & 15) == 0);   // rows of 16-byte-multiple frames stay aligned
    const int4 z4 = make_int4(0, 0, 0, 0);
    int xlo = 1, xhi = 0;
    if (i >= 0) {
        if (lane == 0) {
            int bb[4] = {s_bbox[0], s_bbox[1], s_bbox[2], s_bbox[3]};
            row_active_span(M, y, W, bb, xlo, xhi);
            if (WINDOW) { xlo = max(xlo, x0); xhi = min(xhi, x0 + ww - 1); }
        }
        xlo = __shfl_sync(0xffffffffu, xlo, 0);
        xhi = __shfl_sync(0xffffffffu, xhi, 0);
    }
    if (i < 0 || xlo > xhi) {
        if (vec) { int4 *o4 = reinterpret_cast<int4 *>(orow); for (int k = lane; k < row_bytes / 16; k += 32) o4[k] = z4; }
        else for (int k = lane; k < row_bytes; k += 32) orow[k] = 0;
        return;
    }
    uint8_t *s_row = s_rows + (size_t)warp * row_smem;
    const uint8_t *simg = src + (size_t)(src_index ? src_index[b] : b) * H * W * 3;     // a refused index selects no plane (i < 0 above)
    const uint32_t *mk = masks + ((size_t)b * N_TEX + i) * H * words;
    const int bw = warp_block_w(H, W);
    for (int c = lane; c < ww; c += 32) {
        const int x = x0 + c;
        uchar3 v = make_uchar3(0, 0, 0);
        if (x >= xlo && x <= xhi) {
            const int bx = (x / bw) * bw;
            const RowBase rb = row_base(M, bx, y);
            int X, Y;
            src_coord(M, rb, x - bx, X, Y);
            v = bilinear_tap4<true>(simg, mk, words, 0, H - 1, W, X, Y);
        }
        s_row[3 * c] = v.x; s_row[3 * c + 1] = v.y; s_row[3 * c + 2] = v.z;
    }
    __syncwarp();
    if (vec) {
        int4 *o4 = reinterpret_cast<int4 *>(orow);
        const int4 *s4 = reinterpret_cast<const int4 *>(s_row);
        for (int k = lane; k < row_bytes / 16; k += 32) o4[k] = s4[k];
    } else {
        for (int k = lane; k < row_bytes; k += 32) orow[k] = s_row[k];
    }
}

}  // namespace fusg

// ================================================================================================
// C ABI
// ================================================================================================
using namespace fusg;

// dynamic shared memory opt-in of the solver kernels (per device) and the number of point sets per warp
static int solver_prepare() {
    const cudaError_t e = fusg_once_per_device(3, 0, [] {
        cudaError_t r = cudaFuncSetAttribute(k_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, SOLVER_SMEM_BYTES);
        return r != cudaSuccess ? r : cudaFuncSetAttribute(k_find_homography, cudaFuncAttributeMaxDynamicSharedMemorySize, SOLVER_SMEM_BYTES);
    });
    return fusg_record_cuda(e);
}
// one point set per warp while the warps fit on the device at once (latency of a single solve), up to 32 (throughput)
static int solver_lanes(long long tasks) {
    const long long slots = (long long)fusg_num_sms() * SOLVER_WARPS_PER_SM;         // 4 x 52 KB of scratch per SM
    long long l = (tasks + slots - 1) / slots;
    return (int)(l < 1 ? 1 : (l > 32 ? 32 : l));
}

static size_t warp_smem_bytes(int win) {
    return (size_t)win * ROW_BYTES_MAX + (size_t)win * MASK_WORDS * 4 + (size_t)WARP_NWARPS * ROW_BYTES_MAX + ZERO_BYTES + sizeof(WarpSmemHeader) + 128;
}

// workspace: Minv [B,5,9] f64 | counters [4] i32 (6-point tasks, 4-point tasks, big-window crops, -) | list6 [2B] i32 | list4 [3B] i32 |
//            big_list [B] i32 | PlaneRec [B,5] (56 bytes each) | (frames > 256: plane bit masks [B,5,H,ceil(W/32)] u32)
static size_t warp_ws_base(int B) {
    return (size_t)B * N_TEX * 9 * sizeof(double) + (size_t)(4 + 6 * (size_t)B) * sizeof(int) + (size_t)B * N_TEX * sizeof(PlaneRec);
}

extern "C" size_t fusg_warp_workspace_bytes(int B) { return B <= 0 ? 0 : warp_ws_base(B); }

extern "C" size_t fusg_warp_workspace_bytes_hw(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    size_t n = (warp_ws_base(B) + 15) & ~(size_t)15;
    if (H > MAX_HW || W > MAX_HW) n += (size_t)B * N_TEX * H * ((W + 31) / 32) * sizeof(uint32_t);
    return n;
}

extern "C" int fusg_visibility(const double *K, const double *E, const double *kp3d, uint8_t *vis, int32_t *pts,
                               int32_t *areas, int B, int H, int W, void *stream) {
    if (!K || !E || !kp3d || !vis || B <= 0 || H <= 0 || W <= 0) return FUSG_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    k_visibility<<<(B + VIS_WARPS - 1) / VIS_WARPS, VIS_WARPS * 32, 0, st>>>(K, E, nullptr, kp3d, nullptr, vis, pts, areas, B, H, W);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_get_planes(const uint8_t *img, const int32_t *kp, uint8_t *planes, int B, int H, int W, void *stream) {
    if (!img || !kp || !planes || B <= 0 || H <= 0 || W <= 0) return FUSG_ERR_ARG;
    if (H > 65535 || B > 65535) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    k_get_planes<<<dim3(H, N_TEX, B), 256, 0, st>>>(img, kp, planes, H, W);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_find_homography(const int32_t *src, const int32_t *dst, int n, double *Hm, uint8_t *ok, int N, void *stream) {
    if (!src || !dst || !Hm || !ok || N <= 0) return FUSG_ERR_ARG;
    if (n < 4 || n > 6) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (solver_prepare() != FUSG_OK) return FUSG_ERR_CUDA;
    const int lanes = solver_lanes(N);
    k_find_homography<<<(N + lanes - 1) / lanes, 32, SOLVER_SMEM_BYTES, st>>>(src, dst, n, Hm, ok, N, lanes);
    fusg_count_launch(1);
    return fusg_check_launch();
}

extern "C" int fusg_warp_perspective(const uint8_t *img, const double *Hm, uint8_t *out, int N, int H, int W, void *stream) {
    if (!img || !Hm || !out || N <= 0 || H <= 0 || W <= 0) return FUSG_ERR_ARG;
    if (H > 65535 || N > 65535) return FUSG_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    k_warp_perspective<<<dim3((W + 255) / 256, H, N), 256, 0, st>>>(img, Hm, out, H, W);
    fusg_count_launch(1);
    return fusg_check_launch();
}

// Workspace carve-up shared by the fused entry points (layout at warp_ws_base).
struct WarpWs {
    double *Minv;
    int *counters, *list6, *list4, *big_list;
    PlaneRec *recs;
    uint32_t *masks;              // plane bit masks of the global-memory gather
};
static WarpWs warp_ws(void *workspace, int B) {
    WarpWs w;
    w.Minv = reinterpret_cast<double *>(workspace);
    w.counters = reinterpret_cast<int *>(w.Minv + (size_t)B * N_TEX * 9);
    w.list6 = w.counters + 4; w.list4 = w.list6 + 2 * (size_t)B; w.big_list = w.list4 + 3 * (size_t)B;
    w.recs = reinterpret_cast<PlaneRec *>(w.big_list + (size_t)B);
    w.masks = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(workspace) + ((warp_ws_base(B) + 15) & ~(size_t)15));
    return w;
}

// The front half of every fused entry point: visibility of both poses, plane gating (win != nullptr: the window check of
// fusg_warp_fused_window), homographies.  recs (may be NULL) receives the destination bounds k_warp_rows uses.
static int warp_front(const int32_t *src_index, int n_src, const int32_t *src_kp, const int32_t *dst_kp, const double *K, const double *E_src,
                      const double *E_dst, const double *kp3d, const double *kp3d_dst, const int32_t *win, int max_win_h, uint8_t *vis,
                      int8_t *plane_j, double *H12, const WarpWs &ws, PlaneRec *recs, int B, int H, int W, cudaStream_t st) {
    k_visibility<<<(2 * B + VIS_WARPS - 1) / VIS_WARPS, VIS_WARPS * 32, 0, st>>>(K, E_src, E_dst, kp3d, kp3d_dst, vis, nullptr, nullptr, 2 * B, H, W);
    if (fusg_record_cuda(cudaMemsetAsync(ws.counters, 0, 4 * sizeof(int), st)) != FUSG_OK) return FUSG_ERR_CUDA;
    if (win)
        k_plane_gate<true><<<(B * N_TEX + 255) / 256, 256, 0, st>>>(src_kp, dst_kp, vis, plane_j, H12, ws.Minv, ws.counters, ws.list6, ws.list4,
                                                                     src_index, n_src, win, max_win_h, B, H, W);
    else
        k_plane_gate<false><<<(B * N_TEX + 255) / 256, 256, 0, st>>>(src_kp, dst_kp, vis, plane_j, H12, ws.Minv, ws.counters, ws.list6, ws.list4,
                                                                      src_index, n_src, nullptr, 0, B, H, W);
    fusg_count_launch(2);
    if (solver_prepare() != FUSG_OK) return FUSG_ERR_CUDA;
    // 32 point sets per warp whatever the batch: the lanes of a warp run in lock step, so a fuller warp costs no
    // latency, and the fewest possible SMs lose 52 KB of shared memory to a solver warp (the VUNet convolutions of the
    // same step want all of it); the grid covers the worst case, warps beyond the task count exit at once
    const int lanes = 32;
    const int blocks6 = (2 * B + lanes - 1) / lanes, blocks4 = (3 * B + lanes - 1) / lanes;
    k_solve<<<blocks6 + blocks4, 32, SOLVER_SMEM_BYTES, st>>>(src_kp, dst_kp, plane_j, H12, ws.Minv, ws.counters, ws.list6, ws.list4, recs, blocks6, lanes);
    fusg_count_launch(1);
    return FUSG_OK;
}

// Polygon bit masks of every warped source plane, then the global-memory gather (whole frame, or the windows when win != nullptr).
static int warp_gather_global(const uint8_t *src, const int32_t *src_index, const int32_t *src_kp, const int8_t *plane_j, const WarpWs &ws,
                              uint8_t *warped, const int32_t *win, const long long *win_off, int max_win_h, int B, int H, int W, cudaStream_t st) {
    const int words = (W + 31) / 32;
    k_plane_masks<<<dim3((H + PM_ROWS - 1) / PM_ROWS, N_TEX, B), 32 * PM_ROWS, 0, st>>>(src_kp, plane_j, ws.masks, H, W, words);
    const size_t row_smem = ((size_t)W * 3 + 15) & ~(size_t)15;
    const size_t frame_smem = row_smem * WF_ROWS;
    if (frame_smem > 200 * 1024) return FUSG_ERR_UNSUPPORTED;
    if (win) {
        if (frame_smem > 48 * 1024 &&
            fusg_once_per_device(4, frame_smem, [frame_smem] { return cudaFuncSetAttribute(k_warp_frame<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)frame_smem); }) != cudaSuccess)
            return fusg_check_launch();
        const int rows = max_win_h < H ? max_win_h : H;          // a window that passes window_ok has at most H rows
        k_warp_frame<true><<<dim3((rows + WF_ROWS - 1) / WF_ROWS, N_TEX, B), 32 * WF_ROWS, frame_smem, st>>>(src, src_index, src_kp, plane_j, ws.Minv, ws.masks,
                                                                                                             warped, H, W, words, (int)row_smem, win, win_off, max_win_h);
    } else {
        if (frame_smem > 48 * 1024 &&
            fusg_once_per_device(2, frame_smem, [frame_smem] { return cudaFuncSetAttribute(k_warp_frame<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)frame_smem); }) != cudaSuccess)
            return fusg_check_launch();
        k_warp_frame<false><<<dim3((H + WF_ROWS - 1) / WF_ROWS, N_TEX, B), 32 * WF_ROWS, frame_smem, st>>>(src, src_index, src_kp, plane_j, ws.Minv, ws.masks,
                                                                                                           warped, H, W, words, (int)row_smem, nullptr, nullptr, 0);
    }
    fusg_count_launch(4);
    return FUSG_OK;
}

// src_index == nullptr: crop b reads src[b].  Otherwise src holds n_src images and crop b reads src[src_index[b]].
static int warp_fused_impl(const uint8_t *src, const int32_t *src_index, int n_src, const int32_t *src_kp, const int32_t *dst_kp, const double *K,
                           const double *E_src, const double *E_dst, const double *kp3d, const double *kp3d_dst, uint8_t *warped, uint8_t *vis,
                           int8_t *plane_j, double *H12, void *workspace, size_t workspace_bytes, int B, int H, int W,
                           void *stream) {
    if (!src || !src_kp || !dst_kp || !K || !E_src || !E_dst || !kp3d || !warped || !vis || !plane_j || !workspace) return FUSG_ERR_ARG;
    if (B <= 0) return FUSG_ERR_ARG;
    if (src_index && n_src <= 0) return FUSG_ERR_ARG;
    if (H < 8 || W < 8 || H > 65535 || B > 65535) return FUSG_ERR_UNSUPPORTED;
    const bool frame_path = H > MAX_HW || W > MAX_HW;
    if (workspace_bytes < fusg_warp_workspace_bytes_hw(B, H, W)) return FUSG_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const WarpWs ws = warp_ws(workspace, B);
    if (!frame_path) {
        if (fusg_once_per_device(1, 0, [] {
                cudaError_t e = cudaFuncSetAttribute(k_warp_rows<WIN_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)warp_smem_bytes(WIN_SMALL));
                return e != cudaSuccess ? e : cudaFuncSetAttribute(k_warp_rows<MAX_HW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)warp_smem_bytes(MAX_HW));
            }) != cudaSuccess)
            return fusg_check_launch();
    }
    // The zero fill of the five planes (97 % of the output bytes stay zero) rides inside k_warp_rows as TMA bulk stores issued
    // two crops ahead of the gather (see the kernel); only outputs that are not 16-byte granular are cleared by a memset.
    // (Measured alternatives, 16k crops: a fill kernel of its own costs 2.6 ms when serial; on a helper stream underneath
    // k_visibility / k_solve it gains 0.2 ms as plain stores -- the store flood slows the latency-bound solver by as much as
    // it saves -- and as bulk stores it made the call 2-4x SLOWER; plain stores from the gather's own warps: 6.0 ms against
    // 4.8 ms for this form.  The gather without any fill takes 3.6 ms.)
    const bool bulk_zero = !frame_path && ((size_t)N_TEX * H * W * 3) % 16 == 0 && (reinterpret_cast<uintptr_t>(warped) & 15) == 0;
    if (!frame_path && !bulk_zero) {
        if (fusg_record_cuda(cudaMemsetAsync(warped, 0, (size_t)B * N_TEX * H * W * 3, st)) != FUSG_OK) return FUSG_ERR_CUDA;
        fusg_count_launch(1);
    }
    const int rc = warp_front(src_index, n_src, src_kp, dst_kp, K, E_src, E_dst, kp3d, kp3d_dst, nullptr, 0, vis, plane_j, H12, ws,
                              frame_path ? nullptr : ws.recs, B, H, W, st);
    if (rc != FUSG_OK) return rc;
    if (!frame_path) {
        // persistent: two CTAs per SM stride over the crops
        const int grid = B < 2 * fusg_num_sms() ? B : 2 * fusg_num_sms();
        k_warp_rows<WIN_SMALL><<<grid, WARP_THREADS, warp_smem_bytes(WIN_SMALL), st>>>(src, src_index, src_kp, plane_j, ws.Minv, ws.recs, warped, H, W, ws.counters + 2,
                                                                                       ws.big_list, 0, B, bulk_zero ? ZERO_AHEAD : 0);
        // crops whose polygons span more than WIN_SMALL source rows (a vehicle filling the crop): full-height window
        const int bgrid = B < fusg_num_sms() ? B : fusg_num_sms();
        k_warp_rows<MAX_HW><<<bgrid, WARP_THREADS, warp_smem_bytes(MAX_HW), st>>>(src, src_index, src_kp, plane_j, ws.Minv, ws.recs, warped, H, W, ws.counters + 2,
                                                                                  ws.big_list, 1, B, 0);
        fusg_count_launch(2);
    } else {
        const int grc = warp_gather_global(src, src_index, src_kp, plane_j, ws, warped, nullptr, nullptr, 0, B, H, W, st);
        if (grc != FUSG_OK) return grc;
    }
    return fusg_check_launch();
}

extern "C" size_t fusg_warp_window_workspace_bytes(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    return ((warp_ws_base(B) + 15) & ~(size_t)15) + (size_t)B * N_TEX * H * ((W + 31) / 32) * sizeof(uint32_t);
}

extern "C" int fusg_warp_fused_window(const uint8_t *src, const int32_t *src_index, int n_src, const int32_t *src_kp, const int32_t *dst_kp,
                                      const double *K, const double *E_src, const double *E_dst, const double *kp3d_src, const double *kp3d_dst,
                                      const int32_t *win, const long long *win_off, int max_win_h, uint8_t *warped, uint8_t *vis, int8_t *plane_j,
                                      double *H12, void *workspace, size_t workspace_bytes, int B, int H, int W, void *stream) {
    if (!src || !src_kp || !dst_kp || !K || !E_src || !E_dst || !kp3d_src || !win || !win_off || !warped || !vis || !plane_j || !workspace)
        return FUSG_ERR_ARG;
    if (B <= 0 || max_win_h <= 0) return FUSG_ERR_ARG;
    if (src_index && n_src <= 0) return FUSG_ERR_ARG;
    if (H < 8 || W < 8 || H > 65535 || B > 65535) return FUSG_ERR_UNSUPPORTED;
    if (workspace_bytes < fusg_warp_window_workspace_bytes(B, H, W)) return FUSG_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const WarpWs ws = warp_ws(workspace, B);
    const int rc = warp_front(src_index, n_src, src_kp, dst_kp, K, E_src, E_dst, kp3d_src, kp3d_dst, win, max_win_h, vis, plane_j, H12, ws, nullptr,
                              B, H, W, st);
    if (rc != FUSG_OK) return rc;
    const int grc = warp_gather_global(src, src_index, src_kp, plane_j, ws, warped, win, win_off, max_win_h, B, H, W, st);
    if (grc != FUSG_OK) return grc;
    return fusg_check_launch();
}

extern "C" int fusg_warp_fused(const uint8_t *src, const int32_t *src_kp, const int32_t *dst_kp, const double *K,
                               const double *E_src, const double *E_dst, const double *kp3d, uint8_t *warped, uint8_t *vis,
                               int8_t *plane_j, double *H12, void *workspace, size_t workspace_bytes, int B, int H, int W,
                               void *stream) {
    return warp_fused_impl(src, nullptr, 0, src_kp, dst_kp, K, E_src, E_dst, kp3d, nullptr, warped, vis, plane_j, H12, workspace, workspace_bytes, B, H, W, stream);
}

extern "C" int fusg_warp_fused_traj(const uint8_t *src, const int32_t *src_kp, const int32_t *dst_kp, const double *K,
                                    const double *E_src, const double *E_dst, const double *kp3d_src, const double *kp3d_dst,
                                    uint8_t *warped, uint8_t *vis, int8_t *plane_j, double *H12, void *workspace, size_t workspace_bytes,
                                    int B, int H, int W, void *stream) {
    if (!kp3d_dst) return FUSG_ERR_ARG;
    return warp_fused_impl(src, nullptr, 0, src_kp, dst_kp, K, E_src, E_dst, kp3d_src, kp3d_dst, warped, vis, plane_j, H12, workspace, workspace_bytes, B, H, W, stream);
}

extern "C" int fusg_warp_fused_idx(const uint8_t *src, const int32_t *src_index, int n_src, const int32_t *src_kp, const int32_t *dst_kp,
                                   const double *K, const double *E_src, const double *E_dst, const double *kp3d_src, const double *kp3d_dst,
                                   uint8_t *warped, uint8_t *vis, int8_t *plane_j, double *H12, void *workspace, size_t workspace_bytes,
                                   int B, int H, int W, void *stream) {
    if (!src_index || n_src <= 0) return FUSG_ERR_ARG;
    return warp_fused_impl(src, src_index, n_src, src_kp, dst_kp, K, E_src, E_dst, kp3d_src, kp3d_dst, warped, vis, plane_j, H12, workspace,
                           workspace_bytes, B, H, W, stream);
}
