/*
 * fusg.h -- C ABI of the B200-native novel-view-completion hot path.
 *
 * The reference (alexj94/future_urban_scene_generation) is pure Python; it has no FFI for this
 * path.  Each entry point below names the reference Python interface it stands behind; the
 * Python host layer (future_urban_scene_generation_b200/{warp_learn,vunet}) binds them with
 * ctypes and re-exposes the reference's own module/function names.  INTEGRATION.md shows the
 * binding a reference maintainer would add.
 *
 * Conventions: plain pointers and sizes only; every pointer is a DEVICE pointer unless its name
 * ends in _host; `stream` is a cudaStream_t passed as void*; calls are asynchronous on that
 * stream, never allocate, never synchronise; the return value is 0 or a negative FUSG_ERR_*.
 *
 * Devices and threads: a call works on the CURRENT device of the calling thread (cudaSetDevice), whose
 * memory the pointers must belong to; `stream` must be a stream of that device.  One process may drive
 * several devices, and several host threads may call concurrently: kernel attributes and SM counts are
 * cached per device under a mutex, nothing else is shared.  fusg_last_error / fusg_kernel_launches are
 * process-wide diagnostics.
 *
 * Faults: device-side mbarrier waits are bounded (seconds); a TMA-descriptor or pipeline bug makes the
 * kernel trap (the next call returns FUSG_ERR_CUDA, fusg_last_error names the launch failure) instead
 * of hanging the GPU.
 */
#ifndef FUSG_H_
#define FUSG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FUSG_OK 0
#define FUSG_ERR_ARG (-1)          /* null pointer / non-positive size                    */
#define FUSG_ERR_UNSUPPORTED (-2)  /* shape outside what the kernels cover                */
#define FUSG_ERR_CUDA (-3)         /* a CUDA runtime call failed (see fusg_last_error)    */
#define FUSG_ERR_WORKSPACE (-4)    /* workspace too small                                 */

/* Version / diagnostics ---------------------------------------------------------------- */
int fusg_version(void);
const char *fusg_last_error(void);     /* text of the last CUDA error seen by this library  */
int fusg_kernel_launches(void);        /* number of kernels this library launched so far     */

/* ====================================================================================== */
/* Warp stage                                                                              */
/* ====================================================================================== */

/* Bytes of device workspace fusg_warp_fused needs for a batch of B crops (H, W <= 256), and for any frame size. */
size_t fusg_warp_workspace_bytes(int B);
size_t fusg_warp_workspace_bytes_hw(int B, int H, int W);

/*
 * Fused planar warp for a batch of B vehicle crops.  Stands behind
 *     warp_learn/online_visibility.py:105-150   compute_visibility  (source and destination pose)
 *     warp_learn/planes_utils.py:11-37          get_planes          (polygon masks, never materialised)
 *     warp_learn/planes_utils.py:40-82          warp_unwarp_planes  (first return value only)
 * i.e. the sequence trajectory_inference.py:165-174 runs per vehicle and per future step.
 *
 *   src      [B,H,W,3] u8   source crops (HWC, as cv2 images)
 *   src_kp   [B,12,2]  i32  source-pose plane vertices: the int32-truncated 2D keypoints of
 *                           planes_utils.py:22-27, utils/keypoint_utils.py:9-13 (_KP_NAMES) order
 *   dst_kp   [B,12,2]  i32  destination-pose plane vertices, same convention
 *   K        [B,3,3]   f64  intrinsics
 *   E_src    [B,3,4]   f64  source extrinsic (world->camera), row major
 *   E_dst    [B,3,4]   f64  destination extrinsic
 *   kp3d     [B,12,3]  f64  CAD keypoints, _KP_NAMES order
 *   warped   [B,5,H,W,3] u8 out: planes_warped (left,right,roof,front,back); fully written
 *   vis      [B,2,7]   u8   out: visibility of (left,right,roof,front,back,front_bt,back_bt)
 *                           for the source (index 0) and destination (index 1) pose
 *   plane_j  [B,5]     i8   out: target plane index j of source plane i, or -1 if skipped
 *   H12      [B,5,9]   f64  out (may be NULL): homography of source plane i (zeros if skipped)
 *   workspace, workspace_bytes: device scratch, >= fusg_warp_workspace_bytes(B)
 *
 * H, W >= 8.  Up to 256 x 256 the crop is staged in shared memory (the HBM-bound fast path); larger
 * frames (the reference works on 1280 x 720) gather from global memory with the same arithmetic and need
 * fusg_warp_workspace_bytes_hw(B,H,W) of workspace.  Vertices outside the frame are handled like cv2.fillPoly
 * handles them (clipped edges); only a crop with a vertex beyond +-2^20 px is refused: outputs zero, plane_j = -2.
 */
int fusg_warp_fused(const uint8_t *src, const int32_t *src_kp, const int32_t *dst_kp,
                    const double *K, const double *E_src, const double *E_dst, const double *kp3d,
                    uint8_t *warped, uint8_t *vis, int8_t *plane_j, double *H12,
                    void *workspace, size_t workspace_bytes,
                    int B, int H, int W, void *stream);

/*
 * The same call for the trajectory loop (trajectory_inference.py:359-379), where the destination pose is the SAME camera
 * looking at MOVED keypoints: the destination visibility is computed from kp3d_dst [B,12,3] (e.g. fusg_step_keypoints'
 * output) instead of kp3d_src.  E_dst is normally E_src there.
 */
int fusg_warp_fused_traj(const uint8_t *src, const int32_t *src_kp, const int32_t *dst_kp,
                         const double *K, const double *E_src, const double *E_dst, const double *kp3d_src, const double *kp3d_dst,
                         uint8_t *warped, uint8_t *vis, int8_t *plane_j, double *H12,
                         void *workspace, size_t workspace_bytes, int B, int H, int W, void *stream);

/*
 * The same call with source images shared between crops (the trajectory loop warps one source crop of a vehicle for every
 * future step, trajectory_inference.py:165-174,413): src [n_src,H,W,3] u8 holds n_src images and crop b reads image
 * src_index[b] (src_index [B] i32, device).  Every other array is per crop as above.  kp3d_dst == NULL means fusg_warp_fused,
 * otherwise fusg_warp_fused_traj.  A crop whose index lies outside [0, n_src) is refused like a vertex beyond 2^20 px: outputs
 * zero, plane_j = -2; no source byte is read for it.  A NULL src_index or n_src <= 0 is FUSG_ERR_ARG.  Same workspace.
 */
int fusg_warp_fused_idx(const uint8_t *src, const int32_t *src_index, int n_src, const int32_t *src_kp, const int32_t *dst_kp,
                        const double *K, const double *E_src, const double *E_dst, const double *kp3d_src, const double *kp3d_dst,
                        uint8_t *warped, uint8_t *vis, int8_t *plane_j, double *H12,
                        void *workspace, size_t workspace_bytes, int B, int H, int W, void *stream);

/*
 * The same call writing only a window of each item's five planes: the pixels get_icn_inputs reads (the square crop of
 * warp_learn/models.py:334-342 around the destination sketch mask, clipped to the frame -- trajectory_inference.py:374-391 warps the
 * whole frame and reads only that square).  win [B,4] i32 = (x0, y0, w, h) in frame pixels, win_off [B] i64 = byte offset of item b's
 * block in `warped`; the block holds planes j = 0..4, each [h,w,3] u8 row major, plane j at win_off[b] + j*h*w*3.  Pixel (r, c) of
 * plane j equals warped[b, j, y0 + r, x0 + c] of fusg_warp_fused_idx (src_index != NULL) / fusg_warp_fused(_traj) bit for bit, for any
 * frame size; every byte of every window is written (zeros where no plane writes) and nothing outside the windows.  vis, plane_j and
 * H12 are those of the whole-frame call.  src_index may be NULL (crop b reads src[b], src [B,H,W,3]), otherwise as fusg_warp_fused_idx;
 * kp3d_dst may be NULL (kp3d_src for both poses).  An item is refused (plane_j = -2) like there, and also when its window is empty,
 * not inside the H x W frame or has more than max_win_h rows -- such a window is not written at all; a refused item with a valid
 * window gets an all-zero window.  Workspace >= fusg_warp_window_workspace_bytes(B, H, W).  max_win_h <= 0 is FUSG_ERR_ARG.
 */
size_t fusg_warp_window_workspace_bytes(int B, int H, int W);
int fusg_warp_fused_window(const uint8_t *src, const int32_t *src_index, int n_src, const int32_t *src_kp, const int32_t *dst_kp,
                           const double *K, const double *E_src, const double *E_dst, const double *kp3d_src, const double *kp3d_dst,
                           const int32_t *win, const long long *win_off, int max_win_h,
                           uint8_t *warped, uint8_t *vis, int8_t *plane_j, double *H12,
                           void *workspace, size_t workspace_bytes, int B, int H, int W, void *stream);

/*
 * Per-step keypoint kinematics of the trajectory loop (SURVEY.md section 8f-4) for N (vehicle, future step) items:
 *   moved = v @ z_rot(theta) + tr                         trajectory_inference.py:359-361, utils/geometry.py:80-113
 *   kp2d  = cv2.projectPoints(moved, rvec, tvec, K, 0)    trajectory_inference.py:363-367
 *   verts = np.int32((kp2d / (W,H)) * (W,H))              warp_learn/vehicle_utils.py:24-26, warp_learn/planes_utils.py:22-27
 *   kp3d [V,12,3] f64 CAD keypoints per vehicle; vehicle [N] i32 index into the per-vehicle arrays; rot [N,3,3] f32 = z_rot(theta)
 *   (the reference builds it in float32); tr [N,3] f64; R [V,3,3] f64 = cv2.Rodrigues(rvec); t [V,3]; K [V,3,3]
 *   -> kp3d_out [N,12,3] f64, kp2d_out [N,12,2] f64, verts [N,12,2] i32: the kp3d_dst / dst_kp inputs of fusg_warp_fused_traj.
 * theta / tr per step (the +-20 degree gates of trajectory_inference.py:267-298) are a few scalars per item and stay on the host.
 */
int fusg_step_keypoints(const double *kp3d, const int32_t *vehicle, const float *rot, const double *tr, const double *R, const double *t,
                        const double *K, double *kp3d_out, double *kp2d_out, int32_t *verts, int N, int H, int W, void *stream);

/*
 * Visibility only (compute_visibility, online_visibility.py:105-150) for B poses.
 *   K [B,3,3], E [B,3,4], kp3d [B,12,3] f64 -> vis [B,7] u8, pts [B,12,2] i32 (int()-truncated
 *   projections; may be NULL), areas [B,7,2] i32 (absolute, occluded; may be NULL).
 */
int fusg_visibility(const double *K, const double *E, const double *kp3d,
                    uint8_t *vis, int32_t *pts, int32_t *areas, int B, int H, int W, void *stream);

/*
 * get_planes (planes_utils.py:11-37): planes[b,p] = image[b] * fillPoly(mask of plane p).
 *   img [B,H,W,3] u8, kp [B,12,2] i32 -> planes [B,5,H,W,3] u8.   Any H,W >= 1.
 */
int fusg_get_planes(const uint8_t *img, const int32_t *kp, uint8_t *planes, int B, int H, int W, void *stream);

/*
 * Homographies of cv2.findHomography(src, dst) (method 0) for N point sets of n = 4 or 6 points.
 *   src,dst [N,n,2] i32 -> H [N,9] f64, ok [N] u8 (0 where OpenCV returns None).
 */
int fusg_find_homography(const int32_t *src, const int32_t *dst, int n, double *H, uint8_t *ok, int N, void *stream);

/*
 * cv2.warpPerspective(img, H, (W,H)) with default flags for N images (planes_utils.py:76-77),
 * gathered from global memory (any H,W >= 1).   img [N,H,W,3] u8, Hm [N,9] f64 -> out [N,H,W,3] u8.
 */
int fusg_warp_perspective(const uint8_t *img, const double *Hm, uint8_t *out, int N, int H, int W, void *stream);


/* ====================================================================================== */
/* VUNet convolution engine                                                                */
/* ====================================================================================== */

#define FUSG_DTYPE_BF16 0
#define FUSG_DTYPE_F32 1          /* fp32 verification build: direct kernels only */
#define FUSG_DTYPE_F16 2          /* fp16 activations/weights, fp32 accumulate: the ICN row (normalised activations;
                                   * 8x finer rounding than bf16 at the same tensor-core rate).  tcgen05 path: raw NHWC
                                   * outputs and NCHW fp32 slots only */

#define FUSG_IMPL_AUTO 0
#define FUSG_IMPL_TCGEN05 1       /* implicit-GEMM tcgen05/TMEM kernel fed by TMA (bf16 only) */
#define FUSG_IMPL_DIRECT 2        /* CUDA-core direct convolution (any dtype; the in-library check) */
#define FUSG_IMPL_SMALLCIN 3      /* streaming 1x1 convolution of a network input stored 16 channels wide (cphys0 = pitch0 = 16, cin_real <= 8):
                                   * the first NiN of each encoder, where K is 3 or 6 and the layer is pure HBM streaming */

#define FUSG_OUT_PLAIN 0          /* out[b, y, x, n]                                              */
#define FUSG_OUT_D2S 1            /* DepthToSpace(2), vunet/layers.py:173-194 (block-major):      */
                                  /*   out[b, 2y+blk/2, 2x+blk%2, n % (cout/4)], blk = n/(cout/4) */
#define FUSG_OUT_S2D 2            /* SpaceToDepth(2), vunet/layers.py:197-221:                    */
                                  /*   out[b, y/2, x/2, ((y%2)*2 + x%2)*cout + n]                 */
#define FUSG_OUT_D2S_BLOCK 3      /* one block of a DepthToSpace of a channel concat              */
                                  /*   (vunet/models.py:85-86): out[b, 2y+blk/2, 2x+blk%2, n]     */
#define FUSG_OUT_UNPAIR 4         /* pixel-pair packed layer (fusg_fold_weightnorm_paired):       */
                                  /*   out[b, y, 2x + n/(cout/2), n % (cout/2)]; NCHW fp32 slots  */

#define FUSG_CONV_MAX_OUTS 6

/* One output of a convolution launch.  value = conv + bias (+ residual); source 1 adds the
 * Sampler noise (vunet/layers.py:163-167). */
typedef struct fusg_conv_out {
    void *ptr;          /* NULL = unused slot                                                    */
    int32_t source;     /* 0: value, 1: value + noise                                            */
    int32_t elu;        /* 0: raw, 1: ELU(raw) -- pre-activation for the next layer, 2: tanh(raw)
                         * (the ICN's last Conv2dBlock, warp_learn/models.py:174-175; NCHW fp32 slots)   */
    int32_t layout;     /* 0: NHWC in the activation dtype, 1: NCHW fp32 (API-visible tensors)   */
    int32_t mode;       /* FUSG_OUT_*                                                            */
    int32_t blk;        /* block index for FUSG_OUT_D2S_BLOCK                                    */
    int32_t reserved;
} fusg_conv_out;

/*
 * One fused convolution: MyConv2d (vunet/layers.py:21-39) together with whatever the reference
 * wraps around it -- channel concat of two inputs (torch.cat([x, skip], 1)), bias, residual add
 * (Residual, layers.py:98-102), Sampler noise (layers.py:163-167), ELU of the result for the next
 * pre-activated layer (Activation, layers.py:6-18), DepthToSpace / SpaceToDepth addressing
 * (layers.py:173-221).  Activations are NHWC; a channel-sliced view is expressed by pitch > c.
 */
typedef struct fusg_conv_desc {
    const void *in0, *in1;      /* NHWC inputs, activation dtype; in1 may be NULL                */
    int32_t c0, c1;             /* channels read from in0 / in1 (multiples of 16 for tcgen05)    */
    int32_t pitch0, pitch1;     /* elements between consecutive pixels (>= c)                    */
    int32_t B, H, W;            /* input batch / height / width                                  */
    int32_t ksize, stride;      /* 1 or 3 (padding ksize/2), 1..7 with pad_mode = 1; 1 or 2      */
    const void *weight;         /* [cout_pad][ksize*ksize][c0+c1], activation dtype (folded w_norm) */
    const float *bias;          /* [cout_pad] fp32                                               */
    int32_t cout, cout_pad;     /* real / stored output channels                                 */
    const void *residual;       /* NHWC [B,Ho,Wo,cout] activation dtype, or NULL                 */
    const float *noise;         /* NHWC fp32 [B,Ho,Wo,cout] or NULL                              */
    fusg_conv_out outs[FUSG_CONV_MAX_OUTS];
    int32_t dtype;              /* FUSG_DTYPE_*                                                  */
    int32_t impl;               /* FUSG_IMPL_*                                                   */
    uint64_t zero_kblocks;      /* optional hint: bit (tap * chunks + chunk) set = the weights of that 64-channel
                                 * k-block (chunks = (c0+c1)/64, in0 chunks first) are all zero and the kernel
                                 * may skip it; 0 = no hint.  Never changes the result.              */
    int32_t pad_mode;           /* 0: zero padding of ksize/2 (VUNet).  1: explicit padding `pad` whose VALUES are
                                 * stored in the input tensor itself: in0/in1 are [B, H+2*border, W+2*border, pitch]
                                 * with the logical image at offset (border, border) and border >= pad -- how the
                                 * ICN's ReflectionPad2d convolutions (warp_learn/models.py:43-46,86) are fed  */
    int32_t pad, border;        /* pad_mode 1 only                                                  */
    int32_t cphys0, cphys1;     /* 0, or the number of channels in0 / in1 really hold (< c0 / c1, multiple of 8): channels
                                 * cphys..c-1 read as zero.  The network inputs (6 / 3 real channels) are stored 16 wide and
                                 * widened to a 64- / 32-channel K block by TMA's out-of-bounds zero fill instead of in HBM  */
    int32_t cin_real;           /* optional hint: the number of REAL input channels of in0 when it is smaller than c0 / cphys0 (the
                                 * rest is zero padding whose weights are zero); 0 = unknown.  Lets FUSG_IMPL_AUTO pick FUSG_IMPL_SMALLCIN. */
} fusg_conv_desc;

int fusg_conv2d(const fusg_conv_desc *desc, void *stream);
/* sizeof(fusg_conv_desc) as this library was compiled (binding self-check). */
size_t fusg_sizeof_conv_desc(void);
/* Which kernel FUSG_IMPL_AUTO resolves to for this descriptor (FUSG_IMPL_SMALLCIN, FUSG_IMPL_TCGEN05 or FUSG_IMPL_DIRECT). */
int fusg_conv2d_select(const fusg_conv_desc *desc);
/* Diagnostics: the tiling plan of the calling thread's last tcgen05 launch --
 * plan8 = {msub (128-row sub-tiles per CTA tile), pair (cta_group::2), halo (sliding-window A tiles), ksplit (split-K
 * cluster size), stages, group (k-blocks per barrier round trip), w_resident, fast_epi}.  Tests use it to assert that
 * a case really exercises the variant it is named after. */
void fusg_conv2d_last_plan(int32_t *plan8_host);
/* Persistent conv grids use (SM count - n) CTAs from now on (process-wide; returns the previous value; n < 0 only queries).
 * A pipeline that runs another kernel family next to the convolutions (NovelViewPipeline: the homography solver of the
 * warp stage) reserves a few SMs for it: a persistent CTA that cannot be placed doubles its layer's time.  Default 0. */
int fusg_conv2d_set_sm_reserve(int n);

/* weight_norm fold (vunet/layers.py:29-31): w = g * v / ||v||, repacked from [cout][cin][k][k]
 * fp32 to [cout_pad][k*k][cin_pad] in `dtype` (zero padded).  Run once per load_state_dict. */
int fusg_fold_weightnorm(const float *v, const float *g, void *w_out, int cout, int cin, int ksize,
                         int cout_pad, int cin_pad, int dtype, void *stream);

/* Same fold, for running a narrow stride-1 layer on PIXEL PAIRS: an NHWC tensor [B,H,W,c] is
 * bit-identical to [B,H,W/2,2c], so a k x k convolution c0(+c1) -> cout over W pixels equals a
 * k x 3 (3x3) or 1x1 convolution 2c0(+2c1) -> 2cout over W/2 pixel pairs whose weight matrix holds
 * the original taps at kx = 2s + h - dx + 1 (pair shift s, input half h, output half dx) and zeros
 * elsewhere.  Twice the bytes per TMA row and half the rows per pixel for the 32-channel layers.
 * w_out: [cout_pad][k*k][2*(cin0+cin1)], bias_out: [cout_pad] (bias duplicated per half). */
int fusg_fold_weightnorm_paired(const float *v, const float *g, const float *bias, void *w_out, float *bias_out,
                                int cout, int cin0, int cin1, int ksize, int cout_pad, int dtype, void *stream);

/* NCHW fp32 [B,C,H,W] -> NHWC [B,H,W,cpad] in `dtype` (zero padded channels), optional ELU. */
int fusg_nchw_to_nhwc(const float *in, void *out, int B, int C, int H, int W, int cpad, int elu, int dtype, void *stream);
/* NHWC `dtype` [B,H,W,pitch] (first C channels) -> NCHW fp32 [B,C,H,W]. */
int fusg_nhwc_to_nchw(const void *in, float *out, int B, int C, int H, int W, int pitch, int dtype, void *stream);
/* to_image (warp_learn/planes_utils.py:96-118, from_LAB=False): NCHW fp32 in [-1,1] ->
 * HWC uint8, x = clip((x + 1) / 2 * 255, 0, 255) with the reference's truncating cast.
 *   in [B,3,H,W] f32 -> out [B,H,W,3] u8 */
int fusg_to_image(const float *in, uint8_t *out, int B, int H, int W, void *stream);
/* to_image(..., from_LAB=True) (warp_learn/planes_utils.py:96-118; the ICN's output, trajectory_inference.py:182,391): the same
 * float -> uint8 step, then cv2.cvtColor(COLOR_LAB2BGR) on uint8 -- OpenCV's integer pipeline, bit-exact on all 2^24 (L,a,b) triples.
 *   in [B,3,H,W] f32 (Lab in [-1,1]) -> out [B,H,W,3] u8 BGR; lab_to_yf [512] u16 and inv_gamma [4096] u8 from
 *   future_urban_scene_generation_b200/data/lab8.npz (scripts/make_lab_tables.py), in device memory. */
int fusg_to_image_lab(const float *in, uint8_t *out, const uint16_t *lab_to_yf, const uint8_t *inv_gamma, int B, int H, int W, void *stream);
/* ---- paste-back of completed crops into frames (SURVEY.md section 8f-2) --------------------------------------
 * cv2.resize(src, dsize) with INTER_LINEAR on 8-bit, 3-channel HWC images, batched: item i reads src + src_off[i]
 * ([src_hw[2i], src_hw[2i+1], 3]) and writes dst + dst_off[i] ([dst_hw[2i], dst_hw[2i+1], 3]); offsets in bytes,
 * all arrays in device memory.  Replaces cv2.resize at trajectory_inference.py:191,243,400,435. */
int fusg_resize_u8(const uint8_t *src, const long long *src_off, const int32_t *src_hw, uint8_t *dst, const long long *dst_off,
                   const int32_t *dst_hw, int B, int max_dst_pixels, void *stream);
size_t fusg_paste_workspace_bytes(int F, int Hf, int Wf);
/* The five lines after each network forward (trajectory_inference.py:236-250): for item b = 0..B-1 in order,
 *   crop_inv = resize(crops[b] (S,S,3), (w_orig, h_orig))[pad_y0 : h_orig - pad_y1, pad_x0 : w_orig - pad_x1]
 *   frames[frame][mask_b] = (zeros with crop_inv placed at (x_min, y_min))[mask_b]
 * info [B,9] int32 = frame, h_orig, w_orig, pad_x0, pad_y0, pad_x1, pad_y1, x_min, y_min (crop_info of
 * warp_learn/models.py:337-342); the mask of item b is the uint8 array masks + mask_off[b] of shape
 * (mask_rect[4b+3], mask_rect[4b+2]) placed at frame position (x, y) = (mask_rect[4b], mask_rect[4b+1]) -- a full-frame
 * dst_sketch_mask is rect (0, 0, Wf, Hf).  Later items win where masks overlap, as in the sequential reference.
 * frames [F,Hf,Wf,3] u8 is updated in place. */
int fusg_paste_back(uint8_t *frames, const uint8_t *crops, const uint8_t *masks, const long long *mask_off, const int32_t *mask_rect,
                    const int32_t *info, void *workspace, size_t workspace_bytes, int B, int F, int Hf, int Wf, int S,
                    int max_mask_pixels, void *stream);
/* ---- VUNet input packing (SURVEY.md section 8f-3; trajectory_inference.py:205-227, :414-421) -----------------
 * Item b owns a rectangle rect[4b..] = (x, y, w, h) of frame frame_idx[b]; inside it: a uint8 vehicle mask (non-zero =
 * vehicle, i.e. logical_not(src_sketch_mask)) at masks + off[b], and two uint8 RGB normal sketches at
 * normal_* + 3*off[b]; outside it everything is background (0).  A full-frame item has rect (0, 0, Wf, Hf).
 * fusg_mask_bbox: bbox[b] = (x_min, y_min, x_max, y_max) of the vehicle pixels in frame coordinates
 *   (np.nonzero + min/max at trajectory_inference.py:207-209); an empty mask gives (INT_MAX, INT_MAX, -1, -1). */
int fusg_mask_bbox(const uint8_t *masks, const long long *mask_off, const int32_t *mask_rect, int32_t *bbox, int B, int max_mask_pixels,
                   void *stream);
/* x [B,6,res,res] f32 = cat(to_tensor(resize(square_crop(mask * frame)) with background -> 255),
 *                           to_tensor(resize(square_crop(normal_src))[..., ::-1]));
 * y [B,3,res,res] f32 = to_tensor(resize(square_crop(normal_dst))[..., ::-1])
 * with square_crop = utils/crop_utils.py:4-52 on bbox[b], resize = cv2.resize(..., (res, res)), background = pixels whose
 * resized source normal is (0,0,0), to_tensor = utils/misc_utils.py:35-50.  frames [F,Hf,Wf,3] u8. */
int fusg_pack_vunet_inputs(const uint8_t *frames, const int32_t *frame_idx, const uint8_t *masks, const uint8_t *normal_src,
                           const uint8_t *normal_dst, const long long *off, const int32_t *rect, const int32_t *bbox, float *x, float *y,
                           int B, int Hf, int Wf, int res, void *stream);
/* ---- ICN input packing (SURVEY.md section 8f-1; warp_learn/models.py:323-366 get_icn_inputs) --------------------------------
 * Item b: planes [B,5,Hf,Wf,3] u8 (the warped planes, BGR -- fusg_warp_fused's `warped` for whole frames), normals [B,Hf,Wf,3] u8
 * (destination normal sketch, RGB), central [B,res,res,3] u8 (central crop, RGB), bbox[b] = bounding box of the sketch mask
 * (fusg_mask_bbox).  out [B,21,res,res] f32 = cat(Lab(resize(square_crop(normal))), Lab(central), Lab(resize(square_crop(plane_k))) k=0..4)
 * with square_crop = utils/crop_utils.py:4-52, resize = cv2.resize(..., (res,res)), Lab = cv2.cvtColor(COLOR_RGB2LAB / COLOR_BGR2LAB) on
 * uint8, then ToTensor + Normalize(0.5, 0.5).  The Lab tables (gamma_tab [256] u16, cbrt_tab [3072] u16) and the sorted exception list
 * (exc_keys [n_exc] u32 = R<<16|G<<8|B, exc_vals [n_exc] u16 = a<<8|b) come from future_urban_scene_generation_b200/data/lab8.npz,
 * generated and verified against cv2 on all 2^24 colours by scripts/make_lab_tables.py; exc_bitmap (may be NULL): [2^19] u32, bit
 * (key & 31) of word (key >> 5) set iff key is in exc_keys -- lets 9,999 of 10,000 pixels skip the list search; all in device memory. */
int fusg_pack_icn_inputs(const uint8_t *planes, const uint8_t *normals, const uint8_t *central, const int32_t *bbox,
                         const uint16_t *gamma_tab, const uint16_t *cbrt_tab, const uint32_t *exc_keys, const uint16_t *exc_vals, int n_exc,
                         const uint32_t *exc_bitmap, float *out, int B, int Hf, int Wf, int res, void *stream);
/* The same packing with the warped planes as fusg_warp_fused_window writes them: item b's five planes are the frame window
 * win[b] = (x0, y0, w, h) at planes + win_off[b] (plane k = [h,w,3] u8 at byte k*h*w*3).  The window must hold the square crop of
 * bbox[b] clipped to the Hf x Wf frame (every pixel the crop reads); then out equals fusg_pack_icn_inputs on the whole-frame planes
 * bit for bit.  Every other argument as there. */
int fusg_pack_icn_inputs_window(const uint8_t *planes, const int32_t *win, const long long *win_off, const uint8_t *normals,
                                const uint8_t *central, const int32_t *bbox, const uint16_t *gamma_tab, const uint16_t *cbrt_tab,
                                const uint32_t *exc_keys, const uint16_t *exc_vals, int n_exc, const uint32_t *exc_bitmap, float *out,
                                int B, int Hf, int Wf, int res, void *stream);
/* The tail of the same assembly when the three 256x256 uint8 images already exist (trajectory_inference.py:221-225):
 *   x = cat(to_tensor(mask_bbox), to_tensor(normal_src[..., ::-1])), y = to_tensor(normal_dst[..., ::-1]);
 * inputs [B,res,res,3] u8 -> x [B,6,res,res] f32, y [B,3,res,res] f32.  Lets a host ship 9 bytes per pixel instead of 36. */
int fusg_u8_to_vunet_inputs(const uint8_t *mask_bbox, const uint8_t *normal_src, const uint8_t *normal_dst, float *x, float *y, int B,
                            int res, void *stream);
/* y alone, for a step whose appearance input was encoded beforehand (the trajectory loop, trajectory_inference.py:413-426):
 *   normal_dst [B,res,res,3] u8 -> y [B,3,res,res] f32, the same values fusg_u8_to_vunet_inputs writes to y. */
int fusg_u8_to_vunet_y(const uint8_t *normal_dst, float *y, int B, int res, void *stream);
/* ---- per-item gather of per-vehicle rows --------------------------------------------------------------------
 * For every segment: dst [B,row_bytes] row b = src [n_src,row_bytes] row index[b], or zeros where index[b] is outside
 * [0, n_src).  index [B] i32 (device).  `segs` is a HOST array of nseg <= FUSG_GATHER_MAX_SEGS entries, passed to the kernel
 * by value (one launch, capturable in a graph).  row_bytes must be a non-zero multiple of 16 and src / dst 16-byte aligned
 * (copies are 16-byte vectors); anything else is FUSG_ERR_ARG.  Brings a vehicle's cached appearance tensors to its items. */
#define FUSG_GATHER_MAX_SEGS 8
typedef struct fusg_gather_seg {
    const void *src;
    void *dst;
    int64_t row_bytes;
    int32_t n_src;
    int32_t reserved;
} fusg_gather_seg;
int fusg_gather_rows(const fusg_gather_seg *segs, int nseg, const int32_t *index, int B, void *stream);
/* sizeof(fusg_gather_seg) as this library was compiled (binding self-check). */
size_t fusg_sizeof_gather_seg(void);
/* ====================================================================================== */
/* ICN generator G_Resnet (SURVEY.md section 8f-1; warp_learn/models.py:15-208): the pieces   */
/* between its convolutions.  The convolutions themselves run on fusg_conv2d (pad_mode 1).    */
/* ====================================================================================== */

/* NCHW fp32 [B,C,H,W] -> NHWC [B, H+2*border, W+2*border, cpad] in `dtype`, channels zero padded, the border filled
 * by reflection (nn.ReflectionPad2d, warp_learn/models.py:43-44): the input of the first 7x7 Conv2dBlock (:125-127). */
int fusg_nchw_to_nhwc_reflect(const float *in, void *out, int B, int C, int H, int W, int cpad, int border, int dtype, void *stream);

/* Per-(sample, channel) partial sums of an NHWC [B,HW,C] tensor: partial = [B, nsplit, C, 2] fp32 (sum, sum of squares) of
 * (x - k) over the pixels of split s, followed by [B, C] fp32 shifts k = x[b, pixel 0, c] -- B*nsplit*C*2 + B*C floats in all.
 * The shift keeps the one-pass variance free of cancellation when |mean| >> std.  C a multiple of 8 and <= 256;
 * deterministic (no atomics). */
int fusg_norm_stats(const void *x, float *partial, int B, int HW, int C, int nsplit, int dtype, void *stream);

/* Folds the partial sums (layout above, written by fusg_norm_stats) into per-(sample, channel) scale/shift pairs, ss [B,C,2] fp32, y = x*scale + shift:
 *   kind 0  nn.InstanceNorm2d(affine=False, eps) (warp_learn/models.py:55-56): per (b,c) biased variance,
 *           scale = 1/sqrt(var + eps), shift = -mean*scale;
 *   kind 1  the reference's own LayerNorm (warp_learn/models.py:15-35): per sample over C*H*W, UNBIASED std,
 *           (x - mean)/(std + eps), then gamma[c], beta[c]. */
int fusg_norm_finalize(const float *partial, const float *gamma, const float *beta, float *ss, int B, int HW, int C, int nsplit,
                       int kind, float eps, void *stream);

/* out[b, Y, X, c] = act( x[b, sy, sx, c]*scale[b,c] + shift[b,c] (+ residual[b, sy+rb, sx+rb, c]) ) for every pixel of the
 * padded output [B, up*H + 2*border, up*W + 2*border, C]: (Y,X) -> reflect into the up*H x up*W image
 * (ReflectionPad2d) -> nearest-neighbour source pixel (sy,sx) = (y/up, x/up) (Upsample, warp_learn/models.py:138-147).
 * x [B,H,W,C]; residual (may be NULL) [B, H+2*rb, W+2*rb, C]; relu 0/1; up 1 or 2.  One launch = norm + activation +
 * residual add of a ResBlock (:98-102) + upsample + padding for the next convolution. */
int fusg_norm_apply(const void *x, const float *ss, const void *residual, int rb, void *out, int B, int H, int W, int C, int relu,
                    int up, int border, int dtype, void *stream);

/* NHWC elementwise ELU (activation dtype) over n elements. */
int fusg_elu(const void *in, void *out, size_t n, int dtype, void *stream);

/* ====================================================================================== */
/* Normal-sketch renderer (SURVEY.md section 8f-4)                                          */
/* ====================================================================================== */

/* Replaces warp_learn/render_open3d.py:29-50 `get_rendered(model_ply, w, h, extrinsic, intrinsic)` (Open3D's OpenGL
 * visualiser: vertex colours (vertex_normal + 1) / 2, lighting off, black background) for B items of ONE mesh, each with
 * its own camera and -- as the trajectory loop does, trajectory_inference.py:363 `orig_vertices @ z_rot(theta) + tr` --
 * its own rigid move.
 *   verts [Nv,3] f64, tris [Nt,3] i32;
 *   adj_off [Nv+1], adj_tri [3*Nt] i32: CSR vertex -> incident triangles in ascending triangle order (host, once per mesh);
 *   rot [B,9] f64 row-major (v @ rot) or NULL, tr [B,3] f64 or NULL (tr needs rot);
 *   E [B,12] f64 world->camera 3x4, K [B,9] f64 (fx, fy are read; the principal point is the window centre
 *   (W/2 - 0.5, H/2 - 0.5) like Open3D's view control keeps it, render_open3d.py:19-22);
 *   normals [B,H,W,3] u8 RGB, mask [B,H,W] u8 (1 = background, the reference's `object_mask`);
 *   workspace >= fusg_render_workspace_bytes(B, Nv, H, W).
 * Rasterisation rules (top-left fill, z-buffer ties, perspective-correct interpolation, round(c * 255)) are those of
 * oracle/render_oracle.py, which this entry point reproduces bit for bit. */
size_t fusg_render_workspace_bytes(int B, int Nv, int H, int W);
int fusg_render_normals(const double *verts, const int32_t *tris, const int32_t *adj_off, const int32_t *adj_tri, int Nv, int Nt,
                        const double *rot, const double *tr, const double *E, const double *K, uint8_t *normals, uint8_t *mask,
                        void *workspace, size_t workspace_bytes, int B, int H, int W, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FUSG_H_ */
