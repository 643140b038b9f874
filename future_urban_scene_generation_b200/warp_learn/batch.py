"""Batched fused planar warp: the fast path behind warp_learn (include/fusg.h: fusg_warp_fused).

One call covers, for B crops, what trajectory_inference.py:165-174 does per vehicle:
compute_visibility (source + destination pose) -> get_planes -> warp_unwarp_planes()[0].
"""
from dataclasses import dataclass

import numpy as np

from .. import _lib


@dataclass
class WarpResult:
    warped: "torch.Tensor"    # (B,5,H,W,3) uint8, device (a frame_ops.WindowedPlanes for warp_batch(..., window=))
    vis: "torch.Tensor"       # (B,2,7) uint8: [src|dst] x (left,right,roof,front,back,front_bt,back_bt)
    plane_j: "torch.Tensor"   # (B,5) int8: target plane of source plane i, -1 skipped, -2 refused (a vertex beyond 2^20 px)
    H12: "torch.Tensor"       # (B,5,3,3) float64 (zeros where skipped)


def _dev(torch, a, dtype, shape, device):
    t = torch.as_tensor(a) if not isinstance(a, torch.Tensor) else a
    if t.dtype != dtype:
        t = t.to(dtype)
    t = t.reshape(shape)
    if not t.is_cuda:
        t = t.to(device, non_blocking=True)
    return t.contiguous()


class RefusedCrops(ValueError):
    """Raised when the kernels refused crops (plane_j == -2): a plane vertex or projected keypoint lies beyond
    2^20 pixels, where neither cv2's int32 polygon rasteriser nor the 16.16 edge arithmetic is defined."""

    def __init__(self, indices, reason="fused warp refused {n} crop(s) (vertex magnitude > 2^20 px)"):
        super().__init__(f"{reason.format(n=len(indices))}: {indices[:8]}")
        self.indices = indices


def check_refused(result: "WarpResult"):
    """Synchronises and raises RefusedCrops if any crop was refused.  The reference would warp or raise inside cv2 for
    such inputs; silently returning black planes is the one thing that must not happen."""
    torch = _lib.require_cuda()
    bad = torch.nonzero((result.plane_j == -2).any(dim=1)).flatten()
    if bad.numel():
        raise RefusedCrops(bad.cpu().tolist())
    return result


def warp_batch(src, src_kp, dst_kp, K, E_src, E_dst, kp3d, device=None, out=None, kp3d_dst=None, check=False,
               src_index=None, window=None) -> WarpResult:
    """src (B,H,W,3) u8; src_kp/dst_kp (B,12,2) i32 plane vertices (_KP_NAMES order, already
    truncated as in planes_utils.py:22-27); K (B,3,3) or (3,3); E_* (B,3,4) or (B,4,4); kp3d (B,12,3).
    numpy arrays or torch tensors on host or device.  Asynchronous on the current CUDA stream.
    kp3d_dst (B,12,3), optional: the destination pose's own keypoints (trajectory loop: same camera, moved keypoints,
    trajectory_inference.py:359-379 -- see kinematics.step_keypoints_batch); default: kp3d for both poses.
    Keypoints outside the frame are handled like cv2 does (clipped polygons).  check=True synchronises and raises
    RefusedCrops when a crop came back refused (plane_j == -2); asynchronous callers use check_refused(result)
    once the stream is done (NovelViewPipeline.result does).
    src_index (B,) int32, optional: crop b warps source image src_index[b] of src (n_src,H,W,3) -- one source crop per vehicle
    shared by all its steps (TrajectoryPipeline).  A host-side index is range-checked (ValueError); on the device an index
    outside [0, n_src) refuses that crop (plane_j == -2, zero planes).
    window (frame_ops.IcnWindows, optional): write only each item's ICN crop window (`frame_ops.icn_windows` of the destination
    sketch masks): `warped` is then a frame_ops.WindowedPlanes whose item(b) equals the whole-frame warped[b] cropped to the window
    bit for bit (vis / plane_j / H12 unchanged), for any frame size.  Made for whole frames, where the ICN reads a small square of
    each plane; get_icn_inputs_batch takes it in place of the (B,5,H,W,3) planes.
    window may also be a frame_ops.CropGeometry built with a window_capacity: the windows then stay on the device, `warped` spans
    capacity_bytes bytes, the kernel runs with max_win_h, and an item the geometry refused is refused here (plane_j == -2, none of
    its bytes written) -- no host round trip, so the call can be captured in a CUDA graph."""
    torch = _lib.require_cuda()
    device = torch.device(device if device is not None else "cuda")
    src = _dev(torch, src, torch.uint8, src.shape, device)
    n_src, H, W, ch = src.shape
    if ch != 3:
        raise ValueError("src must be (B,H,W,3) uint8")
    B = n_src
    idx = None
    if src_index is not None:
        it = torch.as_tensor(src_index) if not isinstance(src_index, torch.Tensor) else src_index
        if it.dim() != 1:
            raise ValueError("src_index must be a (B,) integer array")
        if not it.is_cuda and it.numel() and (int(it.min()) < 0 or int(it.max()) >= n_src):
            raise ValueError(f"src_index out of range [0, {n_src})")
        B = int(it.shape[0])
        if B <= 0:
            raise ValueError("src_index is empty")
        idx = _dev(torch, it, torch.int32, (B,), device)

    def _E(E):
        E = torch.as_tensor(E) if not isinstance(E, torch.Tensor) else E
        if E.shape[-2:] == (4, 4):
            E = E[..., :3, :]
        return _dev(torch, E, torch.float64, (B, 3, 4), device)

    Kt = torch.as_tensor(K) if not isinstance(K, torch.Tensor) else K
    if Kt.dim() == 2:
        Kt = Kt.unsqueeze(0).expand(B, 3, 3)
    Kt = _dev(torch, Kt, torch.float64, (B, 3, 3), device)
    Es, Ed = _E(E_src), _E(E_dst)
    X = _dev(torch, kp3d, torch.float64, (B, 12, 3), device)
    skp = _dev(torch, src_kp, torch.int32, (B, 12, 2), device)
    dkp = _dev(torch, dst_kp, torch.int32, (B, 12, 2), device)
    if window is not None:
        if len(window) != B or window.frame_hw != (H, W):
            raise ValueError(f"warp_batch: the windows are for {len(window)} items on {window.frame_hw} frames, the call has {B} on {(H, W)}")
        if window.nbytes <= 0:
            raise ValueError("warp_batch: the crop geometry was built without a window_capacity")
        win_rect, win_off = window.rect_dev.to(device), window.off_dev.to(device)
    if out is None:
        if window is None:
            warped = torch.empty((B, 5, H, W, 3), dtype=torch.uint8, device=device)
        else:
            from ..frame_ops import WindowedPlanes
            warped = WindowedPlanes(torch.empty((window.nbytes,), dtype=torch.uint8, device=device), window)
        out = WarpResult(
            warped=warped,
            vis=torch.empty((B, 2, 7), dtype=torch.uint8, device=device),
            plane_j=torch.empty((B, 5), dtype=torch.int8, device=device),
            H12=torch.empty((B, 5, 3, 3), dtype=torch.float64, device=device))
    L = _lib.lib()
    ws_bytes = L.fusg_warp_workspace_bytes_hw(B, H, W) if window is None else L.fusg_warp_window_workspace_bytes(B, H, W)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=device)
    Xd = _dev(torch, kp3d_dst, torch.float64, (B, 12, 3), device) if kp3d_dst is not None else None
    with torch.cuda.device(device):
        if window is not None:
            rc = L.fusg_warp_fused_window(_lib.ptr(src), _lib.ptr(idx), n_src, _lib.ptr(skp), _lib.ptr(dkp), _lib.ptr(Kt), _lib.ptr(Es),
                                          _lib.ptr(Ed), _lib.ptr(X), _lib.ptr(Xd), _lib.ptr(win_rect), _lib.ptr(win_off),
                                          window.max_h, _lib.ptr(out.warped.data), _lib.ptr(out.vis), _lib.ptr(out.plane_j),
                                          _lib.ptr(out.H12), _lib.ptr(ws), ws_bytes, B, H, W, _lib.stream_ptr(torch))
        elif idx is not None:
            rc = L.fusg_warp_fused_idx(_lib.ptr(src), _lib.ptr(idx), n_src, _lib.ptr(skp), _lib.ptr(dkp), _lib.ptr(Kt), _lib.ptr(Es),
                                       _lib.ptr(Ed), _lib.ptr(X), _lib.ptr(Xd), _lib.ptr(out.warped), _lib.ptr(out.vis),
                                       _lib.ptr(out.plane_j), _lib.ptr(out.H12), _lib.ptr(ws), ws_bytes, B, H, W, _lib.stream_ptr(torch))
        elif Xd is None:
            rc = L.fusg_warp_fused(_lib.ptr(src), _lib.ptr(skp), _lib.ptr(dkp), _lib.ptr(Kt), _lib.ptr(Es), _lib.ptr(Ed),
                                   _lib.ptr(X), _lib.ptr(out.warped), _lib.ptr(out.vis), _lib.ptr(out.plane_j),
                                   _lib.ptr(out.H12), _lib.ptr(ws), ws_bytes, B, H, W, _lib.stream_ptr(torch))
        else:
            rc = L.fusg_warp_fused_traj(_lib.ptr(src), _lib.ptr(skp), _lib.ptr(dkp), _lib.ptr(Kt), _lib.ptr(Es), _lib.ptr(Ed),
                                        _lib.ptr(X), _lib.ptr(Xd), _lib.ptr(out.warped), _lib.ptr(out.vis), _lib.ptr(out.plane_j),
                                        _lib.ptr(out.H12), _lib.ptr(ws), ws_bytes, B, H, W, _lib.stream_ptr(torch))
    _lib.check(rc, "fusg_warp_fused")
    # keep inputs/workspace alive until the stream has consumed them
    out._keep = (src, skp, dkp, Kt, Es, Ed, X, Xd, ws, idx) + ((win_rect, win_off) if window is not None else ())
    return check_refused(out) if check else out
