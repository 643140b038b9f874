"""Paste-back of completed vehicle crops into video frames on the GPU (SURVEY.md section 8f-2).

Mirrors what `trajectory_inference.py` does after each network forward (:184-198 ICN, :236-250 VUNet, :393-407 and
:428-442 in the trajectory loop):

    crop_inv = cv2.resize(net_image, crop_size_orig[::-1])
    crop_inv = crop_inv[pad_xy_before[1]:crop_inv.shape[0] - pad_xy_after[1],
                        pad_xy_before[0]:crop_inv.shape[1] - pad_xy_after[0]]
    out_frame = np.zeros_like(frame)
    out_frame[crop_xy_min[1]: ..., crop_xy_min[0]: ...] = crop_inv
    img_output[dst_sketch_mask] = out_frame[dst_sketch_mask]

`paste_back` is the one-vehicle drop-in (numpy in / numpy out, same arguments as the reference's local variables),
`paste_back_batch` the form a maintainer adopts: every (vehicle, step) of a clip in one call, crops taken straight
from `to_image_batch` on the device, bit-identical to the sequential reference loop (last vehicle wins where masks
overlap).  `resize` is cv2.resize(img, dsize) for uint8 HWC images.  No CPU fallback.
"""
import ctypes as C

import numpy as np

from . import _lib

INFO_FIELDS = 9      # frame, h_orig, w_orig, pad_x0, pad_y0, pad_x1, pad_y1, x_min, y_min


def _dev(torch, a, dtype=None):
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.cuda().contiguous()


def resize_batch(images, dsizes):
    """images: list of uint8 (h, w, 3) arrays / tensors; dsizes: list of (width, height) like cv2.
    Returns a list of uint8 CUDA tensors (height, width, 3) == cv2.resize(image, dsize) (INTER_LINEAR)."""
    torch = _lib.require_cuda()
    assert len(images) == len(dsizes) and len(images) > 0
    srcs = [_dev(torch, im, torch.uint8) for im in images]
    for s in srcs:
        if s.dim() != 3 or s.shape[2] != 3 or s.shape[0] < 1 or s.shape[1] < 1:
            raise ValueError("resize_batch: images must be (h, w, 3) uint8")
    src_off, dst_off, so, do = [], [], 0, 0
    for s, (dw, dh) in zip(srcs, dsizes):
        if dw < 1 or dh < 1:
            raise ValueError("resize_batch: empty destination size")
        src_off.append(so)
        dst_off.append(do)
        so += s.numel()
        do += int(dh) * int(dw) * 3
    src = torch.cat([s.reshape(-1) for s in srcs])
    dst = torch.empty((do,), dtype=torch.uint8, device=src.device)
    src_hw = torch.tensor([[s.shape[0], s.shape[1]] for s in srcs], dtype=torch.int32, device=src.device)
    dst_hw = torch.tensor([[int(dh), int(dw)] for dw, dh in dsizes], dtype=torch.int32, device=src.device)
    t_so = torch.tensor(src_off, dtype=torch.int64, device=src.device)
    t_do = torch.tensor(dst_off, dtype=torch.int64, device=src.device)
    mx = max(int(dh) * int(dw) for dw, dh in dsizes)
    _lib.check(_lib.lib().fusg_resize_u8(_lib.ptr(src), _lib.ptr(t_so), _lib.ptr(src_hw), _lib.ptr(dst), _lib.ptr(t_do), _lib.ptr(dst_hw),
                                         len(srcs), mx, _lib.stream_ptr(torch)), "fusg_resize_u8")
    return [dst[o:o + int(dh) * int(dw) * 3].view(int(dh), int(dw), 3) for o, (dw, dh) in zip(dst_off, dsizes)]


def resize(image, dsize):
    """cv2.resize(image, dsize) for a uint8 (h, w, 3) numpy image; returns numpy."""
    return resize_batch([image], [dsize])[0].cpu().numpy()


def pack_crop_info(crop_infos, frame_index, frame_hw):
    """crop_info dicts (warp_learn/models.py:337-342) + frame index per item -> (B, 9) int32 for fusg_paste_back.
    Raises ValueError where the reference's slice assignment would raise (the un-padded crop must fit the frame)."""
    Hf, Wf = frame_hw
    out = np.zeros((len(crop_infos), INFO_FIELDS), np.int32)
    for b, (ci, fr) in enumerate(zip(crop_infos, frame_index)):
        h, w = (int(v) for v in ci["crop_size_orig"])
        px0, py0 = (int(v) for v in ci["pad_xy_before"])
        px1, py1 = (int(v) for v in ci["pad_xy_after"])
        x_min, y_min = (int(v) for v in ci["crop_xy_min"])
        ch, cw = h - py0 - py1, w - px0 - px1
        if h < 1 or w < 1 or min(px0, py0, px1, py1) < 0 or ch < 1 or cw < 1:
            raise ValueError(f"paste_back: item {b}: empty crop after un-padding")
        if x_min < 0 or y_min < 0 or y_min + ch > Hf or x_min + cw > Wf:
            raise ValueError(f"paste_back: item {b}: crop of shape {(ch, cw)} at {(x_min, y_min)} does not fit the {(Hf, Wf)} frame")
        out[b] = (fr, h, w, px0, py0, px1, py1, x_min, y_min)
    return out


class PastePlan:
    """Device-side description of a batch of paste-back items (masks, rectangles, crop geometry), built once by
    `prepare_paste` and reusable for any frames / crops tensors of the same layout."""

    def __init__(self, masks, off, rect, info, max_mask_pixels, B, frame_hw):
        self.masks, self.off, self.rect, self.info = masks, off, rect, info
        self.max_mask_pixels, self.B, self.frame_hw = max_mask_pixels, B, frame_hw

    @classmethod
    def from_geometry(cls, geometry, vehicle_masks):
        """The plan of `geometry`'s items (crop_geometry): item b pastes into frame geometry.frame_index[b] inside
        vehicle_masks[b] ((B, Hf, Wf) bool / uint8, non-zero = vehicle).  Built with device ops only (capturable); an item with a
        non-zero status pastes nothing, so its frame pixels stay as they were.  Frame indices are not range-checked here."""
        torch = _lib.require_cuda()
        B, (Hf, Wf) = len(geometry), geometry.frame_hw
        if tuple(vehicle_masks.shape) != (B, Hf, Wf):
            raise ValueError(f"paste_back: vehicle_masks are {tuple(vehicle_masks.shape)}, expected {(B, Hf, Wf)}")
        dev = geometry.info.device
        mk = vehicle_masks if isinstance(vehicle_masks, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(vehicle_masks))
        mk = (mk.view(torch.uint8) if mk.dtype == torch.bool else (mk != 0).to(torch.uint8)).to(dev).contiguous().reshape(-1)
        off, rect = _full_frame_rects(torch, B, Hf, Wf, dev)
        rect = rect * (geometry.status == 0).to(torch.int32).view(B, 1)      # a refused item covers no pixel
        return cls(mk, off, rect, geometry.info, Hf * Wf, B, (Hf, Wf))


def prepare_paste(masks, crop_infos, frame_index, frame_hw, n_frames, mask_rects=None):
    torch = _lib.require_cuda()
    Hf, Wf = frame_hw
    B = len(masks)
    if not (len(crop_infos) == len(frame_index) == B) or B == 0:
        raise ValueError("paste_back: one mask / crop_info / frame index per crop")
    if any(f < 0 or f >= n_frames for f in frame_index):
        raise ValueError("paste_back: frame index out of range")
    info = pack_crop_info(crop_infos, frame_index, (Hf, Wf))
    if isinstance(masks, torch.Tensor) and mask_rects is None:
        # stacked full-frame masks (B, Hf, Wf), e.g. already on the device: no per-item work on the host
        if tuple(masks.shape) != (B, Hf, Wf):
            raise ValueError(f"paste_back: stacked masks are {tuple(masks.shape)}, expected {(B, Hf, Wf)}")
        mflat = (masks.view(torch.uint8) if masks.dtype == torch.bool else (masks != 0).to(torch.uint8)).contiguous().reshape(-1).cuda()
        dev = mflat.device
        rect_t = torch.tensor([0, 0, Wf, Hf], dtype=torch.int32, device=dev).repeat(B, 1)
        return PastePlan(mflat, torch.arange(B, dtype=torch.int64, device=dev) * (Hf * Wf), rect_t, torch.from_numpy(info).to(dev), Hf * Wf, B, (Hf, Wf))
    rects = np.zeros((B, 4), np.int32)
    offs, flat, o = [], [], 0
    for b, m in enumerate(masks):
        mt = m if isinstance(m, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(m))
        if mt.dtype == torch.bool:
            mt = mt.view(torch.uint8)                      # numpy/torch bools are one byte, 0 or 1
        elif mt.dtype != torch.uint8:
            mt = (mt != 0).to(torch.uint8)
        if mask_rects is None:
            if tuple(mt.shape) != (Hf, Wf):
                raise ValueError(f"paste_back: mask {b} is {tuple(mt.shape)}, frame is {(Hf, Wf)}")
            rects[b] = (0, 0, Wf, Hf)
        else:
            x, y, w, h = (int(v) for v in mask_rects[b])
            if tuple(mt.shape) != (h, w):
                raise ValueError(f"paste_back: mask {b} is {tuple(mt.shape)}, its rect says {(h, w)}")
            rects[b] = (x, y, w, h)
        offs.append(o)
        flat.append(mt.reshape(-1))
        o += mt.numel()
    mflat = torch.cat(flat).cuda()                         # one H2D for all host masks
    dev = mflat.device
    return PastePlan(mflat, torch.tensor(offs, dtype=torch.int64, device=dev), torch.from_numpy(rects).to(dev),
                     torch.from_numpy(info).to(dev), int((rects[:, 2].astype(np.int64) * rects[:, 3]).max()), B, (Hf, Wf))


def paste_back_packed(frames, crops, plan: PastePlan):
    """frames (F, Hf, Wf, 3) uint8 CUDA tensor, updated in place; crops (B, S, S, 3) uint8 CUDA tensor."""
    torch = _lib.require_cuda()
    F, Hf, Wf = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    B, S = int(crops.shape[0]), int(crops.shape[1])
    if frames.dim() != 4 or frames.shape[3] != 3 or (Hf, Wf) != plan.frame_hw or frames.dtype != torch.uint8:
        raise ValueError("paste_back: frames must be (F, Hf, Wf, 3) uint8 matching the plan")
    if crops.dim() != 4 or crops.shape[2] != S or crops.shape[3] != 3 or B != plan.B or crops.dtype != torch.uint8:
        raise ValueError("paste_back: crops must be (B, S, S, 3) uint8 with one crop per planned item")
    L = _lib.lib()
    ws_bytes = L.fusg_paste_workspace_bytes(F, Hf, Wf)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=frames.device)
    _lib.check(L.fusg_paste_back(_lib.ptr(frames), _lib.ptr(crops), _lib.ptr(plan.masks), _lib.ptr(plan.off), _lib.ptr(plan.rect),
                                 _lib.ptr(plan.info), _lib.ptr(ws), ws_bytes, B, F, Hf, Wf, S, plan.max_mask_pixels,
                                 _lib.stream_ptr(torch)), "fusg_paste_back")
    return frames


def paste_back_batch(frames, crops, masks, crop_infos, frame_index, mask_rects=None):
    """frames: (F, Hf, Wf, 3) uint8 CUDA tensor, updated in place (or numpy -> a new CUDA tensor is returned);
    crops: (B, S, S, 3) uint8 (the `to_image_batch` output); masks: list of B bool/uint8 arrays -- full-frame
    `dst_sketch_mask`s, or sub-rectangles when `mask_rects` [(x, y, w, h)] is given; crop_infos: list of B dicts;
    frame_index: list of B ints.  Items are applied in list order (later items win), like the reference loop."""
    torch = _lib.require_cuda()
    fr = _dev(torch, frames, torch.uint8)
    if fr.dim() != 4 or fr.shape[3] != 3:
        raise ValueError("paste_back_batch: frames must be (F, Hf, Wf, 3) uint8")
    cr = _dev(torch, crops, torch.uint8)
    plan = prepare_paste(masks, crop_infos, frame_index, (int(fr.shape[1]), int(fr.shape[2])), int(fr.shape[0]), mask_rects)
    return paste_back_packed(fr, cr, plan)


def paste_back(img_output, net_image, crop_info, dst_sketch_mask):
    """One vehicle, reference-style: numpy (H, W, 3) uint8 `img_output` is updated in place and returned."""
    out = paste_back_batch(img_output[None], np.asarray(net_image)[None], [dst_sketch_mask], [crop_info], [0])
    img_output[...] = out[0].cpu().numpy()
    return img_output


# ---------------------------------------------------------------------------------------------------------------
# VUNet input packing (SURVEY.md 8f-3): trajectory_inference.py:205-227 / :414-421 on the device
# ---------------------------------------------------------------------------------------------------------------
def pack_vunet_inputs_batch(frames, frame_index, src_sketch_masks, src_sketch_normals, dst_sketch_normals, rects=None, res=256,
                            geometry=None):
    """frames: (F, Hf, Wf, 3) uint8; per item b: `src_sketch_masks[b]` bool (True = background, as the reference holds it
    at that point), `src_sketch_normals[b]` / `dst_sketch_normals[b]` uint8 (h, w, 3) -- full-frame arrays, or sub-rectangles
    `rects[b] = (x, y, w, h)` outside of which the item is background.  Returns CUDA tensors
    (x (B,6,res,res) f32, y_tilde (B,3,res,res) f32, bbox (B,4) int32) == the reference's `x`, `y_tilde` stacked.
    geometry (crop_geometry of the same vehicle masks, optional): the bboxes come from it -- no bbox pass, no synchronisation; the
    inputs must then be stacked full-frame tensors and frame_index a (B,) int32 CUDA tensor: the frame of `frames` each item is cut
    from (not the geometry's frame_index, which says where the item is pasted).  An item with a non-zero status, or whose frame
    index is outside [0, F), gets zero x and y rows -- the range is checked on the device, so the call stays capturable."""
    torch = _lib.require_cuda()
    fr = _dev(torch, frames, torch.uint8)
    if fr.dim() != 4 or fr.shape[3] != 3:
        raise ValueError("pack_vunet_inputs_batch: frames must be (F, Hf, Wf, 3) uint8")
    F, Hf, Wf = int(fr.shape[0]), int(fr.shape[1]), int(fr.shape[2])
    if geometry is not None:
        B = len(geometry)
        if geometry.frame_hw != (Hf, Wf) or rects is not None:
            raise ValueError(f"pack_vunet_inputs_batch: the geometry is for full {geometry.frame_hw} frames, the frames are {(Hf, Wf)}")
        if not (isinstance(frame_index, torch.Tensor) and frame_index.is_cuda and frame_index.dtype == torch.int32
                and tuple(frame_index.shape) == (B,)):
            raise ValueError("pack_vunet_inputs_batch: with a geometry, frame_index is a (B,) int32 CUDA tensor of source frames")
    else:
        B = len(frame_index)
    if B == 0 or not (len(src_sketch_masks) == len(src_sketch_normals) == len(dst_sketch_normals) == B):
        raise ValueError("pack_vunet_inputs_batch: one mask and two normal sketches per item")
    if geometry is None and any(f < 0 or f >= F for f in frame_index):
        raise ValueError("pack_vunet_inputs_batch: frame index out of range")
    if geometry is not None and not all(isinstance(a, torch.Tensor) and a.dim() == d
                                        for a, d in ((src_sketch_masks, 3), (src_sketch_normals, 4), (dst_sketch_normals, 4))):
        raise ValueError("pack_vunet_inputs_batch: with a geometry, the masks and normal sketches are stacked (B,Hf,Wf[,3]) tensors")
    if rects is None and all(isinstance(a, torch.Tensor) and a.dim() == d for a, d in ((src_sketch_masks, 3), (src_sketch_normals, 4), (dst_sketch_normals, 4))):
        # stacked full-frame tensors (B, Hf, Wf[, 3]), e.g. already on the device: no per-item work on the host
        if tuple(src_sketch_masks.shape) != (B, Hf, Wf) or tuple(src_sketch_normals.shape) != (B, Hf, Wf, 3) or tuple(dst_sketch_normals.shape) != (B, Hf, Wf, 3):
            raise ValueError("pack_vunet_inputs_batch: stacked inputs must be (B,Hf,Wf), (B,Hf,Wf,3), (B,Hf,Wf,3)")
        dev = fr.device
        masks = (src_sketch_masks == 0).to(torch.uint8).to(dev).contiguous().reshape(-1)
        nsrc = _dev(torch, src_sketch_normals, torch.uint8).to(dev).reshape(-1)
        ndst = _dev(torch, dst_sketch_normals, torch.uint8).to(dev).reshape(-1)
        if geometry is not None:
            t_off, t_rect = _full_frame_rects(torch, B, Hf, Wf, dev)
            return _pack_vunet_launch(torch, fr, frame_index, masks, nsrc, ndst, t_off, t_rect, Hf * Wf, B, Hf, Wf, res, geometry)
        t_off = torch.arange(B, dtype=torch.int64, device=dev) * (Hf * Wf)
        t_rect = torch.tensor([0, 0, Wf, Hf], dtype=torch.int32, device=dev).repeat(B, 1)
        return _pack_vunet_launch(torch, fr, frame_index, masks, nsrc, ndst, t_off, t_rect, Hf * Wf, B, Hf, Wf, res)
    rect = np.zeros((B, 4), np.int32)
    offs, fm, fs, fd, o = [], [], [], [], 0
    for b in range(B):
        m = torch.from_numpy(np.ascontiguousarray(src_sketch_masks[b])) if not isinstance(src_sketch_masks[b], torch.Tensor) else src_sketch_masks[b]
        ns = torch.from_numpy(np.ascontiguousarray(src_sketch_normals[b])) if not isinstance(src_sketch_normals[b], torch.Tensor) else src_sketch_normals[b]
        nd = torch.from_numpy(np.ascontiguousarray(dst_sketch_normals[b])) if not isinstance(dst_sketch_normals[b], torch.Tensor) else dst_sketch_normals[b]
        h, w = int(m.shape[0]), int(m.shape[1])
        if rects is None:
            if (h, w) != (Hf, Wf):
                raise ValueError(f"pack_vunet_inputs_batch: mask {b} is {(h, w)}, frame is {(Hf, Wf)}")
            rect[b] = (0, 0, Wf, Hf)
        else:
            x, y, rw, rh = (int(v) for v in rects[b])
            if (h, w) != (rh, rw):
                raise ValueError(f"pack_vunet_inputs_batch: mask {b} is {(h, w)}, its rect says {(rh, rw)}")
            rect[b] = (x, y, rw, rh)
        if tuple(ns.shape) != (h, w, 3) or tuple(nd.shape) != (h, w, 3) or ns.dtype != torch.uint8 or nd.dtype != torch.uint8:
            raise ValueError(f"pack_vunet_inputs_batch: normal sketches of item {b} must be uint8 {(h, w, 3)}")
        offs.append(o)
        fm.append((m == 0).to(torch.uint8).reshape(-1))          # vehicle = logical_not(src_sketch_mask)
        fs.append(ns.reshape(-1))
        fd.append(nd.reshape(-1))
        o += h * w
    dev = fr.device
    masks, nsrc, ndst = torch.cat(fm).to(dev), torch.cat(fs).to(dev), torch.cat(fd).to(dev)
    t_off = torch.tensor(offs, dtype=torch.int64, device=dev)
    t_rect = torch.from_numpy(rect).to(dev)
    return _pack_vunet_launch(torch, fr, frame_index, masks, nsrc, ndst, t_off, t_rect, int((rect[:, 2].astype(np.int64) * rect[:, 3]).max()), B, Hf, Wf, res)


def _pack_vunet_launch(torch, fr, frame_index, masks, nsrc, ndst, t_off, t_rect, mx, B, Hf, Wf, res, geometry=None):
    dev = fr.device
    L = _lib.lib()
    if geometry is not None:
        ok = (geometry.status == 0) & (frame_index >= 0) & (frame_index < int(fr.shape[0]))
        t_fidx = torch.where(ok, frame_index, -1).to(torch.int32)           # a negative frame index: the kernel writes zero rows
        bbox = geometry.bbox
    else:
        t_fidx = torch.tensor(list(frame_index), dtype=torch.int32, device=dev)
        bbox = torch.empty((B, 4), dtype=torch.int32, device=dev)
        _lib.check(L.fusg_mask_bbox(_lib.ptr(masks), _lib.ptr(t_off), _lib.ptr(t_rect), _lib.ptr(bbox), B, mx, _lib.stream_ptr(torch)), "fusg_mask_bbox")
        if bool((bbox[:, 2] < 0).any()):
            raise ValueError("pack_vunet_inputs_batch: empty vehicle mask (np.min of an empty array in the reference)")
    x = torch.empty((B, 6, res, res), dtype=torch.float32, device=dev)
    y = torch.empty((B, 3, res, res), dtype=torch.float32, device=dev)
    _lib.check(L.fusg_pack_vunet_inputs(_lib.ptr(fr), _lib.ptr(t_fidx), _lib.ptr(masks), _lib.ptr(nsrc), _lib.ptr(ndst), _lib.ptr(t_off),
                                        _lib.ptr(t_rect), _lib.ptr(bbox), _lib.ptr(x), _lib.ptr(y), B, Hf, Wf, res, _lib.stream_ptr(torch)),
               "fusg_pack_vunet_inputs")
    return x, y, bbox


def pack_vunet_inputs(frame, src_sketch_mask, src_sketch_normal, dst_sketch_normal):
    """One vehicle, reference-style: returns (x (1,6,256,256), y_tilde (1,3,256,256)) CUDA float tensors, the arguments of
    `model_VUnet.forward_enc_up(x)` / `forward_dec_up(y_tilde)` at trajectory_inference.py:230-233."""
    x, y, _ = pack_vunet_inputs_batch(np.asarray(frame)[None], [0], [src_sketch_mask], [src_sketch_normal], [dst_sketch_normal])
    return x, y


def u8_to_vunet_inputs(mask_bbox_u8, normal_src_u8, normal_dst_u8):
    """The three resized uint8 images of trajectory_inference.py:215-220, batched (B,res,res,3) CUDA tensors ->
    (x (B,6,res,res), y_tilde (B,3,res,res)) fp32 on the device == lines :221-225 (to_tensor, [..., ::-1], cat)."""
    torch = _lib.require_cuda()
    B, res = int(mask_bbox_u8.shape[0]), int(mask_bbox_u8.shape[1])
    for t in (mask_bbox_u8, normal_src_u8, normal_dst_u8):
        if tuple(t.shape) != (B, res, res, 3) or t.dtype != torch.uint8:
            raise ValueError("u8_to_vunet_inputs: expected three (B, res, res, 3) uint8 tensors")
    x = torch.empty((B, 6, res, res), dtype=torch.float32, device=mask_bbox_u8.device)
    y = torch.empty((B, 3, res, res), dtype=torch.float32, device=mask_bbox_u8.device)
    _lib.check(_lib.lib().fusg_u8_to_vunet_inputs(_lib.ptr(mask_bbox_u8), _lib.ptr(normal_src_u8), _lib.ptr(normal_dst_u8), _lib.ptr(x), _lib.ptr(y),
                                                  B, res, _lib.stream_ptr(torch)), "fusg_u8_to_vunet_inputs")
    return x, y


def u8_to_vunet_y(normal_dst_u8):
    """y_tilde alone: (B,res,res,3) uint8 CUDA tensor -> (B,3,res,res) fp32, the y of u8_to_vunet_inputs.  For a trajectory
    step, whose appearance input was encoded once per vehicle (trajectory_inference.py:413-426)."""
    torch = _lib.require_cuda()
    B, res = int(normal_dst_u8.shape[0]), int(normal_dst_u8.shape[1])
    if tuple(normal_dst_u8.shape) != (B, res, res, 3) or normal_dst_u8.dtype != torch.uint8:
        raise ValueError("u8_to_vunet_y: expected a (B, res, res, 3) uint8 tensor")
    y = torch.empty((B, 3, res, res), dtype=torch.float32, device=normal_dst_u8.device)
    _lib.check(_lib.lib().fusg_u8_to_vunet_y(_lib.ptr(normal_dst_u8), _lib.ptr(y), B, res, _lib.stream_ptr(torch)), "fusg_u8_to_vunet_y")
    return y


GATHER_MAX_SEGS = 8      # FUSG_GATHER_MAX_SEGS


class GatherSeg(C.Structure):
    """fusg_gather_seg (include/fusg.h)."""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("row_bytes", C.c_int64), ("n_src", C.c_int32), ("reserved", C.c_int32)]


def gather_rows(pairs, index):
    """pairs: up to 8 (src (n_src, ...), dst (B, ...)) contiguous CUDA tensors; index: (B,) int32 CUDA tensor.
    dst[b] = src[index[b]] for every pair (zeros where index[b] is out of range), in ONE launch on the current stream."""
    torch = _lib.require_cuda()
    if not 0 < len(pairs) <= GATHER_MAX_SEGS:
        raise ValueError(f"gather_rows: 1..{GATHER_MAX_SEGS} (src, dst) pairs")
    if index.dtype != torch.int32 or index.dim() != 1 or not index.is_cuda:
        raise ValueError("gather_rows: index must be a (B,) int32 CUDA tensor")
    B = int(index.shape[0])
    segs = (GatherSeg * len(pairs))()
    for s, (src, dst) in zip(segs, pairs):
        if dst.shape[0] != B or src.shape[1:] != dst.shape[1:] or src.dtype != dst.dtype:
            raise ValueError("gather_rows: dst must be (B,) + src.shape[1:] of src's dtype")
        s.src, s.dst = _lib.ptr(src).value, _lib.ptr(dst).value
        s.row_bytes, s.n_src = dst[0].numel() * dst.element_size(), int(src.shape[0])
    _lib.check(_lib.lib().fusg_gather_rows(segs, len(pairs), _lib.ptr(index), B, _lib.stream_ptr(torch)), "fusg_gather_rows")


# ---------------------------------------------------------------------------------------------------------------------
# ICN input packing (SURVEY.md 8f-1): warp_learn/models.py:323-366 get_icn_inputs on the device
# ---------------------------------------------------------------------------------------------------------------------
_LAB_DEV = {}


def _lab_tables(torch, device):
    """OpenCV's 8-bit Lab tables + exception list (data/lab8.npz, see scripts/make_lab_tables.py), uploaded once per device."""
    key = str(device)
    if key not in _LAB_DEV:
        import os
        z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "lab8.npz"))
        keys = z["exc_keys"].astype(np.int64)
        bitmap = np.zeros(1 << 19, np.int64)                 # one bit per colour: is it in the exception list at all
        np.bitwise_or.at(bitmap, keys >> 5, np.int64(1) << (keys & 31))
        _LAB_DEV[key] = (torch.from_numpy(z["gamma_tab"].astype(np.int32)).to(torch.uint16).to(device),
                         torch.from_numpy(z["cbrt_tab"].astype(np.int32)).to(torch.uint16).to(device),
                         torch.from_numpy(z["exc_keys"].astype(np.int64)).to(torch.uint32).to(device),
                         torch.from_numpy(z["exc_vals"].astype(np.int32)).to(torch.uint16).to(device),
                         torch.from_numpy(bitmap).to(torch.uint32).to(device))
    return _LAB_DEV[key]


def square_crop_info(image_hw, bbox):
    """crop_info of warp_learn/models.py:337-342 for a vehicle bounding box (utils/crop_utils.py:4-52 geometry)."""
    image_h, image_w = image_hw
    x_min, y_min, x_max, y_max = (int(v) for v in bbox)
    side_x, side_y = x_max - x_min, y_max - y_min
    major = max(side_x, side_y) * 1.1
    cx, cy = x_min + side_x / 2, y_min + side_y / 2
    pxb = pxa = pyb = pya = 0
    nx0 = int(cx - major / 2.)
    if nx0 < 0:
        pxb, nx0 = -nx0, 0
    nx1 = int(cx + major / 2.) + pxb
    if nx1 > image_w:
        pxa = nx1 - image_w
        nx1 = image_w + pxa
    ny0 = int(cy - major / 2.)
    if ny0 < 0:
        pyb, ny0 = -ny0, 0
    ny1 = int(cy + major / 2.) + pyb
    if ny1 > image_h:
        pya = ny1 - image_h
        ny1 = image_h + pya
    return {"crop_xy_min": (nx0, ny0), "pad_xy_before": (pxb, pyb), "pad_xy_after": (pxa, pya),
            "crop_size_orig": (min(ny1, image_h + pyb + pya) - ny0, min(nx1, image_w + pxb + pxa) - nx0)}


def _full_frame_rects(torch, B, Hf, Wf, dev):
    """(off (B,) int64 = b * Hf * Wf, rect (B,4) int32 = (0, 0, Wf, Hf)): B stacked full-frame masks, made by device fills (no copy)."""
    rect = torch.zeros((B, 4), dtype=torch.int32, device=dev)
    rect[:, 2], rect[:, 3] = Wf, Hf
    return torch.arange(B, dtype=torch.int64, device=dev) * (Hf * Wf), rect


def _mask_bbox(torch, sketch_masks, B, Hf, Wf, dev, what):
    """sketch_masks (B,Hf,Wf) -> (uint8 masks on dev, bbox (B,4) int32 on dev) via fusg_mask_bbox, without synchronising."""
    mk = sketch_masks if isinstance(sketch_masks, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(sketch_masks))
    mk = (mk.view(torch.uint8) if mk.dtype == torch.bool else (mk != 0).to(torch.uint8)).to(dev).contiguous()   # k_mask_bbox tests != 0
    if tuple(mk.shape) != (B, Hf, Wf):
        raise ValueError(f"{what}: sketch_masks must be {(B, Hf, Wf)}, got {tuple(mk.shape)}")
    off, rect = _full_frame_rects(torch, B, Hf, Wf, dev)
    bbox = torch.empty((B, 4), dtype=torch.int32, device=dev)
    _lib.check(_lib.lib().fusg_mask_bbox(_lib.ptr(mk), _lib.ptr(off), _lib.ptr(rect), _lib.ptr(bbox), B, Hf * Wf, _lib.stream_ptr(torch)),
               "fusg_mask_bbox")
    return mk, bbox


def _sketch_mask_bbox(torch, sketch_masks, B, Hf, Wf, dev, what):
    """_mask_bbox plus the bbox on the host.  Synchronises (crop_info is host data in the reference too: a few ints per vehicle)."""
    mk, bbox = _mask_bbox(torch, sketch_masks, B, Hf, Wf, dev, what)
    bb = bbox.cpu().numpy()
    if (bb[:, 2] < 0).any():
        raise ValueError(f"{what}: empty sketch mask (np.min of an empty array in the reference)")
    return mk, bbox, bb


def icn_window_rect(frame_hw, crop_info):
    """(x0, y0, w, h): the frame pixels `get_icn_inputs` reads for this crop_info -- its square crop clipped to the frame (crop
    pixel (cy, cx) is frame pixel (y_min - pad_y_before + cy, x_min - pad_x_before + cx)).  A mask one pixel thin can give a crop
    side of 0, whose resize taps clamp to index -1, the pixel before the crop; where that pixel lies outside the frame nothing is
    read along that axis and the window keeps one (unread) pixel at the border, so that every window is non-empty."""
    Hf, Wf = frame_hw
    (nx0, ny0), (pxb, pyb) = crop_info["crop_xy_min"], crop_info["pad_xy_before"]
    ch, cw = crop_info["crop_size_orig"]

    def span(n0, pad, size, limit):
        lo = n0 - pad if size > 0 else n0 - pad - 1
        a, b = max(lo, 0), min(lo + max(size, 1), limit)
        if b <= a:
            a = min(max(lo, 0), limit - 1)
            b = a + 1
        return a, b

    x0, x1 = span(int(nx0), int(pxb), int(cw), Wf)
    y0, y1 = span(int(ny0), int(pyb), int(ch), Hf)
    return x0, y0, x1 - x0, y1 - y0


class IcnWindows:
    """Per-item frame windows of the ICN branch (`icn_windows`): what `warp_batch(..., window=)` writes and
    `get_icn_inputs_batch` reads.
      bbox (B,4) int32 device / bbox_host numpy: (x_min, y_min, x_max, y_max) of each sketch mask (fusg_mask_bbox)
      crop_infos: square_crop_info of each bbox, as get_icn_inputs_batch returns them
      rect (B,4) int32 numpy / rect_dev: (x0, y0, w, h) = icn_window_rect
      off (B,) int64 numpy / off_dev: byte offset of item b's block, 16-byte aligned; the block holds 5 planes of h*w*3 bytes
      nbytes: total bytes of the blocks; max_h: the tallest window; frame_hw: (Hf, Wf)."""

    def __init__(self, bbox, bbox_host, crop_infos, rect, off, nbytes, frame_hw):
        torch = _lib.require_cuda()
        self.bbox, self.bbox_host, self.crop_infos = bbox, bbox_host, crop_infos
        self.rect, self.off, self.nbytes, self.frame_hw = rect, off, int(nbytes), tuple(frame_hw)
        self.max_h = int(rect[:, 3].max())
        self.rect_dev = torch.from_numpy(rect).to(bbox.device)
        self.off_dev = torch.from_numpy(off).to(bbox.device)

    def __len__(self):
        return int(self.rect.shape[0])

    def window(self, b):
        """(x0, y0, w, h, off) of item b."""
        return tuple(int(v) for v in self.rect[b]) + (int(self.off[b]),)


def window_layout(rects):
    """(B,4) (x0, y0, w, h) -> (off (B,) int64, nbytes): item b's five [h,w,3] planes at off[b], blocks 16-byte aligned."""
    sizes = 5 * rects[:, 2].astype(np.int64) * rects[:, 3] * 3
    off = np.zeros(len(rects), np.int64)
    o = 0
    for b, s in enumerate(sizes):
        off[b] = o
        o += (int(s) + 15) & ~15
    return off, o


def icn_windows(sketch_masks, frame_hw):
    """sketch_masks (B,Hf,Wf) bool / uint8 (non-zero = vehicle, the masks get_icn_inputs_batch will be given), numpy or torch ->
    IcnWindows: for each item, the frame window whose pixels get_icn_inputs reads.  One fusg_mask_bbox pass, synchronised to
    the host.  An empty mask raises ValueError, as get_icn_inputs_batch does."""
    torch = _lib.require_cuda()
    Hf, Wf = (int(v) for v in frame_hw)
    B = int(sketch_masks.shape[0])
    if B == 0:
        raise ValueError("icn_windows: no items")
    dev = sketch_masks.device if isinstance(sketch_masks, torch.Tensor) and sketch_masks.is_cuda else torch.device("cuda")
    _, bbox, bb = _sketch_mask_bbox(torch, sketch_masks, B, Hf, Wf, dev, "icn_windows")
    infos = [square_crop_info((Hf, Wf), bb[b]) for b in range(B)]
    rect = np.array([icn_window_rect((Hf, Wf), ci) for ci in infos], np.int32).reshape(B, 4)
    off, nbytes = window_layout(rect)
    return IcnWindows(bbox, bb, infos, rect, off, nbytes, (Hf, Wf))


class CropGeometry:
    """The crop geometry of a batch of sketch masks, computed on the device by `crop_geometry` (fusg_mask_bbox + fusg_crop_geometry):
      bbox (B,4) int32: (x_min, y_min, x_max, y_max) of each mask, (INT_MAX, INT_MAX, -1, -1) when it is empty
      info (B,9) int32: fusg_paste_back's info == pack_crop_info(square_crop_info(bbox), frame_index)
      win (B,4) int32 / win_off (B,) int64: icn_window_rect / window_layout (None without a window capacity)
      status (B,) int8: 0 ok, 1 empty mask, 2 the window does not fit the capacity (see fusg.h); refused items get win (0, 0, 0, 0)
      frame_index (B,) int32 or None (frame 0), all on the device; capacity_bytes, max_win_h, frame_hw: the host ints chosen by the caller.
    It also offers IcnWindows' interface (rect_dev, off_dev, nbytes, max_h, rect, off), so that warp_batch(..., window=) and
    WindowedPlanes take it in place of icn_windows; rect / off copy the device arrays to the host (they synchronise)."""

    def __init__(self, bbox, info, win, win_off, status, frame_index, capacity_bytes, max_win_h, frame_hw):
        self.bbox, self.info, self.win, self.win_off, self.status, self.frame_index = bbox, info, win, win_off, status, frame_index
        self.capacity_bytes, self.max_win_h, self.frame_hw = int(capacity_bytes), int(max_win_h), tuple(frame_hw)

    def __len__(self):
        return int(self.status.shape[0])

    rect_dev = property(lambda self: self.win)
    off_dev = property(lambda self: self.win_off)
    nbytes = property(lambda self: self.capacity_bytes)
    max_h = property(lambda self: self.max_win_h)
    rect = property(lambda self: self.win.cpu().numpy())
    off = property(lambda self: self.win_off.cpu().numpy())

    def window(self, b):
        """(x0, y0, w, h, off) of item b: one small device-to-host copy (not cached: a graph replay rewrites the device arrays)."""
        torch = _lib.require_cuda()
        return tuple(int(v) for v in torch.cat([self.win[b].to(torch.int64), self.win_off[b:b + 1]]).tolist())

    def crop_infos(self):
        """Synchronises; the crop_info dicts get_icn_inputs_batch returns for the same masks (None for an empty mask)."""
        info, st = self.info.cpu().numpy(), self.status.cpu().numpy()
        return [None if st[b] == 1 else {"crop_xy_min": (int(i[7]), int(i[8])), "pad_xy_before": (int(i[3]), int(i[4])),
                                          "pad_xy_after": (int(i[5]), int(i[6])), "crop_size_orig": (int(i[1]), int(i[2]))}
                for b, i in enumerate(info)]

    def check(self):
        """Synchronises; raises ValueError for empty masks and warp_learn.RefusedCrops for windows that do not fit the capacity."""
        from .warp_learn.batch import RefusedCrops
        st = self.status.cpu().numpy()
        empty = np.nonzero(st == 1)[0].tolist()
        if empty:
            raise ValueError(f"crop_geometry: empty sketch mask (np.min of an empty array in the reference): items {empty[:8]}")
        refused = np.nonzero(st == 2)[0].tolist()
        if refused:
            raise RefusedCrops(refused, reason="crop geometry refused {n} window(s) (past the capacity or taller than max_win_h)")
        return self


def crop_geometry(vehicle_masks, frame_hw, frame_index=None, window_capacity=None):
    """vehicle_masks (B,Hf,Wf) bool / uint8 (non-zero = vehicle), numpy or torch -> CropGeometry, with one fusg_mask_bbox pass and one
    fusg_crop_geometry launch: no synchronisation and, for device masks, no host-to-device copy -- capturable in a CUDA graph.
    frame_index: (B,) int32 CUDA tensor (the frame each item is pasted into) or None (frame 0).  window_capacity (bytes, rows):
    the window buffer warp_batch(..., window=) writes -- its size and the tallest window it serves; needed for windowed warping.
    Fixed per graph, sized by the caller; items past it get status 2.  Nothing is checked on the host: see CropGeometry.check."""
    torch = _lib.require_cuda()
    Hf, Wf = (int(v) for v in frame_hw)
    B = int(vehicle_masks.shape[0])
    if B == 0:
        raise ValueError("crop_geometry: no items")
    dev = vehicle_masks.device if isinstance(vehicle_masks, torch.Tensor) and vehicle_masks.is_cuda else torch.device("cuda")
    if frame_index is not None and not (isinstance(frame_index, torch.Tensor) and frame_index.is_cuda and frame_index.dtype == torch.int32
                                        and tuple(frame_index.shape) == (B,) and frame_index.is_contiguous()):
        raise ValueError("crop_geometry: frame_index must be a contiguous (B,) int32 CUDA tensor")
    cap, rows = (0, 0) if window_capacity is None else (int(v) for v in window_capacity)
    if window_capacity is not None and (cap <= 0 or rows <= 0):
        raise ValueError("crop_geometry: window_capacity is (bytes, rows), both positive")
    _, bbox = _mask_bbox(torch, vehicle_masks, B, Hf, Wf, dev, "crop_geometry")
    info = torch.empty((B, INFO_FIELDS), dtype=torch.int32, device=dev)
    status = torch.empty((B,), dtype=torch.int8, device=dev)
    win = torch.empty((B, 4), dtype=torch.int32, device=dev) if cap else None
    win_off = torch.empty((B,), dtype=torch.int64, device=dev) if cap else None
    _lib.check(_lib.lib().fusg_crop_geometry(_lib.ptr(bbox), _lib.ptr(frame_index), B, Hf, Wf, cap, rows, _lib.ptr(info), _lib.ptr(win),
                                             _lib.ptr(win_off), _lib.ptr(status), _lib.stream_ptr(torch)), "fusg_crop_geometry")
    return CropGeometry(bbox, info, win, win_off, status, frame_index, cap, rows, (Hf, Wf))


class WindowedPlanes:
    """The five warped planes of each item, only inside its window: `warp_batch(..., window=)`'s `warped`.
    data: flat uint8 CUDA tensor of windows.nbytes bytes; item(b) -> (5, h, w, 3) view of item b's planes (BGR).
    windows: the IcnWindows or CropGeometry the planes were warped for."""

    def __init__(self, data, windows: IcnWindows):
        self.data, self.windows = data, windows

    @property
    def rect(self):
        return self.windows.rect

    @property
    def off(self):
        return self.windows.off

    def item(self, b):
        x0, y0, w, h, o = self.windows.window(b)
        return self.data[o:o + 5 * h * w * 3].view(5, h, w, 3)


def get_icn_inputs_batch(planes, sketch_normals, sketch_masks, central_crops, icn_w=256, icn_h=256, geometry=None):
    """`get_icn_inputs` for B vehicles at once.  planes (B,5,Hf,Wf,3) uint8 BGR (e.g. `warp_batch(...).warped` for whole
    frames, still on the device) -- or a WindowedPlanes (`warp_batch(..., window=icn_windows(sketch_masks, (Hf, Wf)))`), which
    holds only the pixels read here and gives the same result bit for bit --, sketch_normals (B,Hf,Wf,3) uint8 RGB, sketch_masks
    (B,Hf,Wf) bool / uint8 (non-zero = vehicle), central_crops (B,icn_h,icn_w,3) uint8 RGB; numpy or torch, host or device.
    Returns (gen_in (B,21,icn_h,icn_w) float32 CUDA tensor == the reference's tensors stacked, list of B crop_info dicts).
    With WindowedPlanes, masks whose bounding boxes differ from those the windows were cut for raise ValueError.
    geometry (crop_geometry of the sketch masks, optional; sketch_masks is then not read, pass None): the crops come from it -- no bbox
    pass, no synchronisation -- and the call returns (gen_in, geometry).  planes are whole frames or warp_batch(..., window=geometry)'s
    WindowedPlanes; an item with a non-zero status gets an all-zero gen_in row (its window, never written, is not read)."""
    if icn_w != icn_h:
        raise NotImplementedError("get_icn_inputs_batch: square ICN inputs only (the reference uses 256 x 256)")
    torch = _lib.require_cuda()
    if geometry is not None:
        return _icn_inputs_from_geometry(torch, planes, sketch_normals, central_crops, icn_h, geometry)
    windowed = isinstance(planes, WindowedPlanes)
    if windowed:
        pl = planes.data
        if pl.dtype != torch.uint8 or pl.dim() != 1 or not pl.is_cuda or pl.numel() < planes.windows.nbytes:
            raise ValueError("get_icn_inputs_batch: WindowedPlanes.data must be a flat uint8 CUDA tensor of windows.nbytes bytes")
        B, (Hf, Wf) = len(planes.windows), planes.windows.frame_hw
    else:
        pl = _dev(torch, planes, torch.uint8)
        if pl.dim() != 5 or pl.shape[1] != 5 or pl.shape[4] != 3:
            raise ValueError("get_icn_inputs_batch: planes must be (B, 5, Hf, Wf, 3) uint8")
        B, Hf, Wf = int(pl.shape[0]), int(pl.shape[2]), int(pl.shape[3])
    dev = pl.device
    nm = _dev(torch, sketch_normals, torch.uint8).to(dev)
    ct = _dev(torch, central_crops, torch.uint8).to(dev)
    if tuple(nm.shape) != (B, Hf, Wf, 3) or tuple(ct.shape) != (B, icn_h, icn_w, 3):
        raise ValueError("get_icn_inputs_batch: sketch_normals (B,Hf,Wf,3), sketch_masks (B,Hf,Wf), central_crops (B,res,res,3) expected")
    _, bbox, bb = _sketch_mask_bbox(torch, sketch_masks, B, Hf, Wf, dev, "get_icn_inputs_batch")
    L = _lib.lib()
    g, c, ek, ev, bm = _lab_tables(torch, dev)
    out = torch.empty((B, 21, icn_h, icn_w), dtype=torch.float32, device=dev)
    if windowed:
        w = planes.windows
        if not np.array_equal(bb, w.bbox_host):
            bad = np.nonzero((bb != w.bbox_host).any(1))[0]
            raise ValueError(f"get_icn_inputs_batch: the sketch masks of items {bad[:8].tolist()} are not those the planes' windows were cut for")
        _lib.check(L.fusg_pack_icn_inputs_window(_lib.ptr(pl), _lib.ptr(w.rect_dev), _lib.ptr(w.off_dev), _lib.ptr(nm), _lib.ptr(ct), _lib.ptr(bbox),
                                                 _lib.ptr(g), _lib.ptr(c), _lib.ptr(ek), _lib.ptr(ev), int(ek.numel()), _lib.ptr(bm), _lib.ptr(out),
                                                 B, Hf, Wf, icn_h, _lib.stream_ptr(torch)), "fusg_pack_icn_inputs_window")
        out._keep = (pl, nm, ct, bbox, w.rect_dev, w.off_dev)
    else:
        _lib.check(L.fusg_pack_icn_inputs(_lib.ptr(pl), _lib.ptr(nm), _lib.ptr(ct), _lib.ptr(bbox), _lib.ptr(g), _lib.ptr(c), _lib.ptr(ek), _lib.ptr(ev),
                                          int(ek.numel()), _lib.ptr(bm), _lib.ptr(out), B, Hf, Wf, icn_h, _lib.stream_ptr(torch)), "fusg_pack_icn_inputs")
        out._keep = (pl, nm, ct, bbox)
    return out, [square_crop_info((Hf, Wf), bb[b]) for b in range(B)]


def _icn_inputs_from_geometry(torch, planes, sketch_normals, central_crops, res, g):
    B, (Hf, Wf) = len(g), g.frame_hw
    if isinstance(planes, WindowedPlanes):
        if planes.windows is not g:
            raise ValueError("get_icn_inputs_batch: the planes were warped for other windows than the geometry's")
        pl, win, win_off = planes.data, g.win, g.win_off
    else:
        pl = _dev(torch, planes, torch.uint8)
        if tuple(pl.shape) != (B, 5, Hf, Wf, 3):
            raise ValueError(f"get_icn_inputs_batch: planes must be {(B, 5, Hf, Wf, 3)} uint8 for this geometry")
        # whole frames are windows too: item b's window is its frame at b * 5*Hf*Wf*3, empty where the geometry refused the item
        win_off, win = _full_frame_rects(torch, B, Hf, Wf, pl.device)
        win, win_off = win * (g.status == 0).to(torch.int32).view(B, 1), win_off * 15
    dev = pl.device
    nm = _dev(torch, sketch_normals, torch.uint8).to(dev)
    ct = _dev(torch, central_crops, torch.uint8).to(dev)
    if tuple(nm.shape) != (B, Hf, Wf, 3) or tuple(ct.shape) != (B, res, res, 3):
        raise ValueError("get_icn_inputs_batch: sketch_normals (B,Hf,Wf,3), central_crops (B,res,res,3) expected")
    gt, c, ek, ev, bm = _lab_tables(torch, dev)
    out = torch.empty((B, 21, res, res), dtype=torch.float32, device=dev)
    _lib.check(_lib.lib().fusg_pack_icn_inputs_window(_lib.ptr(pl), _lib.ptr(win), _lib.ptr(win_off), _lib.ptr(nm), _lib.ptr(ct), _lib.ptr(g.bbox),
                                                      _lib.ptr(gt), _lib.ptr(c), _lib.ptr(ek), _lib.ptr(ev), int(ek.numel()), _lib.ptr(bm),
                                                      _lib.ptr(out), B, Hf, Wf, res, _lib.stream_ptr(torch)), "fusg_pack_icn_inputs_window")
    out._keep = (pl, nm, ct, win, win_off)
    return out, g


def get_icn_inputs(planes, sketch_normal, sketch_mask, central_crop, icn_w, icn_h):
    """Reference signature (warp_learn/models.py:323): one vehicle -> (gen_in (1,21,icn_h,icn_w) CUDA float tensor, crop_info)."""
    out, infos = get_icn_inputs_batch(planes[None], np.asarray(sketch_normal)[None], np.asarray(sketch_mask)[None],
                                      np.asarray(central_crop)[None], icn_w, icn_h)
    return out, infos[0]
