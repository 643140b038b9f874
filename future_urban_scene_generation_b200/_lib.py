"""ctypes binding of the C-ABI library libfusg.so (include/fusg.h).

The product path has no CPU fallback: importing this module without the built library, or
calling into it without a CUDA device, raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfusg.so")

POLY_COORD_MAX = 1 << 20      # csrc/warp_geom.cuh
ERRORS = {-1: "FUSG_ERR_ARG", -2: "FUSG_ERR_UNSUPPORTED", -3: "FUSG_ERR_CUDA", -4: "FUSG_ERR_WORKSPACE"}


class FusgError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise FusgError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i = C.c_void_p, C.c_size_t, C.c_int
    sigs = {
        "fusg_version": ([], i),
        "fusg_last_error": ([], C.c_char_p),
        "fusg_kernel_launches": ([], i),
        "fusg_warp_workspace_bytes": ([i], sz),
        "fusg_warp_workspace_bytes_hw": ([i, i, i], sz),
        "fusg_warp_fused": ([vp] * 11 + [vp, sz, i, i, i, vp], i),
        "fusg_warp_fused_traj": ([vp] * 12 + [vp, sz, i, i, i, vp], i),
        "fusg_warp_fused_idx": ([vp, vp, i] + [vp] * 11 + [vp, sz, i, i, i, vp], i),
        "fusg_warp_window_workspace_bytes": ([i, i, i], sz),
        "fusg_warp_fused_window": ([vp, vp, i] + [vp] * 9 + [i] + [vp] * 4 + [vp, sz, i, i, i, vp], i),
        "fusg_step_keypoints": ([vp] * 10 + [i, i, i, vp], i),
        "fusg_visibility": ([vp] * 6 + [i, i, i, vp], i),
        "fusg_get_planes": ([vp] * 3 + [i, i, i, vp], i),
        "fusg_find_homography": ([vp, vp, i, vp, vp, i, vp], i),
        "fusg_warp_perspective": ([vp] * 3 + [i, i, i, vp], i),
        "fusg_conv2d": ([vp, vp], i),
        "fusg_conv2d_select": ([vp], i),
        "fusg_conv2d_last_plan": ([vp], None),
        "fusg_conv2d_set_sm_reserve": ([i], i),
        "fusg_sizeof_conv_desc": ([], sz),
        "fusg_fold_weightnorm": ([vp, vp, vp, i, i, i, i, i, i, vp], i),
        "fusg_fold_weightnorm_paired": ([vp, vp, vp, vp, vp, i, i, i, i, i, i, vp], i),
        "fusg_nchw_to_nhwc": ([vp, vp, i, i, i, i, i, i, i, vp], i),
        "fusg_nhwc_to_nchw": ([vp, vp, i, i, i, i, i, i, vp], i),
        "fusg_to_image": ([vp, vp, i, i, i, vp], i),
        "fusg_to_image_lab": ([vp, vp, vp, vp, i, i, i, vp], i),
        "fusg_elu": ([vp, vp, sz, i, vp], i),
        "fusg_nchw_to_nhwc_reflect": ([vp, vp, i, i, i, i, i, i, i, vp], i),
        "fusg_norm_stats": ([vp, vp, i, i, i, i, i, vp], i),
        "fusg_norm_finalize": ([vp, vp, vp, vp, i, i, i, i, i, C.c_float, vp], i),
        "fusg_norm_apply": ([vp, vp, vp, i, vp, i, i, i, i, i, i, i, i, vp], i),
        "fusg_resize_u8": ([vp] * 6 + [i, i, vp], i),
        "fusg_paste_workspace_bytes": ([i, i, i], sz),
        "fusg_paste_back": ([vp] * 7 + [sz, i, i, i, i, i, i, vp], i),
        "fusg_u8_to_vunet_inputs": ([vp] * 5 + [i, i, vp], i),
        "fusg_u8_to_vunet_y": ([vp, vp, i, i, vp], i),
        "fusg_gather_rows": ([vp, i, vp, i, vp], i),
        "fusg_sizeof_gather_seg": ([], sz),
        "fusg_mask_bbox": ([vp] * 4 + [i, i, vp], i),
        "fusg_pack_icn_inputs": ([vp] * 8 + [i, vp, vp, i, i, i, i, vp], i),
        "fusg_pack_icn_inputs_window": ([vp] * 10 + [i, vp, vp, i, i, i, i, vp], i),
        "fusg_pack_vunet_inputs": ([vp] * 10 + [i, i, i, i, vp], i),
        "fusg_render_workspace_bytes": ([i, i, i, i], sz),
        "fusg_render_normals": ([vp] * 4 + [i, i] + [vp] * 6 + [vp, sz, i, i, i, vp], i),
    }
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().fusg_last_error().decode() if rc == -3 else ""
        raise FusgError(f"{what} failed: {ERRORS.get(rc, rc)} {msg}")


def conv_last_plan():
    """dict(msub, pair, halo, ksplit, stages, group, w_resident, fast_epi) of this thread's last tcgen05 conv launch."""
    buf = (C.c_int32 * 8)()
    lib().fusg_conv2d_last_plan(buf)
    return dict(zip(("msub", "pair", "halo", "ksplit", "stages", "group", "w_resident", "fast_epi"), list(buf)))


def kernel_launches():
    return lib().fusg_kernel_launches()


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise FusgError("no CUDA device: the B200 path has no CPU fallback")
    return torch


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (or None)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    return C.c_void_p(t.data_ptr())


def stream_ptr(torch):
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
