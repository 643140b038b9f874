"""CPU suite: the C-ABI boundary of the ICN-window pieces (windowed fused warp, ICN packing from windows) -- argument validation --
and the host-side window geometry (icn_window_rect, window_layout) against the square crop it stands for."""
import ctypes
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = ctypes.c_void_p(0x10000)


def test_icn_window_symbols_are_declared():
    hdr = open(os.path.join(ROOT, "include", "fusg.h")).read()
    names = set(re.findall(r"\b(fusg_[a-z0-9_]+)\s*\(", hdr))
    for n in ("fusg_warp_window_workspace_bytes", "fusg_warp_fused_window", "fusg_pack_icn_inputs_window"):
        assert n in names, n


def _warp_win(L, ptrs=None, B=4, H=720, W=1280, max_win_h=64, ws_bytes=None, n_src=0):
    p = dict(src=FAKE, src_index=None, src_kp=FAKE, dst_kp=FAKE, K=FAKE, E_src=FAKE, E_dst=FAKE, kp3d_src=FAKE, kp3d_dst=None, win=FAKE,
             win_off=FAKE, warped=FAKE, vis=FAKE, plane_j=FAKE, H12=None, workspace=FAKE)
    p.update(ptrs or {})
    if ws_bytes is None:
        ws_bytes = L.fusg_warp_window_workspace_bytes(max(B, 1), H, W)
    return L.fusg_warp_fused_window(p["src"], p["src_index"], n_src, p["src_kp"], p["dst_kp"], p["K"], p["E_src"], p["E_dst"], p["kp3d_src"],
                                    p["kp3d_dst"], p["win"], p["win_off"], max_win_h, p["warped"], p["vis"], p["plane_j"], p["H12"],
                                    p["workspace"], ws_bytes, B, H, W, None)


def test_windowed_warp_validates_arguments():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    for name in ("src", "src_kp", "dst_kp", "K", "E_src", "E_dst", "kp3d_src", "win", "win_off", "warped", "vis", "plane_j", "workspace"):
        assert _warp_win(L, {name: None}) == -1, name
    assert _warp_win(L, B=0) == -1
    assert _warp_win(L, B=-3) == -1
    assert _warp_win(L, max_win_h=0) == -1
    assert _warp_win(L, max_win_h=-5) == -1
    assert _warp_win(L, {"src_index": ctypes.c_void_p(0x20000)}, n_src=0) == -1     # an index without source images
    need = L.fusg_warp_window_workspace_bytes(4, 720, 1280)
    assert _warp_win(L, ws_bytes=need - 1) == -4
    assert _warp_win(L, B=4, H=256, W=256, ws_bytes=L.fusg_warp_workspace_bytes_hw(4, 256, 256)) == -4   # the masks are extra at any size


def test_window_workspace_covers_the_plane_masks():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    for B, H, W in ((1, 8, 8), (4, 256, 256), (600, 1080, 1920), (3, 300, 401)):
        base = (L.fusg_warp_workspace_bytes(B) + 15) // 16 * 16
        assert L.fusg_warp_window_workspace_bytes(B, H, W) == base + B * 5 * H * ((W + 31) // 32) * 4
    assert L.fusg_warp_window_workspace_bytes(0, 720, 1280) == 0
    assert L.fusg_warp_window_workspace_bytes(4, 0, 1280) == 0


def test_windowed_icn_pack_validates_arguments():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()

    def call(i_null=None, n_exc=0, B=2, Hf=720, Wf=1280, res=256):
        a = [FAKE] * 10
        if i_null is not None:
            a[i_null] = None
        return L.fusg_pack_icn_inputs_window(*a, n_exc, None, FAKE, B, Hf, Wf, res, None)

    for i in range(8):                          # planes, win, win_off, normals, central, bbox, gamma_tab, cbrt_tab
        assert call(i) == -1, i
    assert call(8, n_exc=5) == -1               # exception list announced but missing
    assert call(B=0) == -1 and call(B=-1) == -1
    assert call(res=0) == -1 and call(Hf=0) == -1 and call(Wf=0) == -1
    assert L.fusg_pack_icn_inputs_window(*[FAKE] * 10, 0, None, None, 2, 720, 1280, 256, None) == -1   # no output


def _axis_reads(n0, pad, size, limit):
    """Brute force along one axis: the frame indices cv2.resize of the square crop reads (crop index c -> frame n0 - pad + c; the taps
    clamp to [0, size - 1], which is {-1} for size 0) that lie in the frame, as (lo, length); one border pixel when there is none."""
    taps = np.arange(size) if size > 0 else np.array([-1])
    f = taps + n0 - pad
    f = f[(f >= 0) & (f < limit)]
    if f.size == 0:
        return min(max(n0 - pad - (size == 0), 0), limit - 1), 1
    return int(f.min()), int(f.max() - f.min() + 1)


def _crop_read_rect(frame_hw, ci):
    Hf, Wf = frame_hw
    (nx0, ny0), (pxb, pyb) = ci["crop_xy_min"], ci["pad_xy_before"]
    ch, cw = ci["crop_size_orig"]
    x0, w = _axis_reads(nx0, pxb, cw, Wf)
    y0, h = _axis_reads(ny0, pyb, ch, Hf)
    return x0, y0, w, h


def test_window_rect_is_the_square_crop_clipped_to_the_frame():
    from future_urban_scene_generation_b200.frame_ops import square_crop_info, icn_window_rect
    rng = np.random.default_rng(7)
    for Hf, Wf in ((256, 256), (300, 400), (720, 1280), (1080, 1920)):
        boxes = []
        for _ in range(400):
            x0, y0 = int(rng.integers(0, Wf)), int(rng.integers(0, Hf))
            x1, y1 = int(rng.integers(x0, Wf)), int(rng.integers(y0, Hf))
            boxes.append((x0, y0, x1, y1))
        # boxes touching every border, the whole frame, thin boxes along the edges
        boxes += [(0, 0, 40, 30), (Wf - 41, 0, Wf - 1, 30), (0, Hf - 31, 40, Hf - 1), (Wf - 41, Hf - 31, Wf - 1, Hf - 1),
                  (0, 0, Wf - 1, Hf - 1), (0, 5, 1, Hf - 6), (Wf - 2, 0, Wf - 1, Hf - 1), (3, 0, Wf - 4, 1), (0, Hf - 1, Wf - 1, Hf - 1),
                  (Wf // 2, 0, Wf // 2 + 1, 0), (0, Hf // 2, 1, Hf // 2 + 1)]
        hit_border = np.zeros(4, bool)
        for bb in boxes:
            ci = square_crop_info((Hf, Wf), bb)
            r = icn_window_rect((Hf, Wf), ci)
            assert r == _crop_read_rect((Hf, Wf), ci), (bb, ci, r)
            x0, y0, w, h = r
            assert 0 <= x0 and 0 <= y0 and w >= 1 and h >= 1 and x0 + w <= Wf and y0 + h <= Hf
            hit_border |= (x0 == 0, y0 == 0, x0 + w == Wf, y0 + h == Hf)
        assert hit_border.all()


def test_window_rect_of_a_one_pixel_mask():
    """A one-pixel mask gives a crop of size 0; the resize taps then clamp to the pixel up and left of it -- or to nothing in the
    frame, at the top-left corner, where the window is one unread pixel."""
    from future_urban_scene_generation_b200.frame_ops import square_crop_info, icn_window_rect
    ci = square_crop_info((720, 1280), (640, 360, 640, 360))
    assert tuple(ci["crop_size_orig"]) == (0, 0)
    assert icn_window_rect((720, 1280), ci) == (639, 359, 1, 1)
    assert icn_window_rect((720, 1280), square_crop_info((720, 1280), (0, 0, 0, 0))) == (0, 0, 1, 1)


def test_window_layout_is_aligned_and_disjoint():
    from future_urban_scene_generation_b200.frame_ops import window_layout
    rng = np.random.default_rng(3)
    rects = np.stack([rng.integers(0, 100, 50), rng.integers(0, 100, 50), rng.integers(1, 300, 50), rng.integers(1, 300, 50)], 1).astype(np.int32)
    off, nbytes = window_layout(rects)
    size = 5 * rects[:, 2].astype(np.int64) * rects[:, 3] * 3
    assert off.dtype == np.int64 and (off % 16 == 0).all() and off[0] == 0
    assert (off[1:] >= off[:-1] + size[:-1]).all() and (off[1:] - off[:-1] - size[:-1] < 16).all()
    assert nbytes >= off[-1] + size[-1] and nbytes % 16 == 0
