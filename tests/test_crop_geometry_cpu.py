"""CPU suite: the C-ABI boundary of fusg_crop_geometry (argument validation) and the vectorised restatement of the host crop geometry
(square_crop_info -> pack_crop_info's fields, icn_window_rect, window_layout) that tests/test_crop_geometry_gpu.py checks the kernel
against on millions of boxes -- here checked against those Python functions themselves."""
import ctypes
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = ctypes.c_void_p(0x10000)


def reference_geometry(bbox, frame_hw, frame_index=None):
    """bbox (B,4) (x_min, y_min, x_max, y_max), non-empty -> (info (B,9) int32, win (B,4) int32, win_off (B,) int64, nbytes): the
    Python geometry of frame_ops in numpy float64, operation for operation (IEEE double, no contraction; trunc = int())."""
    Hf, Wf = frame_hw
    bb = np.asarray(bbox, np.int64)
    x_min, y_min, sx, sy = bb[:, 0], bb[:, 1], bb[:, 2] - bb[:, 0], bb[:, 3] - bb[:, 1]
    major = np.maximum(sx, sy).astype(np.float64) * 1.1
    cx, cy = x_min + sx / 2, y_min + sy / 2

    def axis(c, limit):
        n0 = np.trunc(c - major / 2.).astype(np.int64)
        pb = np.where(n0 < 0, -n0, 0)
        n0 = np.maximum(n0, 0)
        n1 = np.trunc(c + major / 2.).astype(np.int64) + pb
        pa = np.where(n1 > limit, n1 - limit, 0)
        n1 = np.where(n1 > limit, limit + pa, n1)
        size = np.minimum(n1, limit + pb + pa) - n0
        lo = np.where(size > 0, n0 - pb, n0 - pb - 1)           # icn_window_rect's span
        a, e = np.maximum(lo, 0), np.minimum(lo + np.maximum(size, 1), limit)
        empty = e <= a
        a = np.where(empty, np.minimum(np.maximum(lo, 0), limit - 1), a)
        e = np.where(empty, a + 1, e)
        return n0, pb, pa, size, a, e - a

    nx0, pxb, pxa, cw, wx, ww = axis(cx, Wf)
    ny0, pyb, pya, ch, wy, wh = axis(cy, Hf)
    fr = np.zeros(len(bb), np.int64) if frame_index is None else np.asarray(frame_index, np.int64)
    info = np.stack([fr, ch, cw, pxb, pyb, pxa, pya, nx0, ny0], 1).astype(np.int32)
    win = np.stack([wx, wy, ww, wh], 1).astype(np.int32)
    blocks = (5 * ww * wh * 3 + 15) & ~15
    ends = np.cumsum(blocks)
    return info, win, ends - blocks, int(ends[-1]) if len(ends) else 0


def random_boxes(rng, n, frame_hw):
    """n boxes inside the frame: a third random, a third thin (1-px masks, 1-px sides), a third touching a border."""
    Hf, Wf = frame_hw
    x = np.sort(rng.integers(0, Wf, (n, 2)), 1)
    y = np.sort(rng.integers(0, Hf, (n, 2)), 1)
    k = n // 3
    x[k:2 * k, 1] = x[k:2 * k, 0] + rng.integers(0, 2, k)
    y[k:2 * k, 1] = np.where(rng.integers(0, 2, k) == 1, y[k:2 * k, 0], y[k:2 * k, 1])
    x[k:2 * k, 1] = np.minimum(x[k:2 * k, 1], Wf - 1)
    side = rng.integers(0, 4, n - 2 * k)
    t = slice(2 * k, n)
    x[t, 0] = np.where(side == 0, 0, x[t, 0]); x[t, 1] = np.where(side == 1, Wf - 1, x[t, 1])
    y[t, 0] = np.where(side == 2, 0, y[t, 0]); y[t, 1] = np.where(side == 3, Hf - 1, y[t, 1])
    return np.stack([x[:, 0], y[:, 0], x[:, 1], y[:, 1]], 1).astype(np.int32)


def test_crop_geometry_symbol_is_declared():
    hdr = open(os.path.join(ROOT, "include", "fusg.h")).read()
    assert "fusg_crop_geometry" in set(re.findall(r"\b(fusg_[a-z0-9_]+)\s*\(", hdr))


def test_crop_geometry_validates_arguments():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()

    def call(bbox=FAKE, frame_index=None, B=4, Hf=720, Wf=1280, cap=0, rows=0, info=FAKE, win=None, win_off=None, status=FAKE):
        return L.fusg_crop_geometry(bbox, frame_index, B, Hf, Wf, cap, rows, info, win, win_off, status, None)

    assert call(bbox=None) == -1 and call(info=None) == -1 and call(status=None) == -1
    assert call(B=0) == -1 and call(B=-2) == -1
    assert call(Hf=0) == -1 and call(Wf=0) == -1 and call(Hf=-1) == -1
    assert call(cap=-1) == -1 and call(cap=-1, win=FAKE, win_off=FAKE, rows=8) == -1
    assert call(cap=1 << 20, rows=64) == -1                                          # a capacity without windows
    assert call(cap=1 << 20, rows=64, win=FAKE) == -1 and call(cap=1 << 20, rows=64, win_off=FAKE) == -1
    assert call(cap=1 << 20, rows=0, win=FAKE, win_off=FAKE) == -1                   # ... or without a row limit


def test_reference_geometry_is_the_python_geometry():
    """Every box of a 12 x 17 frame and random boxes at 1080p: the vectorised reference equals square_crop_info / icn_window_rect /
    window_layout called box by box."""
    from future_urban_scene_generation_b200.frame_ops import icn_window_rect, square_crop_info, window_layout
    xs = [(a, b) for a in range(17) for b in range(a, 17)]
    ys = [(a, b) for a in range(12) for b in range(a, 12)]
    cases = [((12, 17), np.array([(x0, y0, x1, y1) for x0, x1 in xs for y0, y1 in ys], np.int32)),
             ((1080, 1920), random_boxes(np.random.default_rng(3), 6000, (1080, 1920)))]
    for hw, bb in cases:
        fr = np.arange(len(bb)) % 7
        info, win, off, nbytes = reference_geometry(bb, hw, fr)
        infos = [square_crop_info(hw, b) for b in bb]
        want = np.array([(f, *ci["crop_size_orig"], *ci["pad_xy_before"], *ci["pad_xy_after"], *ci["crop_xy_min"]) for f, ci in zip(fr, infos)],
                        np.int32)
        assert np.array_equal(info, want), hw
        rect = np.array([icn_window_rect(hw, ci) for ci in infos], np.int32)
        assert np.array_equal(win, rect), hw
        w_off, w_bytes = window_layout(rect)
        assert np.array_equal(off, w_off) and nbytes == w_bytes, hw
        assert (info[:, 1] == 0).any()                         # single-pixel masks give a crop side of 0
