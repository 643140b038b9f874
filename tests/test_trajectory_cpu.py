"""CPU suite: the C-ABI boundary of the trajectory pieces (indexed warp, per-item row gather) -- argument validation only."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_trajectory_symbols_are_declared():
    hdr = open(os.path.join(ROOT, "include", "fusg.h")).read()
    names = set(re.findall(r"\b(fusg_[a-z0-9_]+)\s*\(", hdr))
    for n in ("fusg_warp_fused_idx", "fusg_gather_rows", "fusg_sizeof_gather_seg", "fusg_u8_to_vunet_y"):
        assert n in names, n
    assert re.search(r"#define FUSG_GATHER_MAX_SEGS 8\b", hdr)


def test_gather_seg_struct_matches_c_layout():
    from future_urban_scene_generation_b200 import _lib
    from future_urban_scene_generation_b200.frame_ops import GatherSeg, GATHER_MAX_SEGS
    assert ctypes.sizeof(GatherSeg) == _lib.lib().fusg_sizeof_gather_seg() == 32
    assert GATHER_MAX_SEGS == 8


def _warp_idx(L, index, n_src):
    fake = ctypes.c_void_p(0x10000)
    return L.fusg_warp_fused_idx(fake, index, n_src, fake, fake, fake, fake, fake, fake, None,
                                 fake, fake, fake, fake, fake, 1 << 20, 4, 256, 256, None)


def test_indexed_warp_validates_index_arguments():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    assert _warp_idx(L, None, 3) == -1                           # no index
    assert _warp_idx(L, ctypes.c_void_p(0x20000), 0) == -1       # no source images
    assert _warp_idx(L, ctypes.c_void_p(0x20000), -2) == -1


def _segs(rows, ptr=0x100000):
    from future_urban_scene_generation_b200.frame_ops import GatherSeg
    segs = (GatherSeg * len(rows))()
    for s, rb in zip(segs, rows):
        s.src, s.dst, s.row_bytes, s.n_src = ptr, ptr + 0x100000, rb, 3
    return segs


def test_gather_rows_validates_arguments():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    idx = ctypes.c_void_p(0x300000)
    assert L.fusg_gather_rows(_segs([4096, 20]), 2, idx, 4, None) == -1          # row_bytes % 16 != 0
    assert L.fusg_gather_rows(_segs([0]), 1, idx, 4, None) == -1                 # empty row
    assert L.fusg_gather_rows(_segs([4096] * 9), 9, idx, 4, None) == -1          # more than FUSG_GATHER_MAX_SEGS
    assert L.fusg_gather_rows(_segs([4096], ptr=0x100008), 1, idx, 4, None) == -1    # base not 16-byte aligned
    assert L.fusg_gather_rows(_segs([4096]), 0, idx, 4, None) == -1
    assert L.fusg_gather_rows(_segs([4096]), 1, None, 4, None) == -1
    assert L.fusg_gather_rows(_segs([4096]), 1, idx, 0, None) == -1
    assert L.fusg_gather_rows(None, 1, idx, 4, None) == -1
    assert L.fusg_u8_to_vunet_y(None, None, 1, 256, None) == -1
