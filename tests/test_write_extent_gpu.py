"""Write extent of every libfusg entry point that writes device memory (include/fusg.h).

The other GPU tests check the values a kernel writes.  This file checks WHERE it writes: a stray store past the end of an
output, before its start, past the workspace size the library reports, or into the neighbouring items of an `out=` slice
lands in another tensor of the same step and shows up, if at all, as a small error in an unrelated stage; a byte a kernel
promises to write and skips is stale memory.  Such faults live at the shapes that leave a tail (a partly filled batch tile,
cout < cout_pad, ragged packed outputs, pixel counts that are not a multiple of a vector width), so the cases below run
those shapes.

A module fixture wraps every writing entry point of the ctypes library.  Each call -- from a test below directly or through
the package's wrappers -- then runs three times:

  1. once as given, on the caller's tensors (a refusal is returned as it is);
  2. twice with each output and the workspace replaced by a guarded view: the middle of a larger byte buffer, at a multiple
     of 512 bytes (the alignment of a fresh torch tensor, so alignment-dependent paths -- TMA, 16-byte stores, smallcin --
     are the ones a plain tensor takes), with guard bands of max(64 KiB, the bytes of the batch items one tile can cover).
     Guards and interior hold the canary 0xA5 in the first run and 0x5A in the second.

After each guarded run every guard byte must still hold its canary.  An output the contract calls fully written must come
out byte-identical from both runs (a skipped byte keeps its canary and differs); in a partly written output a byte is either
identical in both runs or held both canaries, and the test names which bytes must be the unwritten ones.  The written bytes
are copied back to the caller's tensors, so every value check below also checks the guarded result.  The workspace passed
is exactly the size the library reports.  For fusg_conv2d the kernel choice and the tcgen05 plan must be the same for the
plain and the guarded descriptors.

The last test parses include/fusg.h and asserts that every entry point that writes device memory was called here.
"""
import ctypes as C
import os
import re
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CANARIES = (0xA5, 0x5A)
ALIGN = 512                       # torch's allocation alignment: guarded views sit at a multiple of it
MIN_GUARD = 64 << 10
HOST_ONLY = {"fusg_version", "fusg_last_error", "fusg_kernel_launches", "fusg_conv2d_set_sm_reserve", "fusg_conv2d_last_plan",
             "fusg_conv2d_select", "fusg_mt19937_advance"}
ES = {0: 2, 1: 4, 2: 2}           # bytes per element of FUSG_DTYPE_BF16 / F32 / F16

STATE = {"case": "-", "inject": None, "log": []}
STATS = {}                        # entry point -> {"cases": set, "guard_bytes": int}


def _round(n, a=ALIGN):
    return (n + a - 1) // a * a


class _case:
    """Names the case of the calls made inside it (failure messages, per-entry-point statistics)."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        STATE["case"], STATE["log"] = self.name, []
        return STATE["log"]

    def __exit__(self, *exc):
        STATE["case"] = "-"


class _Raw:
    """A device byte range as a torch tensor (__cuda_array_interface__), to copy results back to the caller's pointer."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _v(a):
    return a.value if hasattr(a, "value") else a


class Out:
    def __init__(self, label, ptr, nbytes, setter, full=True, item=0, ws=False):
        self.label, self.ptr, self.nbytes, self.set, self.full, self.item, self.ws = label, ptr, int(nbytes), setter, full, int(item), ws
        self.guard = _round(max(MIN_GUARD, self.item))


def _arg(a, i, nbytes, label, full=True, item=0):
    p = _v(a[i])
    if not p:
        return None

    def setter(q):
        a[i] = C.c_void_p(q)
    return Out(label, p, nbytes, setter, full, item)


def _ws(a, i, i_bytes, nbytes):
    """The workspace argument, given exactly the size the library reports."""
    a[i_bytes] = int(nbytes)
    o = _arg(a, i, nbytes, "workspace")
    o.ws = True
    return o


def _dev_ints(torch, ptr, n, dtype):
    return torch.as_tensor(_Raw(ptr, n * np.dtype(dtype).itemsize), device="cuda").cpu().numpy().view(dtype)


# ------------------------------------------------------------------------------------------------ outputs of each entry point
def _warp_outs(a, o, B, H, W, ws_bytes):
    return [_arg(a, o, B * 5 * H * W * 3, "warped", item=5 * H * W * 3), _arg(a, o + 1, B * 14, "vis"), _arg(a, o + 2, B * 5, "plane_j"),
            _arg(a, o + 3, B * 360, "H12"), _ws(a, o + 4, o + 5, ws_bytes)]


def _spec_window(torch, L, a):
    B, H, W = _v(a[19]), _v(a[20]), _v(a[21])
    win = _dev_ints(torch, _v(a[10]), 4 * B, np.int32).reshape(B, 4)
    off = _dev_ints(torch, _v(a[11]), B, np.int64)
    end = int(max(off[b] + 5 * win[b, 2] * win[b, 3] * 3 for b in range(B)))
    return [_arg(a, 13, end, "warped windows", full=False, item=int((5 * win[:, 2] * win[:, 3] * 3).max())),
            _arg(a, 14, B * 14, "vis"), _arg(a, 15, B * 5, "plane_j"), _arg(a, 16, B * 360, "H12"),
            _ws(a, 17, 18, L.fusg_warp_window_workspace_bytes(B, H, W))]


def _spec_resize(torch, L, a):
    B = _v(a[6])
    off = _dev_ints(torch, _v(a[4]), B, np.int64)
    hw = _dev_ints(torch, _v(a[5]), 2 * B, np.int32).reshape(B, 2)
    end = int(max(off[b] + hw[b, 0] * hw[b, 1] * 3 for b in range(B)))
    return [_arg(a, 3, end, "dst", full=False, item=int((hw[:, 0] * hw[:, 1] * 3).max()))]


def _conv_slot_bytes(d, s, Ho, Wo):
    o = d.outs[s]
    es = 4 if o.layout == 1 else ES[d.dtype]
    return d.B * Ho * Wo * d.cout * es * (4 if o.mode == 3 else 1)


def _conv_out_hw(d):
    p = d.pad if d.pad_mode else d.ksize // 2
    return (d.H + 2 * p - d.ksize) // d.stride + 1, (d.W + 2 * p - d.ksize) // d.stride + 1


def _spec_conv(torch, L, a):
    from future_urban_scene_generation_b200.vunet.engine import ConvDesc
    d = a[0]._obj
    d2 = ConvDesc.from_buffer_copy(d)
    a[0] = C.byref(d2)
    Ho, Wo = _conv_out_hw(d)
    outs = []
    for s in range(len(d.outs)):
        if not d.outs[s].ptr:
            continue
        n = _conv_slot_bytes(d, s, Ho, Wo)

        def setter(q, s=s):
            d2.outs[s].ptr = q
        outs.append(Out(f"slot {s}", d.outs[s].ptr, n, setter, full=d.outs[s].mode != 3, item=n // d.B))
    return outs


def _spec_gather(torch, L, a):
    segs = type(a[0]).from_buffer_copy(a[0])
    a[0] = segs
    B, outs = _v(a[3]), []
    for s in range(_v(a[1])):
        def setter(q, s=s):
            segs[s].dst = q
        outs.append(Out(f"segment {s}", segs[s].dst, B * segs[s].row_bytes, setter, item=segs[s].row_bytes))
    return outs


def _spec_randn(torch, L, a):
    tbl = type(a[1]).from_buffer_copy(a[1])
    a[1] = tbl
    outs = []
    for i in range(_v(a[2])):
        e = tbl[i]

        def setter(q, i=i):
            tbl[i].out = q
        outs.append(Out(f"draw {i}", e.out, e.b * e.c * e.h * e.w * 4, setter, item=e.c * e.h * e.w * 4))
    return outs


SPECS = {
    "fusg_warp_fused": lambda t, L, a: _warp_outs(a, 7, _v(a[13]), _v(a[14]), _v(a[15]), L.fusg_warp_workspace_bytes_hw(_v(a[13]), _v(a[14]), _v(a[15]))),
    "fusg_warp_fused_traj": lambda t, L, a: _warp_outs(a, 8, _v(a[14]), _v(a[15]), _v(a[16]), L.fusg_warp_workspace_bytes_hw(_v(a[14]), _v(a[15]), _v(a[16]))),
    "fusg_warp_fused_idx": lambda t, L, a: _warp_outs(a, 10, _v(a[16]), _v(a[17]), _v(a[18]), L.fusg_warp_workspace_bytes_hw(_v(a[16]), _v(a[17]), _v(a[18]))),
    "fusg_warp_fused_window": _spec_window,
    "fusg_step_keypoints": lambda t, L, a: [_arg(a, 7, _v(a[10]) * 288, "kp3d_out"), _arg(a, 8, _v(a[10]) * 192, "kp2d_out"),
                                            _arg(a, 9, _v(a[10]) * 96, "verts")],
    "fusg_visibility": lambda t, L, a: [_arg(a, 3, _v(a[6]) * 7, "vis"), _arg(a, 4, _v(a[6]) * 96, "pts"), _arg(a, 5, _v(a[6]) * 56, "areas")],
    "fusg_get_planes": lambda t, L, a: [_arg(a, 2, _v(a[3]) * 15 * _v(a[4]) * _v(a[5]), "planes", item=15 * _v(a[4]) * _v(a[5]))],
    "fusg_find_homography": lambda t, L, a: [_arg(a, 3, _v(a[5]) * 72, "H"), _arg(a, 4, _v(a[5]), "ok")],
    "fusg_warp_perspective": lambda t, L, a: [_arg(a, 2, _v(a[3]) * 3 * _v(a[4]) * _v(a[5]), "out", item=3 * _v(a[4]) * _v(a[5]))],
    "fusg_conv2d": _spec_conv,
    "fusg_fold_weightnorm": lambda t, L, a: [_arg(a, 2, _v(a[6]) * _v(a[5]) ** 2 * _v(a[7]) * ES[_v(a[8])], "w_out")],
    "fusg_fold_weightnorm_paired": lambda t, L, a: [
        _arg(a, 3, _v(a[9]) * _v(a[8]) ** 2 * 2 * (_v(a[6]) + _v(a[7])) * ES[_v(a[10])], "w_out"), _arg(a, 4, _v(a[9]) * 4, "bias_out")],
    "fusg_nchw_to_nhwc": lambda t, L, a: [_arg(a, 1, _v(a[2]) * _v(a[4]) * _v(a[5]) * _v(a[6]) * ES[_v(a[8])], "out")],
    "fusg_nhwc_to_nchw": lambda t, L, a: [_arg(a, 1, _v(a[2]) * _v(a[3]) * _v(a[4]) * _v(a[5]) * 4, "out")],
    "fusg_to_image": lambda t, L, a: [_arg(a, 1, _v(a[2]) * _v(a[3]) * _v(a[4]) * 3, "out")],
    "fusg_to_image_lab": lambda t, L, a: [_arg(a, 1, _v(a[4]) * _v(a[5]) * _v(a[6]) * 3, "out")],
    "fusg_resize_u8": _spec_resize,
    "fusg_paste_back": lambda t, L, a: [_arg(a, 0, _v(a[9]) * _v(a[10]) * _v(a[11]) * 3, "frames", full=False, item=_v(a[10]) * _v(a[11]) * 3),
                                        _ws(a, 6, 7, L.fusg_paste_workspace_bytes(_v(a[9]), _v(a[10]), _v(a[11])))],
    "fusg_mask_bbox": lambda t, L, a: [_arg(a, 3, _v(a[4]) * 16, "bbox")],
    "fusg_pack_vunet_inputs": lambda t, L, a: [_arg(a, 8, _v(a[10]) * 24 * _v(a[13]) ** 2, "x", item=24 * _v(a[13]) ** 2),
                                               _arg(a, 9, _v(a[10]) * 12 * _v(a[13]) ** 2, "y", item=12 * _v(a[13]) ** 2)],
    "fusg_pack_icn_inputs": lambda t, L, a: [_arg(a, 10, _v(a[11]) * 84 * _v(a[14]) ** 2, "out", item=84 * _v(a[14]) ** 2)],
    "fusg_pack_icn_inputs_window": lambda t, L, a: [_arg(a, 12, _v(a[13]) * 84 * _v(a[16]) ** 2, "out", item=84 * _v(a[16]) ** 2)],
    "fusg_u8_to_vunet_inputs": lambda t, L, a: [_arg(a, 3, _v(a[5]) * 24 * _v(a[6]) ** 2, "x"), _arg(a, 4, _v(a[5]) * 12 * _v(a[6]) ** 2, "y")],
    "fusg_u8_to_vunet_y": lambda t, L, a: [_arg(a, 1, _v(a[2]) * 12 * _v(a[3]) ** 2, "y")],
    "fusg_gather_rows": _spec_gather,
    "fusg_randn_mt19937": _spec_randn,
    "fusg_nchw_to_nhwc_reflect": lambda t, L, a: [
        _arg(a, 1, _v(a[2]) * (_v(a[4]) + 2 * _v(a[7])) * (_v(a[5]) + 2 * _v(a[7])) * _v(a[6]) * ES[_v(a[8])], "out")],
    "fusg_norm_stats": lambda t, L, a: [_arg(a, 1, (_v(a[2]) * _v(a[5]) * _v(a[4]) * 2 + _v(a[2]) * _v(a[4])) * 4, "partial")],
    "fusg_norm_finalize": lambda t, L, a: [_arg(a, 3, _v(a[4]) * _v(a[6]) * 8, "ss")],
    "fusg_norm_apply": lambda t, L, a: [_arg(a, 4, _v(a[5]) * (_v(a[10]) * _v(a[6]) + 2 * _v(a[11])) * (_v(a[10]) * _v(a[7]) + 2 * _v(a[11]))
                                             * _v(a[8]) * ES[_v(a[12])], "out")],
    "fusg_elu": lambda t, L, a: [_arg(a, 1, _v(a[2]) * ES[_v(a[3])], "out")],
    "fusg_render_normals": lambda t, L, a: [
        _arg(a, 10, _v(a[14]) * _v(a[15]) * _v(a[16]) * 3, "normals", item=_v(a[15]) * _v(a[16]) * 3),
        _arg(a, 11, _v(a[14]) * _v(a[15]) * _v(a[16]), "mask", item=_v(a[15]) * _v(a[16])),
        _ws(a, 12, 13, L.fusg_render_workspace_bytes(_v(a[14]), _v(a[4]), _v(a[15]), _v(a[16])))],
}


# ------------------------------------------------------------------------------------------------ the guarded call
def _first(mask):
    idx = mask.nonzero().flatten()
    return int(idx.numel()), (int(idx[0]) if idx.numel() else -1), (int(idx[-1]) if idx.numel() else -1)


def _check_guards(name, o, buf, canary):
    n, _, last = _first(buf[:o.guard] != canary)
    if n:
        raise AssertionError(f"{name} [{STATE['case']}] {o.label}: {n} guard byte(s) before the start of the {o.nbytes}-byte view were "
                             f"written, nearest at offset {last - o.guard:+d} from the start (canary 0x{canary:02X})")
    n, first, _ = _first(buf[o.guard + o.nbytes:] != canary)
    if n:
        raise AssertionError(f"{name} [{STATE['case']}] {o.label}: {n} guard byte(s) past the end of the {o.nbytes}-byte view were "
                             f"written, nearest at offset {first:+d} from the end (canary 0x{canary:02X})")


def _guarded_call(torch, L, name, orig, args):
    from future_urban_scene_generation_b200 import _lib
    rc = orig(*args)
    if rc != 0:
        return rc
    torch.cuda.synchronize()
    a = list(args)
    outs = [o for o in SPECS[name](torch, L, a) if o is not None]
    if name == "fusg_conv2d":
        d = args[0]._obj
        impl = L.fusg_conv2d_select(args[0]) if d.impl == 0 else d.impl
        plan = _lib.conv_last_plan() if impl == 1 else None
        if plan:                                    # a whole batch tile of missed masking must land in the guard
            Ho, Wo = _conv_out_hw(d)
            trows = 128 * plan["msub"]
            Wt = min(Wo, 128)
            Bt = trows // (Wt * min(trows // Wt, Ho))
            for o in outs:
                o.guard = _round(max(MIN_GUARD, Bt * o.item))
    runs = [[] for _ in outs]
    for k, c in enumerate(CANARIES):
        bufs = []
        for o in outs:
            buf = torch.full((2 * o.guard + o.nbytes,), c, dtype=torch.uint8, device="cuda")
            o.set(buf.data_ptr() + o.guard)
            bufs.append(buf)
        rc2 = orig(*a)
        assert rc2 == 0, f"{name} [{STATE['case']}]: returned {rc2} on guarded views after 0 on the caller's tensors"
        torch.cuda.synchronize()
        if STATE["inject"] is not None:
            STATE["inject"](k, name, outs, bufs)
        for o, buf, r in zip(outs, bufs, runs):
            _check_guards(name, o, buf, c)
            if not o.ws:
                r.append(buf[o.guard:o.guard + o.nbytes].clone())
    if name == "fusg_conv2d":
        d2 = a[0]._obj
        assert L.fusg_conv2d_select(a[0]) == L.fusg_conv2d_select(args[0]), f"{name} [{STATE['case']}]: the guarded view changed the kernel"
        if plan:
            assert _lib.conv_last_plan() == plan, f"{name} [{STATE['case']}]: the guarded view changed the plan {plan} -> {_lib.conv_last_plan()}"
        del d2
    st = STATS.setdefault(name, {"cases": set(), "guard_bytes": 0})
    st["cases"].add(STATE["case"])
    for o, r in zip(outs, runs):
        st["guard_bytes"] += 2 * 2 * o.guard
        if o.ws:
            continue
        r0, r1 = r
        same = r0 == r1
        unwritten = (r0 == CANARIES[0]) & (r1 == CANARIES[1])
        bad = ~same if o.full else ~same & ~unwritten
        n, first, _ = _first(bad)
        if n:
            what = "not fully written" if o.full else "written differently in the two runs (a value depends on stale memory)"
            raise AssertionError(f"{name} [{STATE['case']}] {o.label}: {what}: {n} of {o.nbytes} byte(s), first at offset {first} "
                                 f"(0x{int(r0[first]):02X} after the 0x{CANARIES[0]:02X} run, 0x{int(r1[first]):02X} after the "
                                 f"0x{CANARIES[1]:02X} run)")
        dst = torch.as_tensor(_Raw(o.ptr, o.nbytes), device="cuda")
        if o.full:
            dst.copy_(r1)
        else:
            dst[~unwritten] = r1[~unwritten]
        STATE["log"].append(dict(name=name, label=o.label, runs=(r0, r1), unwritten=unwritten))
    torch.cuda.synchronize()
    return rc


@pytest.fixture(scope="module", autouse=True)
def guarded(cuda):
    from future_urban_scene_generation_b200 import _lib
    torch = cuda
    L = _lib.lib()
    with pytest.MonkeyPatch.context() as mp:
        for name in SPECS:
            orig = getattr(L, name)
            mp.setattr(L, name, (lambda n, f: lambda *args: _guarded_call(torch, L, n, f, args))(name, orig))
        yield L
    print("\nwrite extent: cases and guard bytes checked per entry point")
    for name in sorted(STATS):
        print(f"  {name:32s} {len(STATS[name]['cases']):3d} cases {STATS[name]['guard_bytes']:>14,d} guard bytes")


def _unwritten(log, name, label=None):
    hits = [e for e in log if e["name"] == name and (label is None or e["label"] == label)]
    assert hits, f"no guarded {name} {label or ''} call in this case"
    return hits[-1]["unwritten"]


def _bytes_of(torch, elem_mask, es):
    return elem_mask.reshape(-1, 1).expand(-1, es).reshape(-1)


# ================================================================================================ 2. the harness can fail
def test_harness_catches_a_byte_past_the_end(cuda, guarded):
    torch = cuda
    from future_urban_scene_generation_b200 import _lib

    def one_past(k, name, outs, bufs):
        o, buf = outs[0], bufs[0]
        buf[o.guard + o.nbytes] = 0
    x = torch.zeros(1, 3, 7, 9, device="cuda")
    out = torch.empty(1, 7, 9, 3, dtype=torch.uint8, device="cuda")
    STATE["inject"] = one_past
    try:
        with _case("self-test one byte past the end"):
            with pytest.raises(AssertionError, match=r"fusg_to_image \[self-test one byte past the end\] out: 1 guard byte\(s\) past the end "
                                                     r"of the 189-byte view were written, nearest at offset \+0 from the end"):
                guarded.fusg_to_image(_lib.ptr(x), _lib.ptr(out), 1, 7, 9, _lib.stream_ptr(torch))
    finally:
        STATE["inject"] = None


def test_harness_catches_a_skipped_byte(cuda, guarded):
    torch = cuda
    from future_urban_scene_generation_b200 import _lib

    def skip(k, name, outs, bufs):
        if k == 1:                                  # the second run "skips" byte 100: it keeps that run's canary
            bufs[0][outs[0].guard + 100] = CANARIES[1]
    x = torch.zeros(1, 3, 7, 9, device="cuda")      # every byte 127: never either canary
    out = torch.empty(1, 7, 9, 3, dtype=torch.uint8, device="cuda")
    STATE["inject"] = skip
    try:
        with _case("self-test skipped byte"):
            with pytest.raises(AssertionError, match=r"fusg_to_image \[self-test skipped byte\] out: not fully written: 1 of 189 byte\(s\), "
                                                     r"first at offset 100"):
                guarded.fusg_to_image(_lib.ptr(x), _lib.ptr(out), 1, 7, 9, _lib.stream_ptr(torch))
    finally:
        STATE["inject"] = None


# ================================================================================================ 3. fusg_conv2d
TD = {"bf16": 0, "fp32": 1, "fp16": 2}
# name: B, H(=W unless given), cins, cout, k, stride, dtype, impl, mode, slots (source, elu, layout), residual, noise, extra
CONV_CASES = [
    # partly filled last batch tile (derived Bt > 1, B % Bt != 0)
    dict(name="plain fe1 B=5 8x8", B=5, H=8, cins=(128,), cout=128, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(msub=1, fast_epi=1), Bt=2),
    dict(name="plain fe0 noise+fp32 B=5 8x8", B=5, H=8, cins=(128,), cout=128, mode=0, slots=((1, 0, 0), (1, 1, 0), (0, 0, 1), (1, 0, 1)),
         noise=True, plan=dict(fast_epi=0), Bt=2),
    dict(name="d2s B=33 4x4", B=33, H=4, cins=(128,), cout=128, mode=1, slots=((0, 0, 0), (0, 1, 0)), plan=dict(fast_epi=1), Bt=8),
    dict(name="d2s fp32 slot B=5 8x8", B=5, H=8, cins=(128,), cout=128, mode=1, slots=((0, 0, 1),), plan=dict(fast_epi=0), Bt=2),
    dict(name="s2d B=5 8x8", B=5, H=8, cins=(128,), cout=128, mode=2, slots=((0, 0, 0), (0, 1, 0), (0, 0, 1)), residual=True,
         plan=dict(fast_epi=0), Bt=2),
    dict(name="s2d fe1 B=33 4x4", B=33, H=4, cins=(128,), cout=128, mode=2, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(fast_epi=1), Bt=8),
    dict(name="d2s_block noise B=33 2x2", B=33, H=2, cins=(512,), cout=128, mode=3, blk=2, slots=((1, 0, 0), (1, 1, 0), (1, 0, 1)),
         noise=True, plan=dict(fast_epi=0), Bt=32),
    dict(name="d2s_block fe1 B=5 8x8", B=5, H=8, cins=(128,), cout=128, mode=3, blk=1, slots=((0, 0, 0), (0, 1, 0)), plan=dict(fast_epi=1), Bt=2),
    dict(name="ksplit B=33 2x2", B=33, H=2, cins=(512, 512), cout=512, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(ksplit=8), Bt=32),
    dict(name="unpair fe3 cout=6 B=5 8x8", B=5, H=8, cins=(32,), cout=6, mode=4, slots=((0, 0, 1),), plan=dict(fast_epi=3), Bt=2),
    dict(name="fp16 B=5 8x8", B=5, H=8, cins=(64,), cout=64, dtype="fp16", mode=0, slots=((0, 0, 0),), Bt=2),
    # an fp16 raw NHWC slot next to another output: the general tcgen05 epilogue stores bf16, so AUTO must pick the direct kernel
    dict(name="fp16 raw+fp32 auto B=5 8x8", B=5, H=8, cins=(64,), cout=64, dtype="fp16", impl=0, mode=0, slots=((0, 0, 0), (0, 0, 1)),
         expect_impl=2),
    dict(name="fp16 cout=3 B=33 4x4", B=33, H=4, cins=(64,), cout=3, dtype="fp16", mode=0, slots=((0, 2, 1),), Bt=8),
    # the large-frame variants (their plans need Bt = 1)
    dict(name="fe2 staged B=3 32x32", B=3, H=32, cins=(128,), cout=128, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(fast_epi=2)),
    dict(name="halo k=3 cat64 B=4 256", B=4, H=256, cins=(64, 64), cout=64, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(halo=1, w_resident=0)),
    dict(name="halo+w_resident B=4 256", B=4, H=256, cins=(64,), cout=64, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(halo=1, w_resident=1)),
    dict(name="fused under halo B=4 256", B=4, H=256, cins=(64, 64), cout=64, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         fused=True, plan=dict(halo=1)),
    dict(name="pair B=10 128", B=10, H=128, cins=(128,), cout=128, mode=0, slots=((0, 0, 0), (0, 1, 0)), residual=True,
         plan=dict(msub=2, pair=1)),
    dict(name="msub2 no halo s2 B=10 256", B=10, H=256, cins=(128,), cout=128, stride=2, mode=0, slots=((0, 0, 0), (0, 1, 0)),
         plan=dict(msub=2, halo=0, pair=0)),
    dict(name="halo k=5 fp16 bordered B=4 256", B=4, H=256, cins=(128,), cout=64, k=5, dtype="fp16", pad_mode=1, pad=2, border=2,
         slots=((0, 0, 0),), plan=dict(halo=1)),
    dict(name="halo k=7 fp16 bordered B=4 256", B=4, H=256, cins=(64,), cout=64, k=7, dtype="fp16", pad_mode=1, pad=3, border=3,
         slots=((0, 0, 0),), plan=dict(halo=1)),
    # direct kernel
    dict(name="direct fp32 80x96 cout=3", B=2, H=80, W=96, cins=(32,), cout=3, dtype="fp32", impl=2, slots=((0, 0, 1), (0, 2, 1))),
    dict(name="direct fp32 7x9 s2", B=3, H=7, W=9, cins=(16,), cout=32, stride=2, dtype="fp32", impl=2, slots=((0, 0, 0), (0, 1, 0), (0, 0, 1)),
         residual=True),
    dict(name="direct bf16 7x9 s2 cout=3", B=3, H=7, W=9, cins=(32,), cout=3, stride=2, impl=2, slots=((0, 0, 0), (0, 0, 1))),
    dict(name="direct bf16 80x96 noise", B=1, H=80, W=96, cins=(32, 32), cout=32, impl=2, slots=((0, 0, 0), (1, 1, 0), (1, 0, 1)), noise=True),
    dict(name="direct fp32 bordered 7x9", B=2, H=7, W=9, cins=(16,), cout=3, k=3, dtype="fp32", impl=2, pad_mode=1, pad=1, border=2,
         slots=((0, 0, 1),)),
    dict(name="direct bf16 bordered s2 7x9", B=3, H=7, W=9, cins=(32,), cout=16, k=3, stride=2, impl=2, pad_mode=1, pad=1, border=3,
         slots=((0, 0, 0),)),
]


def _slot_shape(mode, layout, B, Ho, Wo, cout):
    nhwc = {0: (B, Ho, Wo, cout), 1: (B, 2 * Ho, 2 * Wo, cout // 4), 2: (B, Ho // 2, Wo // 2, 4 * cout), 3: (B, 2 * Ho, 2 * Wo, cout)}
    nchw = {0: (B, cout, Ho, Wo), 1: (B, cout // 4, 2 * Ho, 2 * Wo), 2: (B, 4 * cout, Ho // 2, Wo // 2), 3: (B, cout, 2 * Ho, 2 * Wo),
            4: (B, cout // 2, Ho, 2 * Wo)}
    return nchw[mode] if layout == 1 else nhwc[mode]


def _place(torch, t, mode, blk):
    from oracle import vunet_oracle as VO
    if mode == 1:
        return VO.depth_to_space(t)
    if mode == 2:
        return VO.space_to_depth(t)
    if mode == 3:
        full = torch.zeros(t.shape[0], 4 * t.shape[1], t.shape[2], t.shape[3], dtype=t.dtype, device=t.device)
        full[:, blk * t.shape[1]:(blk + 1) * t.shape[1]] = t
        return VO.depth_to_space(full)
    if mode == 4:
        B, c, H, W = t.shape
        return t.view(B, 2, c // 2, H, W).permute(0, 2, 3, 4, 1).reshape(B, c // 2, H, 2 * W)
    return t


@pytest.mark.parametrize("case", CONV_CASES, ids=[c["name"] for c in CONV_CASES])
def test_conv2d(cuda, guarded, case):
    torch = cuda
    import torch.nn.functional as F
    from future_urban_scene_generation_b200 import _lib
    from future_urban_scene_generation_b200.vunet.engine import ConvDesc
    from oracle import launch_oracle as LO
    c = dict(W=None, k=3, stride=1, dtype="bf16", impl=1, mode=0, blk=0, residual=False, noise=False, pad_mode=0, pad=0, border=0,
             fused=False, plan={}, Bt=None, expect_impl=None)
    c.update(case)
    B, H, W, k, cout = c["B"], c["H"], c["W"] or c["H"], c["k"], c["cout"]
    td = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[c["dtype"]]
    g = torch.Generator().manual_seed(zlib.crc32(c["name"].encode()))
    bd = c["border"] if c["pad_mode"] else 0
    xs = [torch.randn(B, H + 2 * bd, W + 2 * bd, ci, generator=g).to(td).cuda() for ci in c["cins"]]
    cin = sum(c["cins"])
    w = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    if c["fused"]:                                 # a 1x1 NiN over in1 folded into the centre tap of the 3x3 over in0
        centre = w[:, c["cins"][0]:, k // 2, k // 2].clone()
        w[:, c["cins"][0]:] = 0
        w[:, c["cins"][0]:, k // 2, k // 2] = centre
    w = w.to(td).cuda()
    cout_pad = (cout + 15) // 16 * 16
    wp = torch.zeros(cout_pad, k * k, cin, dtype=td, device="cuda")
    wp[:cout] = w.permute(0, 2, 3, 1).reshape(cout, k * k, cin)
    bias = torch.zeros(cout_pad, device="cuda")
    bias[:cout] = torch.randn(cout, generator=g).cuda() * 0.1
    p = c["pad"] if c["pad_mode"] else k // 2
    Ho, Wo = (H + 2 * p - k) // c["stride"] + 1, (W + 2 * p - k) // c["stride"] + 1
    res = torch.randn(B, Ho, Wo, cout, generator=g).to(td).cuda() if c["residual"] else None
    noise = torch.randn(B, Ho, Wo, cout, generator=g).cuda() if c["noise"] else None
    d = ConvDesc()
    d.in0, d.c0, d.pitch0 = xs[0].data_ptr(), c["cins"][0], c["cins"][0]
    if len(xs) > 1:
        d.in1, d.c1, d.pitch1 = xs[1].data_ptr(), c["cins"][1], c["cins"][1]
    d.B, d.H, d.W, d.ksize, d.stride = B, H, W, k, c["stride"]
    d.weight, d.bias, d.cout, d.cout_pad = wp.data_ptr(), bias.data_ptr(), cout, cout_pad
    d.residual = res.data_ptr() if res is not None else None
    d.noise = noise.data_ptr() if noise is not None else None
    d.pad_mode, d.pad, d.border = c["pad_mode"], c["pad"], c["border"]
    if c["fused"]:
        d.zero_kblocks = LO.zero_kblocks(wp.float().cpu().numpy())
        assert d.zero_kblocks
    outs = []
    for s, (src, elu, layout) in enumerate(c["slots"]):
        t = torch.full(_slot_shape(c["mode"], layout, B, Ho, Wo, cout), float("nan"), dtype=torch.float32 if layout else td, device="cuda")
        d.outs[s].ptr, d.outs[s].source, d.outs[s].elu, d.outs[s].layout = t.data_ptr(), src, elu, layout
        d.outs[s].mode, d.outs[s].blk = c["mode"], c["blk"]
        outs.append(t)
    d.dtype, d.impl = TD[c["dtype"]], c["impl"]
    L = guarded
    if c["expect_impl"] is not None:
        assert L.fusg_conv2d_select(C.byref(d)) == c["expect_impl"]
    with _case(c["name"]) as log:
        _lib.check(L.fusg_conv2d(C.byref(d), _lib.stream_ptr(torch)), "fusg_conv2d")
        torch.cuda.synchronize()
    if c["impl"] == 1:
        plan = _lib.conv_last_plan()
        for key, val in c["plan"].items():
            assert plan[key] == val, (c["name"], plan)
        trows = 128 * plan["msub"]
        Wt = min(Wo, 128)
        Bt = trows // (Wt * min(trows // Wt, Ho))
        if c["Bt"] is not None:
            assert Bt == c["Bt"] and B % Bt != 0, (c["name"], Bt)
    # fp64 reference of the same (rounded) operands
    x = torch.cat(xs, -1).double().permute(0, 3, 1, 2)
    if c["pad_mode"]:
        x = x[:, :, bd - p:bd + H + p, bd - p:bd + W + p]
    y = F.conv2d(x, w.double(), bias[:cout].double(), stride=c["stride"], padding=0 if c["pad_mode"] else p)
    if res is not None:
        y = y + res.double().permute(0, 3, 1, 2)
    z = y + noise.double().permute(0, 3, 1, 2) if noise is not None else None
    scale = max(1.0, y.abs().max().item(), z.abs().max().item() if z is not None else 0.0)
    for s, ((src, elu, layout), t) in enumerate(zip(c["slots"], outs)):
        base = z if src else y
        val = F.elu(base) if elu == 1 else (torch.tanh(base) if elu == 2 else base)
        ref = _place(torch, val, c["mode"], c["blk"])
        got = (t if layout else t.permute(0, 3, 1, 2)).double()
        if c["mode"] == 3:                          # one quadrant written; the other three must be the canary in both runs
            q = torch.zeros(2 * Ho, 2 * Wo, dtype=torch.bool, device="cuda")
            q[c["blk"] // 2::2, c["blk"] % 2::2] = True
            quad = q.expand(B, 2 * Ho, 2 * Wo).unsqueeze(-1).expand(B, 2 * Ho, 2 * Wo, cout)
            quad = quad if layout == 0 else quad.permute(0, 3, 1, 2)
            es = 4 if layout else ES[d.dtype]
            assert torch.equal(_unwritten(log, "fusg_conv2d", f"slot {s}"), _bytes_of(torch, ~quad.contiguous(), es)), (c["name"], s)
            quad_nchw = quad if layout else quad.permute(0, 3, 1, 2)
            got, ref = got[quad_nchw], ref[quad_nchw]
        if c["dtype"] == "fp32":
            tol = 2e-5
        elif layout == 1:
            tol = 2e-3 * scale
        else:
            tol = (1.0 / 64 if elu else 1.0 / 128) * scale
        err = (got - ref).abs().max().item()
        assert err < tol, (c["name"], s, err, tol)


@pytest.mark.parametrize("cout", [32, 128])
def test_conv2d_smallcin(cuda, guarded, cout):
    """FUSG_IMPL_SMALLCIN at pixel counts that are not a multiple of ppc * SC_PIX (B*H*W = 189)."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    from future_urban_scene_generation_b200.vunet.engine import ConvDesc
    g = torch.Generator().manual_seed(cout)
    B, H, W, cin = 3, 7, 9, 6
    assert (B * H * W) % (256 // (cout // 8) * 4) != 0
    xin = torch.zeros(B, H, W, 16, dtype=torch.bfloat16, device="cuda")
    xin[..., :cin] = torch.randn(B, H, W, cin, generator=g).cuda().bfloat16()
    w = torch.zeros(cout, 1, 64, dtype=torch.bfloat16, device="cuda")
    w[:, 0, :cin] = (torch.randn(cout, cin, generator=g) / cin ** 0.5).cuda().bfloat16()
    bias = (torch.randn(cout, generator=g) * 0.1).cuda()
    raw = torch.empty(B, H, W, cout, dtype=torch.bfloat16, device="cuda")
    elu = torch.empty_like(raw)
    d = ConvDesc()
    d.in0, d.c0, d.pitch0, d.cphys0, d.cin_real = xin.data_ptr(), 64, 16, 16, cin
    d.B, d.H, d.W, d.ksize, d.stride = B, H, W, 1, 1
    d.weight, d.bias, d.cout, d.cout_pad = w.data_ptr(), bias.data_ptr(), cout, cout
    d.outs[0].ptr, d.outs[1].ptr, d.outs[1].elu = raw.data_ptr(), elu.data_ptr(), 1
    d.dtype, d.impl = 0, 0
    assert guarded.fusg_conv2d_select(C.byref(d)) == 3
    with _case(f"smallcin cout={cout} 3x7x9"):
        _lib.check(guarded.fusg_conv2d(C.byref(d), _lib.stream_ptr(torch)), "fusg_conv2d")
        torch.cuda.synchronize()
    ref = torch.einsum("bhwc,oc->bhwo", xin[..., :cin].double(), w[:, 0, :cin].double()) + bias.double()
    assert (raw.double() - ref).abs().max().item() < 1.0 / 128 * max(1.0, ref.abs().max().item())
    assert (elu.double() - torch.nn.functional.elu(raw.double())).abs().max().item() < 1.0 / 128


# ================================================================================================ 3. weight folds and layouts
def _ulps(torch, a, b):
    ia, ib = a.view(torch.int16).int(), b.view(torch.int16).int()
    return (ia - ib).abs()


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_fold_weightnorm(cuda, guarded, dtype):
    """Pad rows (cout_pad > cout) and pad columns (cin_pad > cin) are written as zeros; at most 1 ulp from the fp64 fold, and
    only at rounding midpoints."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    from oracle import launch_oracle as LO
    td = {"bf16": torch.bfloat16, "fp16": torch.float16}[dtype]
    g = torch.Generator().manual_seed(7)
    st = _lib.stream_ptr(torch)

    def compare(got, want64):
        want = torch.from_numpy(want64).to(td)
        _, step = LO.rounded(torch.from_numpy(want64), td)
        dd = _ulps(torch, got.cpu(), want)
        assert int(dd.max()) <= 1
        amb = step > 0 if step is not None else torch.zeros_like(dd, dtype=torch.bool)
        assert not bool(((dd > 0) & ~amb).any())
    for cout, cin, k, cout_pad, cin_pad in ((3, 21, 3, 16, 32), (5, 6, 1, 16, 16), (40, 37, 3, 48, 64)):
        v = torch.randn(cout, cin, k, k, generator=g)
        gn = torch.rand(cout, generator=g) + 0.5
        out = torch.full((cout_pad, k * k, cin_pad), float("nan"), dtype=td, device="cuda")
        vd, gd = v.cuda(), gn.cuda()
        with _case(f"fold {dtype} {cout}x{cin}x{k} -> {cout_pad}x{cin_pad}"):
            _lib.check(guarded.fusg_fold_weightnorm(_lib.ptr(vd), _lib.ptr(gd), _lib.ptr(out), cout, cin, k, cout_pad, cin_pad,
                                                    TD[dtype], st), "fold")
            torch.cuda.synchronize()
        compare(out, LO.pack_plain(LO.fold(v, gn.view(-1, 1, 1, 1)).cpu().numpy(), cout_pad, cin_pad))
    for cout, c0, c1, k, cout_pad in ((3, 32, 0, 3, 16), (5, 16, 16, 1, 16)):
        v = torch.randn(cout, c0 + c1, k, k, generator=g)
        gn = torch.rand(cout, generator=g) + 0.5
        b = torch.randn(cout, generator=g)
        out = torch.full((cout_pad, k * k, 2 * (c0 + c1)), float("nan"), dtype=td, device="cuda")
        bout = torch.full((cout_pad,), float("nan"), device="cuda")
        vd, gd, bd = v.cuda(), gn.cuda(), b.cuda()
        with _case(f"fold paired {dtype} {cout}x{c0}+{c1}x{k} -> {cout_pad}"):
            _lib.check(guarded.fusg_fold_weightnorm_paired(_lib.ptr(vd), _lib.ptr(gd), _lib.ptr(bd), _lib.ptr(out), _lib.ptr(bout),
                                                           cout, c0, c1, k, cout_pad, TD[dtype], st), "fold paired")
            torch.cuda.synchronize()
        want, want_b = LO.pack_paired(LO.fold(v, gn.view(-1, 1, 1, 1)).cpu().numpy(), b.double().numpy(), c0, c1, cout_pad)
        compare(out, want)
        assert torch.equal(bout.cpu(), torch.from_numpy(want_b).float())


# ================================================================================================ 3. layout and pointwise kernels
@pytest.mark.parametrize("B,C_,H,W,cpad,elu,dtype", [
    (2, 21, 7, 9, 32, 0, "bf16"),        # split path: npix < 16384, cpad > C
    (1, 6, 160, 128, 16, 0, "bf16"),     # plain path
    (3, 5, 33, 33, 16, 1, "fp16"),       # ELU
    (1, 3, 7, 9, 8, 0, "fp32"),
])
def test_nchw_to_nhwc(cuda, guarded, B, C_, H, W, cpad, elu, dtype):
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    td = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[dtype]
    x = torch.randn(B, C_, H, W, generator=torch.Generator().manual_seed(B * C_)).cuda()
    out = torch.empty(B, H, W, cpad, dtype=td, device="cuda")
    with _case(f"nchw_to_nhwc {B}x{C_}x{H}x{W} cpad {cpad} elu {elu} {dtype}"):
        _lib.check(guarded.fusg_nchw_to_nhwc(_lib.ptr(x), _lib.ptr(out), B, C_, H, W, cpad, elu, TD[dtype], _lib.stream_ptr(torch)), "nchw_to_nhwc")
        torch.cuda.synchronize()
    assert not bool(out[..., C_:].float().any())                       # pad channels fully written as zeros
    ref = x.permute(0, 2, 3, 1)
    if elu:
        ref = torch.nn.functional.elu(ref.double())
        assert (out[..., :C_].double() - ref).abs().max().item() < 1.0 / 64 * max(1.0, ref.abs().max().item())
    else:
        assert torch.equal(out[..., :C_], ref.to(td))


@pytest.mark.parametrize("border", [1, 2, 3])
def test_nchw_to_nhwc_reflect(cuda, guarded, border):
    torch = cuda
    import torch.nn.functional as F
    from future_urban_scene_generation_b200 import _lib
    B, C_, H, W, cpad = 2, 21, 7, 9, 32
    x = torch.randn(B, C_, H, W, generator=torch.Generator().manual_seed(border)).cuda()
    out = torch.empty(B, H + 2 * border, W + 2 * border, cpad, dtype=torch.bfloat16, device="cuda")
    with _case(f"reflect border {border}"):
        _lib.check(guarded.fusg_nchw_to_nhwc_reflect(_lib.ptr(x), _lib.ptr(out), B, C_, H, W, cpad, border, 0, _lib.stream_ptr(torch)), "reflect")
        torch.cuda.synchronize()
    ref = F.pad(x, (border,) * 4, mode="reflect").permute(0, 2, 3, 1).to(torch.bfloat16)
    assert torch.equal(out[..., :C_], ref) and not bool(out[..., C_:].float().any())


@pytest.mark.parametrize("B", [1, 3])
def test_nhwc_to_nchw_to_image(cuda, guarded, B):
    """pitch > C; H*W*3 = 189 is not a multiple of 256."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    from oracle import frame_oracle as FO
    H, W, C_, pitch = 7, 9, 3, 16
    st = _lib.stream_ptr(torch)
    g = torch.Generator().manual_seed(B)
    x = (torch.rand(B, H, W, pitch, generator=g) * 2.4 - 1.2).to(torch.bfloat16).cuda()
    nchw = torch.empty(B, C_, H, W, device="cuda")
    with _case(f"nhwc_to_nchw B={B} pitch {pitch}"):
        _lib.check(guarded.fusg_nhwc_to_nchw(_lib.ptr(x), _lib.ptr(nchw), B, C_, H, W, pitch, 0, st), "nhwc_to_nchw")
        torch.cuda.synchronize()
    assert torch.equal(nchw, x[..., :C_].permute(0, 3, 1, 2).float())
    img = torch.empty(B, H, W, 3, dtype=torch.uint8, device="cuda")
    with _case(f"to_image B={B} 7x9"):
        _lib.check(guarded.fusg_to_image(_lib.ptr(nchw), _lib.ptr(img), B, H, W, st), "to_image")
        torch.cuda.synchronize()
    xf = nchw.cpu().numpy().astype(np.float32)
    ref = np.clip((xf + np.float32(1)) / np.float32(2) * np.float32(255), 0, 255).astype(np.uint8).transpose(0, 2, 3, 1)
    assert np.array_equal(img.cpu().numpy(), ref)
    z = np.load(os.path.join(ROOT, "future_urban_scene_generation_b200", "data", "lab8.npz"))
    yf = torch.from_numpy(z["lab_to_yf"].astype(np.uint16).view(np.int16)).cuda()
    ig = torch.from_numpy(z["inv_gamma"].astype(np.uint8)).cuda()
    lab = torch.empty(B, H, W, 3, dtype=torch.uint8, device="cuda")
    with _case(f"to_image_lab B={B} 7x9"):
        _lib.check(guarded.fusg_to_image_lab(_lib.ptr(nchw), _lib.ptr(lab), _lib.ptr(yf), _lib.ptr(ig), B, H, W, st), "to_image_lab")
        torch.cuda.synchronize()
    for b in range(B):
        assert np.array_equal(lab[b].cpu().numpy(), FO.to_image_lab(xf[b])), b


@pytest.mark.parametrize("n", [1, 257, 1000003])
@pytest.mark.parametrize("dtype", ["bf16", "fp16", "fp32"])
def test_elu(cuda, guarded, n, dtype):
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    td = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[dtype]
    x = (torch.randn(n, generator=torch.Generator().manual_seed(n)) * 3).to(td).cuda()
    out = torch.empty_like(x)
    with _case(f"elu n={n} {dtype}"):
        _lib.check(guarded.fusg_elu(_lib.ptr(x), _lib.ptr(out), n, TD[dtype], _lib.stream_ptr(torch)), "elu")
        torch.cuda.synchronize()
    ref = torch.nn.functional.elu(x.double())
    assert (out.double() - ref).abs().max().item() < (2e-5 if dtype == "fp32" else 1.0 / 64 * max(1.0, ref.abs().max().item()))


# ================================================================================================ 3. ICN norm passes
@pytest.mark.parametrize("up,border", [(1, 0), (2, 1), (1, 2), (2, 3)])
def test_norm_passes(cuda, guarded, up, border):
    """B = 3, H*W = 37*41 = 1517 pixels in nsplit = 2 splits (a tail), instance norm with a residual and LayerNorm."""
    torch = cuda
    import torch.nn.functional as F
    from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
    from oracle import icn_oracle as IO
    m = G_Resnet(21, dtype="fp16")
    m.load_state_dict(IO.make_state_dict(0), strict=True)
    e = m.cuda().eval().engine()
    g = torch.Generator().manual_seed(up * 10 + border)
    B, C_, H, W = 3, 64, 37, 41
    assert (H * W) // 512 == 2 and (H * W) % 2
    x = torch.randn(B, C_, H, W, generator=g).cuda() * 2 + 0.5
    raw = x.permute(0, 2, 3, 1).contiguous().to(e.tdtype)
    rawf = raw.float().permute(0, 3, 1, 2)
    with _case(f"norm inst B=3 37x41 up {up} border {border}"):
        resid = e.to_padded(torch.randn(B, C_, H, W, generator=g).cuda(), 1)
        residf = resid.t[:, 1:-1, 1:-1, :].float().permute(0, 3, 1, 2)
        out = e.norm("t", raw, H, W, "inst", residual=resid, relu=True, up=up, border=border)
        torch.cuda.synchronize()
    want = F.relu(F.instance_norm(rawf.double(), eps=1e-5) + residf.double())
    want = F.interpolate(want, scale_factor=up, mode="nearest") if up > 1 else want
    want = (F.pad(want, (border,) * 4, mode="reflect") if border else want).permute(0, 2, 3, 1)
    assert out.t.shape == want.shape
    assert (out.t.double() - want).abs().max().item() <= 1e-3 * max(1.0, want.abs().max().item())
    gamma, beta = torch.rand(C_, generator=g).cuda(), torch.randn(C_, generator=g).cuda() * 0.1
    with _case(f"norm ln B=3 37x41 up {up} border {border}"):
        out = e.norm("t", raw, H, W, "ln", gamma, beta, relu=False, up=up, border=border)
        torch.cuda.synchronize()
    flat = rawf.double().reshape(B, -1)
    want = (rawf.double() - flat.mean(1).view(-1, 1, 1, 1)) / (flat.std(1).view(-1, 1, 1, 1) + 1e-5)
    want = want * gamma.double().view(1, -1, 1, 1) + beta.double().view(1, -1, 1, 1)
    want = F.interpolate(want, scale_factor=up, mode="nearest") if up > 1 else want
    want = (F.pad(want, (border,) * 4, mode="reflect") if border else want).permute(0, 2, 3, 1)
    assert (out.t.double() - want).abs().max().item() <= 1e-3 * max(1.0, want.abs().max().item())


# ================================================================================================ 3. Sampler noise
@pytest.mark.parametrize("B", [1, 5])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_randn(cuda, guarded, B, layout):
    """Several draws into consecutive slices of one buffer."""
    torch = cuda
    from future_urban_scene_generation_b200.noise import randn_cpu_exact
    shapes = [(B, 16, 5, 3), (B, 128, 2, 2), (B, 32, 1, 1)]
    sizes = [int(np.prod(s)) for s in shapes]
    buf = torch.full((sum(sizes),), float("nan"), device="cuda")
    outs, o = [], 0
    for s, n in zip(shapes, sizes):
        v = buf[o:o + n]
        outs.append(v.view(s if layout == "nchw" else (s[0], s[2], s[3], s[1])))
        o += n
    g = torch.Generator().manual_seed(40 + B)
    ref_g = torch.Generator()
    ref_g.set_state(g.get_state())
    with _case(f"randn B={B} {layout}"):
        randn_cpu_exact(shapes, layout=layout, generator=g, out=outs)
        torch.cuda.synchronize()
    for s, t in zip(shapes, outs):
        r = torch.randn(*s, generator=ref_g)
        t = t.cpu() if layout == "nchw" else t.cpu().permute(0, 3, 1, 2)
        assert torch.equal(t.contiguous().view(torch.int32), r.view(torch.int32)), s


# ================================================================================================ 3. warp stage
def _oracle_warp(batch, idx=None):
    from oracle import warp_oracle as O
    n = len(batch["src_kp"])
    outs = [O.warp_fused(batch["src"][i if idx is None else idx[i]], batch["src_kp"][i], batch["dst_kp"][i], batch["K"][i],
                         batch["E_src"][i], batch["E_dst"][i], batch["kp3d"][i]) for i in range(n)]
    return [np.stack([o[k] for o in outs]) for k in range(4)]


def _assert_warp(res, ref):
    warped, vis, pj, H12 = ref
    assert np.array_equal(res.vis.cpu().numpy(), vis)
    assert np.array_equal(res.plane_j.cpu().numpy(), pj)
    assert np.array_equal(res.H12.cpu().numpy().view(np.uint64), H12.view(np.uint64))
    assert np.array_equal(res.warped.cpu().numpy(), warped)


@pytest.mark.parametrize("B,hw", [(1, (100, 77)), (33, (100, 77)), (3, (300, 400))])
def test_warp_fused(cuda, guarded, B, hw):
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    h, w = hw
    b = synth.make_warp_batch(0, B, h, w)
    with _case(f"warp_fused B={B} {h}x{w}"):
        res = warp_batch(b["src"], b["src_kp"], b["dst_kp"], b["K"], b["E_src"], b["E_dst"], b["kp3d"])
        cuda.cuda.synchronize()
    _assert_warp(res, _oracle_warp(b))


def test_warp_fused_traj_and_idx(cuda, guarded):
    """B = 33 items sharing 5 source crops (src_index) with moved destination keypoints; the _traj form on the gathered crops."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    h, w, B = 100, 77, 33
    b = synth.make_warp_batch(200, B, h, w)
    idx = np.arange(B, dtype=np.int32) % 5
    src5 = b["src"][:5]
    kd = b["kp3d"][::-1].copy()
    args = (b["src_kp"], b["dst_kp"], b["K"], b["E_src"], b["E_dst"], b["kp3d"])
    with _case("warp_fused_idx B=33 n_src=5 moved"):
        r_idx = warp_batch(src5, *args, kp3d_dst=kd, src_index=torch.as_tensor(idx).cuda())
        torch.cuda.synchronize()
    with _case("warp_fused_traj B=33 moved"):
        r_traj = warp_batch(src5[idx], *args, kp3d_dst=kd)
        torch.cuda.synchronize()
    for f in ("vis", "plane_j"):
        assert torch.equal(getattr(r_idx, f), getattr(r_traj, f))
    assert torch.equal(r_idx.H12.view(torch.int64), r_traj.H12.view(torch.int64)) and torch.equal(r_idx.warped, r_traj.warped)
    with _case("warp_fused_idx B=33 n_src=5"):
        r0 = warp_batch(src5, *args, src_index=torch.as_tensor(idx).cuda())
        torch.cuda.synchronize()
    _assert_warp(r0, _oracle_warp(dict(b, src=src5), idx))


def test_warp_fused_large_batch_list_path(cuda, guarded):
    """1683 crops of 256^2 = 8415 (crop, plane) tasks: the list path; 51 copies of a 33-crop batch checked against the oracle."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    U, R = 33, 51
    b = synth.make_warp_batch(500, U)
    ref = _oracle_warp(b)
    dev = {k: torch.from_numpy(np.ascontiguousarray(np.concatenate([v] * R, 0))).cuda() for k, v in b.items()}
    with _case("warp_fused list path B=1683"):
        res = warp_batch(dev["src"], dev["src_kp"], dev["dst_kp"], dev["K"], dev["E_src"], dev["E_dst"], dev["kp3d"])
        torch.cuda.synchronize()
    want = torch.from_numpy(ref[0]).cuda()
    for r in range(R):
        sl = slice(r * U, (r + 1) * U)
        assert torch.equal(res.warped[sl], want), r
        assert np.array_equal(res.plane_j[sl].cpu().numpy(), ref[2]), r
    del dev


@pytest.mark.parametrize("B", [1, 7])
def test_warp_fused_window(cuda, guarded, B):
    """Whole 300x400 frames: every window byte equals the whole-frame warp cropped; the gaps between windows stay unwritten."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import icn_windows
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    H, W = 300, 400
    b = synth.make_warp_batch(300, B, H, W)
    kp = torch.as_tensor(b["dst_kp"]).long()
    x0 = kp[:, :, 0].min(1).values.clamp(0, W - 1); x1 = kp[:, :, 0].max(1).values.clamp(0, W - 1)
    y0 = kp[:, :, 1].min(1).values.clamp(0, H - 1); y1 = kp[:, :, 1].max(1).values.clamp(0, H - 1)
    ys, xs = torch.arange(H).view(1, H, 1), torch.arange(W).view(1, 1, W)
    masks = ((ys >= y0.view(-1, 1, 1)) & (ys <= y1.view(-1, 1, 1)) & (xs >= x0.view(-1, 1, 1)) & (xs <= x1.view(-1, 1, 1))).cuda()
    windows = icn_windows(masks, (H, W))
    args = (b["src_kp"], b["dst_kp"], b["K"], b["E_src"], b["E_dst"], b["kp3d"])
    with _case(f"warp_fused full frames B={B} 300x400"):
        full = warp_batch(b["src"], *args)
        torch.cuda.synchronize()
    with _case(f"warp_fused_window B={B} 300x400") as log:
        win = warp_batch(b["src"], *args, window=windows)
        torch.cuda.synchronize()
    _assert_warp(full, _oracle_warp(b))
    assert torch.equal(win.vis, full.vis) and torch.equal(win.plane_j, full.plane_j)
    assert not bool((win.plane_j == -2).any())
    end = 0
    written = np.zeros(windows.nbytes, bool)
    for i in range(B):
        wx, wy, ww, wh = (int(v) for v in windows.rect[i])
        o = int(windows.off[i])
        assert torch.equal(win.warped.item(i), full.warped[i, :, wy:wy + wh, wx:wx + ww]), i
        written[o:o + 5 * wh * ww * 3] = True
        end = max(end, o + 5 * wh * ww * 3)
    unw = _unwritten(log, "fusg_warp_fused_window", "warped windows").cpu().numpy()
    assert np.array_equal(unw, ~written[:end])


@pytest.mark.parametrize("N,hw", [(1, (101, 77)), (33, (101, 77))])
def test_visibility_planes_homography_perspective(cuda, guarded, N, hw):
    torch = cuda
    from future_urban_scene_generation_b200 import _lib, synth
    from oracle import warp_oracle as O
    h, w = hw
    st = _lib.stream_ptr(torch)
    b = synth.make_warp_batch(700, N, h, w)
    K, E, X = (torch.from_numpy(np.ascontiguousarray(b[k])).cuda() for k in ("K", "E_src", "kp3d"))
    vis = torch.empty(N, 7, dtype=torch.uint8, device="cuda")
    pts = torch.empty(N, 12, 2, dtype=torch.int32, device="cuda")
    areas = torch.empty(N, 7, 2, dtype=torch.int32, device="cuda")
    with _case(f"visibility N={N} {h}x{w}"):
        _lib.check(guarded.fusg_visibility(_lib.ptr(K), _lib.ptr(E), _lib.ptr(X), _lib.ptr(vis), _lib.ptr(pts), _lib.ptr(areas), N, h, w, st), "vis")
        torch.cuda.synchronize()
    for i in range(N):
        _, opts = O.compute_visibility(b["E_src"][i], b["K"][i], b["kp3d"][i], h, w, return_pts=True)
        ovis, oareas = O.visibility_from_pts(opts, O.plane_distances(b["E_src"][i], b["kp3d"][i]), h, w, return_areas=True)
        assert np.array_equal(pts[i].cpu().numpy(), opts) and np.array_equal(areas[i].cpu().numpy(), oareas)
        assert np.array_equal(vis[i].cpu().numpy(), ovis)
    img = torch.from_numpy(b["src"]).cuda()
    kp = torch.from_numpy(b["src_kp"]).cuda()
    planes = torch.empty(N, 5, h, w, 3, dtype=torch.uint8, device="cuda")
    with _case(f"get_planes N={N} {h}x{w}"):
        _lib.check(guarded.fusg_get_planes(_lib.ptr(img), _lib.ptr(kp), _lib.ptr(planes), N, h, w, st), "get_planes")
        torch.cuda.synchronize()
    for i in range(N):
        assert np.array_equal(planes[i].cpu().numpy(), O.get_planes(b["src"][i], b["src_kp"][i])), i
    tbl = O.plane_table(0)
    src = np.ascontiguousarray(b["src_kp"][:, tbl]).astype(np.int32)
    dst = np.ascontiguousarray(b["dst_kp"][:, tbl]).astype(np.int32)
    n = src.shape[1]
    Hm = torch.empty(N, 9, dtype=torch.float64, device="cuda")
    ok = torch.empty(N, dtype=torch.uint8, device="cuda")
    ts, tdst = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    with _case(f"find_homography N={N} n={n}"):
        _lib.check(guarded.fusg_find_homography(_lib.ptr(ts), _lib.ptr(tdst), n, _lib.ptr(Hm),
                                                _lib.ptr(ok), N, st), "find_homography")
        torch.cuda.synchronize()
    for i in range(N):
        Ho = O.find_homography(src[i], dst[i])
        assert (Ho is not None) == bool(ok[i])
        if Ho is not None:
            assert np.array_equal(Ho.ravel().view(np.uint64), Hm[i].cpu().numpy().view(np.uint64)) or np.isnan(Ho).any(), i
    Hw = torch.from_numpy(np.stack([np.eye(3) + np.array([[0.01 * i, 0.02, 3.5], [-0.01, 0.005 * i, -2.25], [1e-5 * i, 0, 0]]) for i in range(N)]).reshape(N, 9)).cuda()
    pw = torch.empty(N, h, w, 3, dtype=torch.uint8, device="cuda")
    with _case(f"warp_perspective N={N} {h}x{w}"):
        _lib.check(guarded.fusg_warp_perspective(_lib.ptr(img), _lib.ptr(Hw), _lib.ptr(pw), N, h, w, st), "warp_perspective")
        torch.cuda.synchronize()
    for i in range(N):
        assert np.array_equal(pw[i].cpu().numpy(), O.warp_perspective(b["src"][i], Hw[i].cpu().numpy().reshape(3, 3))), i


def test_step_keypoints(cuda, guarded):
    """N = 33 items of 5 vehicles (not a multiple of the block)."""
    from future_urban_scene_generation_b200 import kinematics as KM, synth
    from oracle import kinematics_oracle as KO
    H, W, V, N = 720, 1280, 5, 33
    cases = [synth.make_trajectory_case(v, steps=8, h=H, w=W) for v in range(V)]
    poses = [KM.trajectory_poses(c["meter_coords"]) for c in cases]
    veh = (np.arange(N) % V).astype(np.int32)
    step = np.arange(N) // V
    rot = np.stack([poses[veh[n]][2][step[n]] for n in range(N)])
    tr = np.stack([poses[veh[n]][1][step[n]] for n in range(N)])
    kp3d = np.stack([c["kp3d"] for c in cases])
    R, t, K = (np.stack([c[k] for c in cases]) for k in ("R", "t", "K"))
    with _case("step_keypoints N=33"):
        m, k2, vv = KM.step_keypoints_batch(kp3d, veh, rot, tr, R, t, K, H, W)
        cuda.cuda.synchronize()
    m, k2, vv = m.cpu().numpy(), k2.cpu().numpy(), vv.cpu().numpy()
    for n in range(N):
        o_m, o_2, o_v = KO.step(kp3d[veh[n]], rot[n], tr[n], R[veh[n]], t[veh[n]], K[veh[n]], H, W)
        assert np.array_equal(m[n], o_m) and np.array_equal(k2[n], o_2) and np.array_equal(vv[n], o_v), n


# ================================================================================================ 3. frame operations
def test_resize_ragged_with_gaps(cuda, guarded):
    """A ragged batch packed with 16-byte-aligned gaps through dst_off: each item writes exactly its own rectangle."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    from oracle import frame_oracle as FO
    rng = np.random.default_rng(11)
    srcs = [rng.integers(0, 256, (int(rng.integers(5, 90)), int(rng.integers(5, 90)), 3), dtype=np.uint8) for _ in range(9)]
    dsz = [(int(rng.integers(1, 70)), int(rng.integers(1, 70))) for _ in range(9)]          # (w, h) like cv2
    so, do, s, o = [], [], 0, 0
    for im, (dw, dh) in zip(srcs, dsz):
        so.append(s); s += im.size
        do.append(o); o = _round(o + dw * dh * 3 + 1, 16)
    src = torch.from_numpy(np.concatenate([im.reshape(-1) for im in srcs])).cuda()
    dst = torch.zeros(o, dtype=torch.uint8, device="cuda")
    t_so, t_do = torch.tensor(so, dtype=torch.int64, device="cuda"), torch.tensor(do, dtype=torch.int64, device="cuda")
    src_hw = torch.tensor([im.shape[:2] for im in srcs], dtype=torch.int32, device="cuda")
    dst_hw = torch.tensor([(h, w) for w, h in dsz], dtype=torch.int32, device="cuda")
    with _case("resize ragged B=9") as log:
        _lib.check(guarded.fusg_resize_u8(_lib.ptr(src), _lib.ptr(t_so), _lib.ptr(src_hw), _lib.ptr(dst), _lib.ptr(t_do), _lib.ptr(dst_hw), 9,
                                          max(w * h for w, h in dsz), _lib.stream_ptr(torch)), "resize")
        torch.cuda.synchronize()
    d = dst.cpu().numpy()
    mask = np.ones(do[-1] + dsz[-1][0] * dsz[-1][1] * 3, bool)
    for im, (dw, dh), off in zip(srcs, dsz, do):
        assert np.array_equal(d[off:off + dw * dh * 3].reshape(dh, dw, 3), FO.resize_linear_u8(im, (dw, dh)))
        mask[off:off + dw * dh * 3] = False
    assert np.array_equal(_unwritten(log, "fusg_resize_u8").cpu().numpy(), mask)


def test_paste_back_frames_no_item_names(cuda, guarded):
    """Four frames, items on frames 0 and 2 only: pixels outside the masks and frames 1 and 3 keep the canary of each run."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import paste_back_batch
    from oracle import frame_oracle as FO
    Hf, Wf = 90, 130
    items = [synth.make_paste_case(i, (Hf, Wf)) for i in range(5)]
    fidx = [0, 2, 0, 2, 2]
    infos = [FO.square_crop_info((Hf, Wf), bb) for bb, _, _ in items]
    frames = torch.zeros(4, Hf, Wf, 3, dtype=torch.uint8, device="cuda")
    with _case("paste_back F=4 B=5") as log:
        paste_back_batch(frames, np.stack([n for _, _, n in items]), [m for _, m, _ in items], infos, fidx)
        torch.cuda.synchronize()
    runs = [e for e in log if e["name"] == "fusg_paste_back"][-1]["runs"]
    for c, r in zip(CANARIES, runs):
        ref = np.full((4, Hf, Wf, 3), c, np.uint8)
        for (bb, m, net), info, f in zip(items, infos, fidx):
            FO.paste_back(ref[f], net, info, m)
        assert np.array_equal(r.cpu().numpy().reshape(4, Hf, Wf, 3), ref), hex(c)
    assert any(m.any() for _, m, _ in items)


@pytest.mark.parametrize("B", [1, 3])
def test_pack_vunet_inputs_and_mask_bbox(cuda, guarded, B):
    torch = cuda
    from future_urban_scene_generation_b200 import _lib, synth
    from future_urban_scene_generation_b200.frame_ops import pack_vunet_inputs_batch
    from oracle import frame_oracle as FO
    Hf, Wf = 72, 97
    frames = np.random.default_rng(B).integers(0, 256, (2, Hf, Wf, 3), dtype=np.uint8)
    cases = [synth.make_pack_case(i, (Hf, Wf)) for i in range(B)]
    fidx = [i % 2 for i in range(B)]
    with _case(f"pack_vunet_inputs B={B}"):
        x, y, bbox = pack_vunet_inputs_batch(frames, fidx, [c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases])
        torch.cuda.synchronize()
    for b in range(B):
        rx, ry, _ = FO.pack_vunet_inputs(frames[fidx[b]], *cases[b])
        assert np.array_equal(x[b].cpu().numpy(), rx.reshape(x[b].shape)) and np.array_equal(y[b].cpu().numpy(), ry.reshape(y[b].shape)), b
    # fusg_mask_bbox with an empty mask among odd-sized ones
    ms = [np.zeros((5, 7), np.uint8), (np.random.default_rng(3).random((9, 11)) > 0.7).astype(np.uint8), np.zeros((3, 3), np.uint8)]
    ms[2][1, 2] = 1
    off = np.cumsum([0] + [m.size for m in ms[:-1]])
    rect = np.array([[4, 6, 7, 5], [0, 1, 11, 9], [20, 30, 3, 3]], np.int32)
    bb = torch.empty(3, 4, dtype=torch.int32, device="cuda")
    t_m = torch.from_numpy(np.concatenate([m.ravel() for m in ms])).cuda()
    t_off, t_rect = torch.from_numpy(off.astype(np.int64)).cuda(), torch.from_numpy(rect).cuda()
    with _case("mask_bbox B=3 with an empty mask"):
        _lib.check(guarded.fusg_mask_bbox(_lib.ptr(t_m), _lib.ptr(t_off), _lib.ptr(t_rect), _lib.ptr(bb), 3, 99, _lib.stream_ptr(torch)), "mask_bbox")
        torch.cuda.synchronize()
    want = [[2 ** 31 - 1, 2 ** 31 - 1, -1, -1]]
    for m, (rx0, ry0, _, _) in zip(ms[1:], rect[1:]):
        yy, xx = np.nonzero(m)
        want.append([rx0 + xx.min(), ry0 + yy.min(), rx0 + xx.max(), ry0 + yy.max()])
    assert bb.cpu().numpy().tolist() == want


@pytest.mark.parametrize("B", [1, 3])
def test_pack_icn_inputs_whole_and_window(cuda, guarded, B):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import get_icn_inputs_batch, icn_windows
    from future_urban_scene_generation_b200.frame_ops import WindowedPlanes
    from oracle import frame_oracle as FO
    Hf, Wf = 90, 130
    cs = [synth.make_icn_pack_case(i, (Hf, Wf)) for i in range(B)]
    planes = np.stack([c[0] for c in cs]); normals = np.stack([c[1] for c in cs])
    masks = np.stack([c[2] for c in cs]); central = np.stack([c[3] for c in cs])
    with _case(f"pack_icn_inputs B={B}"):
        out, _ = get_icn_inputs_batch(planes, normals, masks, central)
        torch.cuda.synchronize()
    for b in range(B):
        ref, _ = FO.get_icn_inputs(planes[b], normals[b], masks[b], central[b])
        assert np.array_equal(out[b].cpu().numpy(), ref), b
    windows = icn_windows(masks, (Hf, Wf))
    data = torch.zeros(windows.nbytes, dtype=torch.uint8, device="cuda")
    for b in range(B):
        x0, y0, w, h = (int(v) for v in windows.rect[b])
        o = int(windows.off[b])
        data[o:o + 5 * h * w * 3] = torch.from_numpy(np.ascontiguousarray(planes[b, :, y0:y0 + h, x0:x0 + w])).cuda().reshape(-1)
    with _case(f"pack_icn_inputs_window B={B}"):
        outw, _ = get_icn_inputs_batch(WindowedPlanes(data, windows), normals, masks, central)
        torch.cuda.synchronize()
    assert torch.equal(outw, out)


@pytest.mark.parametrize("B", [1, 3])
def test_u8_to_vunet(cuda, guarded, B):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import u8_to_vunet_inputs, u8_to_vunet_y
    res = 40
    m, ns, nd = (torch.from_numpy(a).cuda() for a in synth.make_vunet_inputs_u8(3, B, res))
    rx, ry = synth.make_vunet_inputs(3, B, res)
    with _case(f"u8_to_vunet_inputs B={B} res {res}"):
        x, y = u8_to_vunet_inputs(m, ns, nd)
        torch.cuda.synchronize()
    with _case(f"u8_to_vunet_y B={B} res {res}"):
        y2 = u8_to_vunet_y(nd)
        torch.cuda.synchronize()
    assert np.array_equal(x.cpu().numpy(), rx) and np.array_equal(y.cpu().numpy(), ry) and torch.equal(y, y2)


def test_gather_rows(cuda, guarded):
    """Three segments, one of an odd number (3) of 16-byte vectors per row; B = 33 with indices out of range."""
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import gather_rows
    g = torch.Generator().manual_seed(2)
    srcs = [torch.randint(0, 255, (5, 48), generator=g, dtype=torch.uint8).cuda(), torch.randn(5, 7, 4, generator=g).cuda(),
            torch.randn(5, 3, 8, generator=g).to(torch.bfloat16).cuda()]
    index = torch.tensor([(i * 3) % 7 - 1 for i in range(33)], dtype=torch.int32, device="cuda")
    dsts = [torch.full((33,) + tuple(s.shape[1:]), 7, dtype=s.dtype, device="cuda") for s in srcs]
    with _case("gather_rows B=33 3 segments"):
        gather_rows(list(zip(srcs, dsts)), index)
        torch.cuda.synchronize()
    ok = (index >= 0) & (index < 5)
    for s, d in zip(srcs, dsts):
        want = torch.zeros_like(d)
        want[ok] = s[index[ok].long()]
        assert torch.equal(d, want)


# ================================================================================================ 3. renderer
@pytest.mark.parametrize("hw", [(37, 53), (1080, 1920)])
def test_render_normals_into_a_slice(cuda, guarded, hw):
    """out= the items [1, 4) of a batch of 5: the neighbouring items are untouched; item 2 is moved entirely out of frame."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.warp_learn.render import render_normals_batch
    from oracle import render_oracle as RO
    h, w = hw
    V, T = synth.make_car_mesh(1)
    cams = [synth.make_pose_pair(60 + i, h, w) for i in range(3)]
    E, K = np.stack([c["E_src"] for c in cams]), np.stack([c["K"] for c in cams])
    rot = np.stack([np.eye(3)] * 3)
    tr = np.array([[0, 0, 0], [1e4, 0, 0], [0, 0, 0]], np.float64)
    normals = torch.full((5, h, w, 3), 0x77, dtype=torch.uint8, device="cuda")
    mask = torch.full((5, h, w), 0x77, dtype=torch.uint8, device="cuda")
    with _case(f"render_normals out=[1:4] {h}x{w}"):
        render_normals_batch((V, T), E, K, h, w, rot=rot, tr=tr, out=(normals[1:4], mask[1:4]))
        torch.cuda.synchronize()
    for b in (0, 4):
        assert bool((normals[b] == 0x77).all()) and bool((mask[b] == 0x77).all())
    assert bool((mask[2] == 1).all()) and not bool(normals[2].any())          # out of frame: all background
    for i in (0, 2):
        if h * w <= 1 << 16:
            ref_img, ref_mask = RO.render_normals(V, T, E[i], K[i], h, w, rot=rot[i], tr=tr[i])
            assert np.array_equal(normals[1 + i].cpu().numpy(), ref_img) and np.array_equal(mask[1 + i].cpu().numpy(), ref_mask), i
        else:                                       # (the software rasteriser is slow at 1080p: its background rule only)
            assert torch.equal(mask[1 + i].bool(), (normals[1 + i] == 0).all(-1))
            assert 0 < int((mask[1 + i] == 0).sum()) < h * w


# ================================================================================================ 4. coverage
def test_every_writing_entry_point_has_a_case():
    """Runs last: every function of include/fusg.h that writes device memory was called by a case above."""
    text = open(os.path.join(ROOT, "include", "fusg.h")).read()
    names = set(re.findall(r"^\s*(?:int|size_t|void|const char \*)\s*\**\s*(fusg_\w+)\s*\(", text, re.M))
    writing = {n for n in names if n not in HOST_ONLY and not n.startswith("fusg_sizeof_") and not n.endswith("_workspace_bytes")
               and not n.endswith("_workspace_bytes_hw")}
    assert len(names) > 30 and "fusg_conv2d" in writing
    assert not writing - set(SPECS), f"entry points without a write-extent spec: {sorted(writing - set(SPECS))}"
    missing = sorted(n for n in writing if not STATS.get(n, {}).get("cases"))
    assert not missing, f"entry points that write device memory but no case here called: {missing}"
