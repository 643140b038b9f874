"""fusg_crop_geometry / frame_ops.crop_geometry: the crop geometry of the sketch masks computed on the device, against the Python
geometry it replaces (square_crop_info, pack_crop_info, icn_window_rect, window_layout) bit for bit; its refusals (statuses) and what
every consumer does with a refused item; and the frame-level chain masks -> geometry -> windowed warp -> get_icn_inputs -> ICN ->
y_tilde packing -> paste-back, run with the host geometry, with the device geometry eagerly (no synchronisation) and replayed from
one captured CUDA graph on a second set of inputs -- all bit-identical."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_crop_geometry_cpu import random_boxes, reference_geometry

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = 0xA5
BIG = 1 << 60


def _kernel(torch, bbox, hw, frame_index=None, cap=0, rows=0):
    """fusg_crop_geometry on a host bbox array -> numpy (info, win, win_off, status)."""
    from future_urban_scene_generation_b200 import _lib
    B = len(bbox)
    bb = torch.as_tensor(np.ascontiguousarray(bbox, np.int32)).cuda()
    fi = None if frame_index is None else torch.as_tensor(np.asarray(frame_index, np.int32)).cuda()
    info = torch.full((B, 9), -7, dtype=torch.int32, device="cuda")
    win = torch.full((B, 4), -7, dtype=torch.int32, device="cuda")
    off = torch.full((B,), -7, dtype=torch.int64, device="cuda")
    st = torch.full((B,), -7, dtype=torch.int8, device="cuda")
    _lib.check(_lib.lib().fusg_crop_geometry(_lib.ptr(bb), _lib.ptr(fi), B, hw[0], hw[1], cap, rows, _lib.ptr(info), _lib.ptr(win), _lib.ptr(off),
                                             _lib.ptr(st), _lib.stream_ptr(torch)), "fusg_crop_geometry")
    return info.cpu().numpy(), win.cpu().numpy(), off.cpu().numpy(), st.cpu().numpy()


def _assert_geometry(torch, bbox, hw, frame_index):
    info, win, off, st = _kernel(torch, bbox, hw, frame_index, BIG, hw[0])
    r_info, r_win, r_off, _ = reference_geometry(bbox, hw, frame_index)
    assert not st.any()
    for name, got, want in (("info", info, r_info), ("win", win, r_win), ("win_off", off, r_off)):
        bad = np.nonzero((got != want).reshape(len(bbox), -1).any(1))[0]
        assert bad.size == 0, f"{name} differs for {bad.size} boxes, first {bbox[bad[0]]}: {got[bad[0]]} != {want[bad[0]]}"


# ---------------------------------------------------------------------------------------------------- 1. the kernel, bit for bit
def test_every_box_of_a_40x56_frame(cuda):
    H, W = 40, 56
    xs = np.array([(a, b) for a in range(W) for b in range(a, W)], np.int32)
    ys = np.array([(a, b) for a in range(H) for b in range(a, H)], np.int32)
    bb = np.empty((len(xs) * len(ys), 4), np.int32)
    bb[:, 0], bb[:, 2] = np.repeat(xs[:, 0], len(ys)), np.repeat(xs[:, 1], len(ys))
    bb[:, 1], bb[:, 3] = np.tile(ys[:, 0], len(xs)), np.tile(ys[:, 1], len(xs))
    assert len(bb) > 1_300_000
    _assert_geometry(cuda, bb, (H, W), None)
    _assert_geometry(cuda, bb[::97], (H, W), np.arange(len(bb[::97])) % 20)


@pytest.mark.parametrize("hw", [(256, 256), (300, 400), (720, 1280), (1080, 1920)])
def test_random_boxes(cuda, hw):
    bb = random_boxes(np.random.default_rng(hw[0] * 7 + hw[1]), 200_000, hw)
    assert ((bb[:, 0] == bb[:, 2]) & (bb[:, 1] == bb[:, 3])).any()                       # 1-px masks
    assert (bb[:, 0] == 0).any() and (bb[:, 1] == 0).any() and (bb[:, 2] == hw[1] - 1).any() and (bb[:, 3] == hw[0] - 1).any()
    _assert_geometry(cuda, bb, hw, None)
    _assert_geometry(cuda, bb, hw, np.random.default_rng(5).integers(0, 600, len(bb)))


def test_write_extent(cuda):
    """fusg_crop_geometry writes all of its outputs and nothing outside them (the harness of test_write_extent_gpu.py, whose coverage
    check this entry point joins here)."""
    import test_write_extent_gpu as WE
    from future_urban_scene_generation_b200 import _lib
    torch = cuda
    nb = lambda a: WE._v(a[2])
    WE.SPECS["fusg_crop_geometry"] = lambda t, L, a: [WE._arg(a, 7, nb(a) * 36, "info"), WE._arg(a, 8, nb(a) * 16, "win"),
                                                      WE._arg(a, 9, nb(a) * 8, "win_off"), WE._arg(a, 10, nb(a), "status")]
    L = _lib.lib()
    orig = L.fusg_crop_geometry
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(L, "fusg_crop_geometry", lambda *args: WE._guarded_call(torch, L, "fusg_crop_geometry", orig, args))
        for B, cap in ((1, 0), (1037, 0), (1037, 200_000), (3000, BIG)):
            bb = random_boxes(np.random.default_rng(B), B, (300, 400))
            bb[::50] = (0x7fffffff, 0x7fffffff, -1, -1)                                # empty masks among them
            with WE._case(f"crop_geometry B={B} capacity={cap}"):
                _kernel(torch, bb, (300, 400), None, cap, 300 if cap else 0)
            with WE._case(f"crop_geometry B={B} capacity={cap}, called without windows"):
                t = torch.as_tensor(bb).cuda()
                info = torch.empty((B, 9), dtype=torch.int32, device="cuda")
                st = torch.empty((B,), dtype=torch.int8, device="cuda")
                _lib.check(L.fusg_crop_geometry(_lib.ptr(t), None, B, 300, 400, 0, 0, _lib.ptr(info), None, None, _lib.ptr(st),
                                                _lib.stream_ptr(torch)), "fusg_crop_geometry")
                torch.cuda.synchronize()
                assert np.array_equal(st.cpu().numpy(), np.where(bb[:, 2] < 0, 1, 0))
    assert len(WE.STATS["fusg_crop_geometry"]["cases"]) == 8


# ---------------------------------------------------------------------------------------------------- 2. statuses and refused items
def _items(torch, H, W, V=4, S=4, seed=0, ellipse_max=(600, 400)):
    """Trajectory items as scripts/bench_clip.py builds them: kinematics keypoints, an ellipse silhouette in the keypoints' bounding
    box, normal sketches inside it, random central crops; all on the device."""
    from future_urban_scene_generation_b200 import kinematics, synth
    dev = torch.device("cuda")
    N = V * S
    cases = []
    for v in range(V):
        c = synth.make_trajectory_case(seed + v, steps=S, h=H, w=W)
        f = 1650.0 * W / 1920.0
        c["K"] = np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]])
        cases.append(c)
    kp3d = np.stack([c["kp3d"] for c in cases])
    R, t, K = np.stack([c["R"] for c in cases]), np.stack([c["t"] for c in cases]), np.stack([c["K"] for c in cases])
    E = np.concatenate([R, t[:, :, None]], 2)
    src_kp = np.int32((np.stack([synth.project(K[v], np.vstack([E[v], [0, 0, 0, 1]]), kp3d[v]) for v in range(V)]) / [W, H]) * [W, H])
    poses = [kinematics.trajectory_poses(c["meter_coords"]) for c in cases]
    veh = np.repeat(np.arange(V), S).astype(np.int32)
    moved, _, dst_kp = kinematics.step_keypoints_batch(kp3d, veh, np.concatenate([p[2] for p in poses]), np.concatenate([p[1] for p in poses]),
                                                       R, t, K, H, W)
    vi = torch.as_tensor(veh, device=dev).long()
    kp = dst_kp.float()
    yy, xx = torch.arange(H, device=dev, dtype=torch.float32).view(1, H, 1), torch.arange(W, device=dev, dtype=torch.float32).view(1, 1, W)
    x0, x1, y0, y1 = kp[:, :, 0].min(1).values, kp[:, :, 0].max(1).values, kp[:, :, 1].min(1).values, kp[:, :, 1].max(1).values
    cx, cy = ((x0 + x1) / 2).clamp(20, W - 20).view(-1, 1, 1), ((y0 + y1) / 2).clamp(20, H - 20).view(-1, 1, 1)
    rx = ((x1 - x0) / 2 + 6).clamp(8, ellipse_max[0] * W / 1920).view(-1, 1, 1)
    ry = ((y1 - y0) / 2 + 6).clamp(8, ellipse_max[1] * H / 1080).view(-1, 1, 1)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    masks = ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0
    return dict(
        N=N, V=V, S=S, hw=(H, W),
        frames=torch.randint(0, 256, (V, H, W, 3), generator=g, device=dev, dtype=torch.uint8),
        src_kp=torch.as_tensor(src_kp, device=dev)[vi].contiguous(), dst_kp=dst_kp.to(torch.int32).contiguous(),
        K=torch.as_tensor(K, device=dev)[vi].contiguous(), E=torch.as_tensor(E, device=dev)[vi].contiguous(),
        kp3d=torch.as_tensor(kp3d, device=dev)[vi].contiguous(), moved=moved.contiguous(), idx=torch.as_tensor(veh, device=dev),
        masks=masks, normals=torch.randint(1, 256, (N, H, W, 3), generator=g, device=dev, dtype=torch.uint8) * masks.unsqueeze(-1).to(torch.uint8),
        central=torch.randint(0, 256, (N, 256, 256, 3), generator=g, device=dev, dtype=torch.uint8),
        step=torch.as_tensor(np.tile(np.arange(S), V).astype(np.int32), device=dev),
        background=torch.randint(0, 256, (S, H, W, 3), generator=g, device=dev, dtype=torch.uint8))


def _warp(sc, window, out=None):
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    return warp_batch(sc["frames"], sc["src_kp"], sc["dst_kp"], sc["K"], sc["E"], sc["E"], sc["kp3d"], kp3d_dst=sc["moved"], src_index=sc["idx"],
                      window=window, out=out)


def _expected(rect, empty, cap, rows):
    """(status, block ends) the window layout of `rect` gives: empty items take no bytes, a block ending past cap refuses its item."""
    blocks = (5 * rect[:, 2].astype(np.int64) * rect[:, 3] * 3 + 15) & ~15
    blocks[empty] = 0
    ends = np.cumsum(blocks)
    st = np.where((ends > cap) | (rect[:, 3] > rows), 2, 0).astype(np.int8)
    st[empty] = 1
    first = int(np.argmax(ends > cap)) if (ends > cap).any() else len(st)
    assert (st[first:] != 0).all()                                             # the first overflowing item and every later one
    return st, ends


def test_statuses_and_refused_items(cuda):
    """Empty mask -> 1; the first block past the capacity and every later item -> 2; a window taller than max_win_h -> 2.  For each
    refused item the windowed warp leaves its sentinel bytes alone, its gen_in and y_tilde rows are zero, the composited frames keep
    their pixels inside its mask, and check() raises."""
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import (PastePlan, WindowedPlanes, crop_geometry, get_icn_inputs_batch, icn_windows,
                                                             pack_vunet_inputs_batch, paste_back_packed)
    from future_urban_scene_generation_b200.warp_learn import RefusedCrops
    from future_urban_scene_generation_b200.warp_learn.batch import WarpResult
    H, W = 300, 400
    sc = _items(torch, H, W, V=3, S=4)
    N = sc["N"]
    ref = icn_windows(sc["masks"], (H, W))
    full = crop_geometry(sc["masks"], (H, W), frame_index=sc["step"], window_capacity=(ref.nbytes, ref.max_h))
    assert not full.status.any() and torch.equal(full.win.cpu(), torch.from_numpy(ref.rect)) and np.array_equal(full.off, ref.off)
    assert full.crop_infos() == ref.crop_infos
    masks = sc["masks"].clone()
    masks[2] = False                                                           # item 2: empty
    hs = ref.rect[:, 3]
    tall = max((b for b in range(N) if b != 2), key=lambda b: hs[b])
    rows = int(hs[tall]) - 1
    cut = int(_expected(ref.rect, [2], BIG, N)[1][N - 5])                      # items N-4.. end past the capacity
    want, _ = _expected(ref.rect, [2], cut, rows)
    g = crop_geometry(masks, (H, W), frame_index=sc["step"], window_capacity=(cut, rows))
    st = g.status.cpu().numpy()
    assert np.array_equal(st, want), (st, want)
    assert want[tall] == 2 and (want[N - 4:] == 2).all() and want[2] == 1
    refused = np.nonzero(want)[0].tolist()
    assert (g.win.cpu().numpy()[refused] == 0).all()
    # the windowed warp: refused items are not written at all
    data = torch.full((cut + 4096,), SENTINEL, dtype=torch.uint8, device="cuda")
    out = WarpResult(warped=WindowedPlanes(data, g), vis=torch.empty((N, 2, 7), dtype=torch.uint8, device="cuda"),
                     plane_j=torch.empty((N, 5), dtype=torch.int8, device="cuda"), H12=torch.empty((N, 5, 3, 3), dtype=torch.float64, device="cuda"))
    res = _warp(sc, g, out)
    torch.cuda.synchronize()
    written = np.zeros(data.numel(), bool)
    g_rect, g_off = g.rect, g.off                                              # item 2 takes no bytes: the later offsets move down
    for b in range(N):
        if st[b] == 0:
            assert np.array_equal(g_rect[b], ref.rect[b]), b
            x0, y0, w, h = (int(v) for v in g_rect[b])
            written[int(g_off[b]):int(g_off[b]) + 5 * w * h * 3] = True
    assert bool((data[torch.from_numpy(~written).cuda()] == SENTINEL).all())
    assert (res.plane_j.cpu().numpy()[refused] == -2).all()
    # ICN and VUNet inputs: zero rows for refused items, the host form's rows for the others
    gen_in, same = get_icn_inputs_batch(res.warped, sc["normals"], None, sc["central"], geometry=g)
    assert same is g
    ok = [b for b in range(N) if st[b] == 0]
    host_full = _warp(sc, ref)
    gen_ref, _ = get_icn_inputs_batch(host_full.warped, sc["normals"], sc["masks"], sc["central"])
    x, y, _ = pack_vunet_inputs_batch(sc["frames"], sc["idx"], ~masks, sc["normals"], sc["normals"], geometry=g)
    x_ref, y_ref, _ = pack_vunet_inputs_batch(sc["frames"], sc["idx"].tolist(), ~sc["masks"], sc["normals"], sc["normals"])
    torch.cuda.synchronize()
    assert not gen_in[refused].any() and not x[refused].any() and not y[refused].any()
    assert torch.equal(gen_in[ok], gen_ref[ok]) and torch.equal(x[ok], x_ref[ok]) and torch.equal(y[ok], y_ref[ok])
    # paste: a refused item leaves its frame pixels alone
    crops = torch.randint(0, 256, (N, 256, 256, 3), dtype=torch.uint8, device="cuda")
    frames = sc["background"].clone()
    paste_back_packed(frames, crops, PastePlan.from_geometry(g, masks))
    torch.cuda.synchronize()
    fr, step = frames.cpu().numpy(), sc["step"].cpu().numpy()
    bg, mk = sc["background"].cpu().numpy(), masks.cpu().numpy()
    for b in refused:
        cover = np.zeros((H, W), bool)
        for o in ok:
            if step[o] == step[b]:
                cover |= mk[o]
        only = mk[b] & ~cover
        assert np.array_equal(fr[step[b]][only], bg[step[b]][only]), b
    assert not np.array_equal(fr, bg)
    with pytest.raises(ValueError, match="empty sketch mask"):
        g.check()
    g2 = crop_geometry(sc["masks"], (H, W), window_capacity=(cut, rows))
    want2, _ = _expected(ref.rect, [], cut, rows)
    with pytest.raises(RefusedCrops) as ei:
        g2.check()
    assert ei.value.indices == np.nonzero(want2)[0].tolist()
    assert crop_geometry(sc["masks"], (H, W), window_capacity=(ref.nbytes, ref.max_h)).check().status.shape == (N,)


def test_frame_indices_outside_the_frames_are_refused_on_the_device(cuda):
    """Frame indices are device data nobody range-checks on the host: a source index outside [0, F) gives zero x / y rows, a paste
    index outside [0, F) pastes nothing; every other item is what it is with valid indices."""
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import PastePlan, crop_geometry, pack_vunet_inputs_batch, paste_back_packed
    H, W = 300, 400
    sc = _items(torch, H, W, V=3, S=4, seed=3)
    N, V, S = sc["N"], sc["V"], sc["S"]
    bad = [1, 6, 10]
    src = sc["idx"].clone()
    src[bad] = torch.tensor([V, -1, V + 100], dtype=torch.int32, device="cuda")
    step = sc["step"].clone()
    step[bad] = torch.tensor([S, -2, S + 100], dtype=torch.int32, device="cuda")
    g_ok = crop_geometry(sc["masks"], (H, W), frame_index=sc["step"])
    g_bad = crop_geometry(sc["masks"], (H, W), frame_index=step)
    x, y, _ = pack_vunet_inputs_batch(sc["frames"], src, ~sc["masks"], sc["normals"], sc["normals"], geometry=g_bad)
    x_ref, y_ref, _ = pack_vunet_inputs_batch(sc["frames"], sc["idx"], ~sc["masks"], sc["normals"], sc["normals"], geometry=g_ok)
    crops = torch.randint(0, 256, (N, 256, 256, 3), dtype=torch.uint8, device="cuda")
    keep = torch.ones(N, dtype=torch.bool, device="cuda")
    keep[bad] = False
    f_bad = paste_back_packed(sc["background"].clone(), crops, PastePlan.from_geometry(g_bad, sc["masks"]))
    f_ref = paste_back_packed(sc["background"].clone(), crops, PastePlan.from_geometry(g_ok, sc["masks"] & keep.view(N, 1, 1)))
    torch.cuda.synchronize()
    good = [b for b in range(N) if b not in bad]
    assert not x[bad].any() and not y[bad].any()
    assert torch.equal(x[good], x_ref[good]) and torch.equal(y[good], y_ref[good])
    assert torch.equal(f_bad, f_ref) and not torch.equal(f_bad, sc["background"])


# ---------------------------------------------------------------------------------------------------- 3. the chain, three ways
def _icn_model(torch):
    from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
    torch.manual_seed(0)
    return G_Resnet(21).cuda().eval()


def _host_chain(torch, sc, icn, chunk=100):
    from future_urban_scene_generation_b200.frame_ops import get_icn_inputs_batch, icn_windows, pack_vunet_inputs_batch, paste_back_batch
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch
    windows = icn_windows(sc["masks"], sc["hw"])
    res = _warp(sc, windows)
    gen_in, infos = get_icn_inputs_batch(res.warped, sc["normals"], sc["masks"], sc["central"])
    icn_out = torch.cat([icn(gen_in[i:i + chunk]) for i in range(0, sc["N"], chunk)])
    icn_img = to_image_batch(icn_out, from_LAB=True)
    _, y, _ = pack_vunet_inputs_batch(sc["frames"], sc["idx"].tolist(), ~sc["masks"], sc["normals"], sc["normals"])
    step = sc["step"].tolist()
    f_icn = paste_back_batch(sc["background"].clone(), icn_img, sc["masks"], infos, step)
    f_vun = paste_back_batch(sc["background"].clone(), to_image_batch(y), sc["masks"], infos, step)
    return dict(windows=windows, res=res, gen_in=gen_in, icn_out=icn_out, y=y, f_icn=f_icn, f_vun=f_vun)


def _device_chain(torch, sc, icn, cap, chunk=100):
    from future_urban_scene_generation_b200.frame_ops import (PastePlan, crop_geometry, get_icn_inputs_batch, pack_vunet_inputs_batch,
                                                             paste_back_packed)
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch
    g = crop_geometry(sc["masks"], sc["hw"], frame_index=sc["step"], window_capacity=cap)
    res = _warp(sc, g)
    gen_in, _ = get_icn_inputs_batch(res.warped, sc["normals"], None, sc["central"], geometry=g)
    icn_out = torch.cat([icn(gen_in[i:i + chunk]) for i in range(0, sc["N"], chunk)])
    icn_img = to_image_batch(icn_out, from_LAB=True)
    _, y, _ = pack_vunet_inputs_batch(sc["frames"], sc["idx"], ~sc["masks"], sc["normals"], sc["normals"], geometry=g)
    plan = PastePlan.from_geometry(g, sc["masks"])
    f_icn = paste_back_packed(sc["background"].clone(), icn_img, plan)
    f_vun = paste_back_packed(sc["background"].clone(), to_image_batch(y), plan)
    return dict(g=g, res=res, gen_in=gen_in, icn_out=icn_out, y=y, f_icn=f_icn, f_vun=f_vun)


def _assert_chains_equal(torch, host, dev):
    w = host["windows"]
    assert not dev["g"].status.any()
    assert torch.equal(dev["g"].win.cpu(), torch.from_numpy(w.rect)) and np.array_equal(dev["g"].off, w.off)
    hr, dr = host["res"], dev["res"]
    assert torch.equal(hr.vis, dr.vis) and torch.equal(hr.plane_j, dr.plane_j)
    assert torch.equal(hr.H12.view(torch.int64), dr.H12.view(torch.int64))
    written = np.zeros(w.nbytes, bool)
    for b in range(len(w)):
        x0, y0, ww, wh = (int(v) for v in w.rect[b])
        written[int(w.off[b]):int(w.off[b]) + 5 * ww * wh * 3] = True
    wm = torch.from_numpy(written).cuda()
    assert torch.equal(hr.warped.data[:w.nbytes][wm], dr.warped.data[:w.nbytes][wm])
    for k in ("gen_in", "icn_out", "y"):
        assert torch.equal(host[k].view(torch.int32), dev[k].view(torch.int32)), k
    for k in ("f_icn", "f_vun"):
        assert torch.equal(host[k], dev[k]), k


def _copy_inputs(dst, src):
    for k, v in src.items():
        if hasattr(v, "copy_") and k != "hw":
            dst[k].copy_(v)


@pytest.mark.parametrize("hw", [(720, 1280), (1080, 1920)])
def test_chain_host_eager_and_graph(cuda, hw):
    """600 items (30 vehicles x 20 steps): host geometry vs device geometry (eager, under sync debug mode "error") vs one captured graph
    of the device chain replayed on a second set of masks, keypoints and normals."""
    torch = cuda
    H, W = hw
    icn = _icn_model(torch)
    sc1, sc2 = _items(torch, H, W, V=30, S=20, seed=0), _items(torch, H, W, V=30, S=20, seed=40)
    host1 = _host_chain(torch, sc1, icn)
    host2 = _host_chain(torch, sc2, icn)
    w1, w2 = host1["windows"], host2["windows"]
    cap = (max(w1.nbytes, w2.nbytes), max(w1.max_h, w2.max_h))
    _device_chain(torch, sc1, icn, cap)                               # warm-up: Lab tables, weights, allocator
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        eager = _device_chain(torch, sc1, icn, cap)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    _assert_chains_equal(torch, host1, eager)
    del eager
    static = {k: (v.clone() if hasattr(v, "clone") else v) for k, v in sc1.items()}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _device_chain(torch, static, icn, cap)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _device_chain(torch, static, icn, cap)
    graph.replay()
    torch.cuda.synchronize()
    _assert_chains_equal(torch, host1, out)
    _copy_inputs(static, sc2)
    graph.replay()
    torch.cuda.synchronize()
    _assert_chains_equal(torch, host2, out)
    assert not torch.equal(host1["f_icn"], host2["f_icn"])


def test_one_bbox_pass_for_the_destination_masks(cuda):
    """The device chain runs fusg_mask_bbox once on the destination masks; the host chain three times (icn_windows, get_icn_inputs,
    y_tilde packing)."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    icn = _icn_model(torch)
    sc = _items(torch, 300, 400, V=3, S=4, seed=7)
    L = _lib.lib()
    orig, calls = L.fusg_mask_bbox, []
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(L, "fusg_mask_bbox", lambda *a: (calls.append(int(a[4])), orig(*a))[1])
        host = _host_chain(torch, sc, icn)
        n_host = len(calls)
        calls.clear()
        _device_chain(torch, sc, icn, (host["windows"].nbytes, host["windows"].max_h))
        torch.cuda.synchronize()
    assert n_host == 3 and calls == [sc["N"]]


# ---------------------------------------------------------------------------------------------------- 4. the clip script
def test_clip_script_device_geometry_matches_the_default(cuda):
    runs = {}
    for extra in ([], ["--device-geometry"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_clip.py"), "--vehicles", "3", "--steps", "2", "--chunk", "4",
                              "--reps", "1"] + extra, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        d = json.loads(out.stdout.strip().splitlines()[-1])
        assert d["items"] == 6 and d["device_geometry"] == bool(extra)
        runs[bool(extra)] = d
    assert runs[True]["sha1"] == runs[False]["sha1"]
    assert runs[True]["mask_bbox_passes"].count(6) == 1 and runs[False]["mask_bbox_passes"].count(6) == 2
