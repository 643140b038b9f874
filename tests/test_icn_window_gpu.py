"""The ICN-window form of the whole-frame chain: the fused warp writing only each item's ICN crop window
(fusg_warp_fused_window / warp_batch(..., window=)) and get_icn_inputs_batch reading those windows, against the full-frame
warp and packing they replace -- bit for bit."""
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "frame_golden.json")))
SENTINEL = 0xA5


def _box_masks(torch, dst_kp, H, W):
    """(B,H,W) bool: the bounding box of each item's destination keypoints clipped to the frame (never empty) -- a silhouette stand-in
    whose window follows the vehicle to the frame border."""
    kp = torch.as_tensor(dst_kp).reshape(-1, 12, 2).long().cpu()
    x0 = kp[:, :, 0].min(1).values.clamp(0, W - 1); x1 = kp[:, :, 0].max(1).values.clamp(0, W - 1)
    y0 = kp[:, :, 1].min(1).values.clamp(0, H - 1); y1 = kp[:, :, 1].max(1).values.clamp(0, H - 1)
    ys, xs = torch.arange(H).view(1, H, 1), torch.arange(W).view(1, 1, W)
    return ((ys >= y0.view(-1, 1, 1)) & (ys <= y1.view(-1, 1, 1)) & (xs >= x0.view(-1, 1, 1)) & (xs <= x1.view(-1, 1, 1))).cuda()


def _trajectory_items(torch, H, W, V=3, S=4):
    """Trajectory items from kinematics.step_keypoints_batch, as tests/test_trajectory_gpu.py builds them: (frames (V,H,W,3),
    per-item vehicle index, warp arguments, moved keypoints)."""
    from future_urban_scene_generation_b200 import kinematics as KM, synth
    cases = [synth.make_trajectory_case(v, steps=S, h=H, w=W) for v in range(V)]
    for c in cases:
        c["K"] = np.array([[1.3 * W, 0, W / 2.0], [0, 1.3 * W, H / 2.0], [0, 0, 1.0]])
    kp3d = np.stack([c["kp3d"] for c in cases])
    R, t, K = np.stack([c["R"] for c in cases]), np.stack([c["t"] for c in cases]), np.stack([c["K"] for c in cases])
    E = np.concatenate([R, t[:, :, None]], 2)
    src_kp = np.int32(np.stack([synth.project(K[v], np.vstack([E[v], [0, 0, 0, 1]]), kp3d[v]) for v in range(V)]))
    poses = [KM.trajectory_poses(c["meter_coords"]) for c in cases]
    veh = np.repeat(np.arange(V), S).astype(np.int32)
    moved, _, dst_kp = KM.step_keypoints_batch(kp3d, veh, np.concatenate([p[2] for p in poses]), np.concatenate([p[1] for p in poses]),
                                               R, t, K, H, W)
    order = np.array([5, 0, 11, 2, 2, 7, 1, 9, 4, 10, 3, 6, 8], np.int64)
    o = torch.as_tensor(order).cuda()
    wb = dict(src_kp=src_kp[veh[order]], dst_kp=dst_kp[o].cpu().numpy(), K=K[veh[order]], E_src=E[veh[order]], E_dst=E[veh[order]],
              kp3d=kp3d[veh[order]])
    frames = np.stack([np.random.default_rng(500 + v).integers(0, 256, (H, W, 3), dtype=np.uint8) for v in range(V)])
    return frames, veh[order], wb, moved[o]


def _args(wb):
    return (wb["src_kp"], wb["dst_kp"], wb["K"], wb["E_src"], wb["E_dst"], wb["kp3d"])


def _assert_windows_match(torch, win_res, full_res, windows, items=None):
    """item(b) == the whole-frame planes cropped to the window; vis / plane_j / H12 bits identical."""
    assert torch.equal(win_res.vis, full_res.vis)
    assert torch.equal(win_res.plane_j, full_res.plane_j)
    assert torch.equal(win_res.H12.view(torch.int64), full_res.H12.view(torch.int64))
    for b in (range(len(windows)) if items is None else items):
        x0, y0, w, h = (int(v) for v in windows.rect[b])
        assert torch.equal(win_res.warped.item(b), full_res.warped[b, :, y0:y0 + h, x0:x0 + w]), b


def _prefilled(torch, windows, guard=4096):
    """A WarpResult whose window buffer (plus a guard band after the last window) holds the sentinel."""
    from future_urban_scene_generation_b200.frame_ops import WindowedPlanes
    from future_urban_scene_generation_b200.warp_learn.batch import WarpResult
    B = len(windows)
    data = torch.full((windows.nbytes + guard,), SENTINEL, dtype=torch.uint8, device="cuda")
    return WarpResult(warped=WindowedPlanes(data, windows), vis=torch.empty((B, 2, 7), dtype=torch.uint8, device="cuda"),
                      plane_j=torch.empty((B, 5), dtype=torch.int8, device="cuda"), H12=torch.empty((B, 5, 3, 3), dtype=torch.float64, device="cuda"))


def _unwritten(windows, total):
    """Byte mask (numpy bool) of the buffer bytes outside every window: alignment gaps and the guard band."""
    m = np.ones(total, bool)
    for b in range(len(windows)):
        x0, y0, w, h = (int(v) for v in windows.rect[b])
        o = int(windows.off[b])
        m[o:o + 5 * h * w * 3] = False
    return m


# ---------------------------------------------------------------------------------------------------- 1 + 2. the windowed warp
@pytest.mark.parametrize("hw", [(256, 256), (300, 400), (720, 1280), (1080, 1920)])
@pytest.mark.parametrize("indexed", [False, True])
@pytest.mark.parametrize("moved", [False, True])
def test_windowed_warp_equals_full_frame_cropped(cuda, hw, indexed, moved):
    """Whole-frame trajectory items: every window byte equals the full-frame warp (k_warp_rows at 256^2, k_warp_frame above), every
    window byte is written and no byte outside the windows is."""
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import icn_windows
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    H, W = hw
    frames, veh, wb, kd = _trajectory_items(torch, H, W)
    kd = kd if moved else None
    fr = torch.as_tensor(frames).cuda()
    windows = icn_windows(_box_masks(torch, wb["dst_kp"], H, W), (H, W))
    if indexed:
        idx = torch.as_tensor(veh).cuda()
        full = warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx)
        out = _prefilled(torch, windows)
        win = warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx, window=windows, out=out)
    else:
        src = fr[torch.as_tensor(veh).long().cuda()].contiguous()
        full = warp_batch(src, *_args(wb), kp3d_dst=kd)
        out = _prefilled(torch, windows)
        win = warp_batch(src, *_args(wb), kp3d_dst=kd, window=windows, out=out)
    torch.cuda.synchronize()
    assert win is out
    _assert_windows_match(torch, win, full, windows)
    assert int((win.plane_j >= 0).sum()) > 0 and any(int(win.warped.item(b).count_nonzero()) > 0 for b in range(len(windows)))
    data = win.warped.data.cpu().numpy()
    assert (data[_unwritten(windows, data.size)] == SENTINEL).all()


@pytest.mark.parametrize("hw", [(256, 256), (300, 400)])
def test_windowed_warp_out_of_frame_vehicles(cuda, hw):
    """Vehicles that straddle a frame border (synth.make_warp_batch(out_of_frame=True)): windows touching the border."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import icn_windows
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    H, W = hw
    B = 10
    wb = synth.make_warp_batch(70, B, h=H, w=W, out_of_frame=True)
    src = torch.as_tensor(wb["src"]).cuda()
    windows = icn_windows(_box_masks(torch, wb["dst_kp"], H, W), (H, W))
    r = windows.rect
    assert ((r[:, 0] == 0) | (r[:, 1] == 0) | (r[:, 0] + r[:, 2] == W) | (r[:, 1] + r[:, 3] == H)).sum() >= 3
    full = warp_batch(src, *_args(wb))
    win = warp_batch(src, *_args(wb), window=windows, out=_prefilled(torch, windows))
    torch.cuda.synchronize()
    _assert_windows_match(torch, win, full, windows)
    data = win.warped.data.cpu().numpy()
    assert (data[_unwritten(windows, data.size)] == SENTINEL).all()


# ---------------------------------------------------------------------------------------------------- 3. refusals
def test_windowed_warp_refusals(cuda):
    """An absurd vertex and a device src_index out of range: plane_j = -2 and an all-zero window.  A window outside the frame or
    taller than max_win_h: that item alone is refused and its block is not written.  check=True raises RefusedCrops."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    from future_urban_scene_generation_b200.frame_ops import icn_windows
    from future_urban_scene_generation_b200.warp_learn import warp_batch, RefusedCrops
    H, W = 720, 1280
    frames, veh, wb, kd = _trajectory_items(torch, H, W)
    B = len(veh)
    wb["src_kp"] = wb["src_kp"].copy()
    wb["src_kp"][1, 3] = (_lib.POLY_COORD_MAX * 2, 5)                     # item 1: absurd vertex
    idx = torch.as_tensor(veh).cuda()
    idx[4] = 17                                                             # item 4: no such source image
    fr = torch.as_tensor(frames).cuda()
    windows = icn_windows(_box_masks(torch, wb["dst_kp"], H, W), (H, W))
    # item 6: a window that leaves the frame; the tallest of the others: taller than max_win_h
    windows.rect[6, 0] = W - windows.rect[6, 2] + 1
    windows.rect_dev = torch.from_numpy(windows.rect).cuda()
    hs = windows.rect[:, 3]
    tall = max((b for b in range(B) if b not in (1, 4, 6)), key=lambda b: hs[b])
    windows.max_h = int(hs[tall]) - 1
    nowrite = sorted({6} | {b for b in range(B) if b != 6 and hs[b] > windows.max_h})
    zeroed = [b for b in (1, 4) if b not in nowrite]
    assert zeroed and tall in nowrite
    full = warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx)
    win = warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx, window=windows, out=_prefilled(torch, windows))
    torch.cuda.synchronize()
    refused = sorted(set(zeroed) | set(nowrite))
    pj = win.plane_j.cpu()
    for b in refused:
        assert (pj[b] == -2).all(), b
        assert int(win.H12[b].abs().sum()) == 0
    ok = [b for b in range(B) if b not in refused]
    assert not (pj[ok] == -2).any()
    assert torch.equal(win.plane_j[ok], full.plane_j[ok]) and torch.equal(win.vis, full.vis)
    assert torch.equal(win.H12[ok].view(torch.int64), full.H12[ok].view(torch.int64))
    for b in ok:
        x0, y0, w, h = (int(v) for v in windows.rect[b])
        assert torch.equal(win.warped.item(b), full.warped[b, :, y0:y0 + h, x0:x0 + w]), b
    for b in zeroed:
        assert int(win.warped.item(b).count_nonzero()) == 0, b
    data = win.warped.data
    for b in nowrite:
        x0, y0, w, h = (int(v) for v in windows.rect[b])
        o = int(windows.off[b])
        assert bool((data[o:o + 5 * h * w * 3] == SENTINEL).all()), b
    with pytest.raises(RefusedCrops) as ei:
        warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx, window=windows, check=True)
    assert ei.value.indices == refused


# ---------------------------------------------------------------------------------------------------- 4. ICN inputs from windows
def _cut_windows(torch, planes, windows):
    """Whole-frame planes (B,5,H,W,3) -> WindowedPlanes holding their windows."""
    from future_urban_scene_generation_b200.frame_ops import WindowedPlanes
    wp = WindowedPlanes(torch.zeros((windows.nbytes,), dtype=torch.uint8, device="cuda"), windows)
    for b in range(len(windows)):
        x0, y0, w, h = (int(v) for v in windows.rect[b])
        wp.item(b).copy_(planes[b, :, y0:y0 + h, x0:x0 + w])
    return wp


def _assert_same_inputs(torch, a, b):
    assert torch.equal(a[0].view(torch.int32), b[0].view(torch.int32))
    assert a[1] == b[1]


def test_icn_inputs_from_windows_match_the_goldens(cuda):
    """The golden get_icn_inputs cases (crops hanging over the border) with the full planes cut into windows."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import get_icn_inputs_batch, icn_windows
    for c in GOLD["icn_inputs"]:
        planes, normal, mask, central = synth.make_icn_pack_case(c["idx"], tuple(c["frame_hw"]))
        pl = torch.as_tensor(planes[None]).cuda()
        windows = icn_windows(mask[None], tuple(c["frame_hw"]))
        full = get_icn_inputs_batch(pl, normal[None], mask[None], central[None])
        win = get_icn_inputs_batch(_cut_windows(torch, pl, windows), normal[None], mask[None], central[None])
        torch.cuda.synchronize()
        _assert_same_inputs(torch, win, full)
        assert hashlib.sha1(np.ascontiguousarray(win[0][0].cpu().numpy()).tobytes()).hexdigest() == c["sha1"], c["idx"]
        assert win[1] == windows.crop_infos


def test_icn_inputs_from_windows_exact_halving(cuda):
    """A crop of exactly 512 px takes the 2x2 box-average branch."""
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import get_icn_inputs_batch, icn_windows, square_crop_info
    H, W = 720, 1280
    found = []
    for side in range(440, 480):
        for x0, y0 in ((300, 100), (0, 150), (W - side - 1, 0)):
            if square_crop_info((H, W), (x0, y0, x0 + side, y0 + side))["crop_size_orig"] == (512, 512):
                found.append((x0, y0, side))
    assert found
    rng = np.random.default_rng(11)
    B = len(found)
    masks = np.zeros((B, H, W), bool)
    for b, (x0, y0, side) in enumerate(found):
        masks[b, y0:y0 + side + 1, x0:x0 + side + 1] = True
    planes = torch.as_tensor(rng.integers(0, 256, (B, 5, H, W, 3), dtype=np.uint8)).cuda()
    normals = rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)
    central = rng.integers(0, 256, (B, 256, 256, 3), dtype=np.uint8)
    windows = icn_windows(masks, (H, W))
    full = get_icn_inputs_batch(planes, normals, masks, central)
    win = get_icn_inputs_batch(_cut_windows(torch, planes, windows), normals, masks, central)
    torch.cuda.synchronize()
    _assert_same_inputs(torch, win, full)
    assert all(ci["crop_size_orig"] == (512, 512) for ci in win[1])


@pytest.mark.parametrize("hw", [(720, 1280), (1080, 1920)])
def test_warp_to_icn_inputs_chain_from_windows(cuda, hw):
    """sketch masks -> icn_windows -> windowed warp (src_index, moved keypoints) -> get_icn_inputs_batch equals the whole-frame
    chain; masks that are not those the windows were cut for raise ValueError."""
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import get_icn_inputs_batch, icn_windows
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    H, W = hw
    frames, veh, wb, kd = _trajectory_items(torch, H, W)
    B = len(veh)
    masks = _box_masks(torch, wb["dst_kp"], H, W)
    g = torch.Generator(device="cuda").manual_seed(4)
    normals = torch.randint(0, 256, (B, H, W, 3), generator=g, device="cuda", dtype=torch.uint8) * masks.unsqueeze(-1).to(torch.uint8)
    central = torch.randint(0, 256, (B, 256, 256, 3), generator=g, device="cuda", dtype=torch.uint8)
    fr, idx = torch.as_tensor(frames).cuda(), torch.as_tensor(veh).cuda()
    full = warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx)
    ref = get_icn_inputs_batch(full.warped, normals, masks, central)
    windows = icn_windows(masks, (H, W))
    win = warp_batch(fr, *_args(wb), kp3d_dst=kd, src_index=idx, window=windows)
    got = get_icn_inputs_batch(win.warped, normals, masks, central)
    torch.cuda.synchronize()
    _assert_same_inputs(torch, got, ref)
    assert sum(int(win.warped.item(b).count_nonzero()) for b in range(B)) > 0      # the windows carry warped pixels
    shifted = torch.roll(masks, 1, dims=2)
    with pytest.raises(ValueError):
        get_icn_inputs_batch(win.warped, normals, shifted, central)


# ---------------------------------------------------------------------------------------------------- 5. the clip script
def test_clip_script_icn_window_mode_matches_the_default(cuda):
    import subprocess
    import sys
    hashes = []
    for extra in ([], ["--icn-window"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_clip.py"), "--vehicles", "3", "--steps", "2", "--chunk", "4",
                              "--reps", "1"] + extra, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        d = json.loads(out.stdout.strip().splitlines()[-1])
        assert d["items"] == 6 and d["icn_window"] == bool(extra)
        hashes.append((d["sha1"]["frames_icn"], d["sha1"]["frames_vun"]))
    assert hashes[0] == hashes[1]
