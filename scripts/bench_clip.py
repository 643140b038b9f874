"""BASELINE config 5 end to end on one B200: a Cityflow-shape clip -- 30 vehicles x 20 future trajectory steps on 1920x1080
frames -- through every row of SURVEY.md section 8 in the reference's order (trajectory_inference.py:255-445), device resident:

  kinematics   trajectory_poses (host scalars) + fusg_step_keypoints           :267-298, :359-367
  warp         fusg_warp_fused_traj on whole frames (5 planes per item)        :374-379
  icn inputs   fusg_mask_bbox + fusg_pack_icn_inputs                           :387-388
  icn          G_Resnet forward                                                :391
  vunet        enc_up/enc_down once per vehicle, dec_up/dec_down per item      :230-233, :413-425
  paste        to_image + fusg_paste_back into the 20 result frames, both generators   :393-407, :426-442

Synthetic scene (synth.make_trajectory_case; synthetic CAD meshes rendered by the device rasteriser stand in for the Open3D
renderer).

--icn-window runs the ICN branch in its windowed form instead: sketches -> icn_windows -> fused warp of only each item's ICN crop
window, reading the one source frame through src_index (no N-fold copy of the frame) -> get_icn_inputs_batch from the windows.
--device-geometry computes the crop geometry of the destination masks once, on the device (frame_ops.crop_geometry: one bbox pass, no
host round trip), and feeds it to the ICN packing, the y_tilde packing and both paste-backs, which then run no bbox pass of their own.
The JSON line carries the SHA-1 of both generators' composited frames, so that the forms can be compared, and the batch size of every
fusg_mask_bbox pass of the last clip.
usage: python scripts/bench_clip.py [--vehicles 30] [--steps 20] [--icn-window | --device-geometry] [--out clip.json]"""
import argparse
import hashlib
import json
import os
import sys
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from future_urban_scene_generation_b200 import synth, kinematics, _lib
from future_urban_scene_generation_b200.warp_learn import warp_batch
from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch
from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
from future_urban_scene_generation_b200.frame_ops import (PastePlan, crop_geometry, get_icn_inputs_batch, icn_windows, pack_vunet_inputs_batch,
                                                         paste_back_batch, paste_back_packed)

ap = argparse.ArgumentParser()
ap.add_argument("--vehicles", type=int, default=30)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--chunk", type=int, default=100)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--icn-window", action="store_true", help="warp only the ICN crop windows (see the module docstring)")
ap.add_argument("--device-geometry", action="store_true", help="one device-side crop geometry for the whole chain (module docstring)")
ap.add_argument("--out", default=None)
args = ap.parse_args()
if args.icn_window and args.device_geometry:
    ap.error("--icn-window and --device-geometry are separate forms")
V, S, H, W = args.vehicles, args.steps, 1080, 1920
N = V * S
dev = torch.device("cuda")
torch.manual_seed(0)

# ---- scene (host, outside the timed region) --------------------------------------------------------------------------------
cases = []
for v in range(V):
    c = synth.make_trajectory_case(v, steps=S, h=H, w=W)
    c["K"] = np.array([[1650.0, 0, W / 2.0], [0, 1650.0, H / 2.0], [0, 0, 1.0]])
    cases.append(c)
frame = np.random.default_rng(1).integers(0, 256, (H, W, 3), dtype=np.uint8)
veh_of_item = np.repeat(np.arange(V), S)
step_of_item = np.tile(np.arange(S), V)
kp3d = np.stack([c["kp3d"] for c in cases])
R = np.stack([c["R"] for c in cases])
t = np.stack([c["t"] for c in cases])
K = np.stack([c["K"] for c in cases])
E = np.concatenate([R, t[:, :, None]], 2)                       # (V,3,4)
src_kp2d = np.stack([synth.project(K[v], np.vstack([E[v], [0, 0, 0, 1]]), kp3d[v]) for v in range(V)])
src_kp = np.int32((src_kp2d / [W, H]) * [W, H])

from future_urban_scene_generation_b200.warp_learn.render import render_normals_batch, MeshOnDevice
meshes = [MeshOnDevice(*synth.make_car_mesh(v % 10)) for v in range(V)]
vunet = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).cuda().eval()
icn = G_Resnet(21).cuda().eval()
frames_dev = torch.from_numpy(frame).to(dev)
mask_bbox_passes = []                                                  # batch size of every fusg_mask_bbox call
_mask_bbox = _lib.lib().fusg_mask_bbox
_lib.lib().fusg_mask_bbox = lambda *a: (mask_bbox_passes.append(int(a[4])), _mask_bbox(*a))[1]
yy = torch.arange(H, device=dev, dtype=torch.float32).view(1, H, 1)
xx = torch.arange(W, device=dev, dtype=torch.float32).view(1, 1, W)


def ellipse_masks(kp):
    """(n,12,2) int vertices -> (n,H,W) bool: an ellipse inscribed in the keypoints' bounding box (the vehicle silhouette stand-in)."""
    kp = kp.float()
    x0, x1 = kp[:, :, 0].min(1).values, kp[:, :, 0].max(1).values
    y0, y1 = kp[:, :, 1].min(1).values, kp[:, :, 1].max(1).values
    cx, cy = ((x0 + x1) / 2).clamp(20, W - 20).view(-1, 1, 1), ((y0 + y1) / 2).clamp(20, H - 20).view(-1, 1, 1)   # never empty
    rx, ry = ((x1 - x0) / 2 + 6).clamp(8, 600).view(-1, 1, 1), ((y1 - y0) / 2 + 6).clamp(8, 400).view(-1, 1, 1)
    return ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0


def normals_for(masks, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    base = torch.randint(1, 256, (1, H, W, 3), generator=g, device=dev, dtype=torch.uint8)
    return base * masks.unsqueeze(-1).to(torch.uint8)


def clip():
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in
          ("kinematics", "warp", "sketches", "icn_inputs", "icn", "vunet_inputs", "vunet", "paste") + (("icn_windows",) if args.icn_window else ())
          + (("crop_geometry",) if args.device_geometry else ())}
    # 1. kinematics
    ev["kinematics"][0].record()
    poses = [kinematics.trajectory_poses(c["meter_coords"]) for c in cases]
    rot = np.concatenate([p[2] for p in poses])
    tr = np.concatenate([p[1] for p in poses])
    moved, kp2d, dst_kp = kinematics.step_keypoints_batch(kp3d, veh_of_item, rot, tr, R, t, K, H, W)
    global dst_kp_last
    dst_kp_last = dst_kp
    ev["kinematics"][1].record()
    vi = torch.as_tensor(veh_of_item, device=dev)

    def warp(window=None):
        # fused warp for every (vehicle, step): whole frames, or (window) only each item's ICN crop window of the one source frame
        ev["warp"][0].record()
        if window is None:
            src, idx = frames_dev.unsqueeze(0).expand(N, H, W, 3).contiguous(), None
        else:
            src, idx = frames_dev.unsqueeze(0), torch.zeros(N, dtype=torch.int32, device=dev)
        r = warp_batch(src, torch.as_tensor(src_kp, device=dev)[vi], dst_kp, torch.as_tensor(K, device=dev)[vi], torch.as_tensor(E, device=dev)[vi],
                       torch.as_tensor(E, device=dev)[vi], torch.as_tensor(kp3d, device=dev)[vi], kp3d_dst=moved, src_index=idx, window=window)
        ev["warp"][1].record()
        return r

    # 2. fused warp of the whole frame (default; with --icn-window it follows the sketches, whose masks place the windows)
    if not args.icn_window:
        res = warp()
    # 2b. normal sketches + object masks of every (vehicle, step): the device rasteriser (render_open3d.get_rendered's job)
    ev["sketches"][0].record()
    E4 = torch.as_tensor(E, device=dev)
    K4 = torch.as_tensor(K, device=dev)
    rot_t, tr_t = torch.as_tensor(rot, device=dev).double(), torch.as_tensor(tr, device=dev)
    dst_normals = torch.empty((N, H, W, 3), dtype=torch.uint8, device=dev)
    src_normals = torch.empty((V, H, W, 3), dtype=torch.uint8, device=dev)
    dst_bg = torch.empty((N, H, W), dtype=torch.bool, device=dev)
    src_bg = torch.empty((V, H, W), dtype=torch.bool, device=dev)
    for v in range(V):
        sl = slice(v * S, (v + 1) * S)
        render_normals_batch(meshes[v], E4[v:v + 1].expand(S, 3, 4), K4[v:v + 1].expand(S, 3, 3), H, W, rot=rot_t[sl], tr=tr_t[sl],
                             out=(dst_normals[sl], dst_bg[sl]))
        render_normals_batch(meshes[v], E4[v:v + 1], K4[v:v + 1], H, W, out=(src_normals[v:v + 1], src_bg[v:v + 1]))
    dst_masks, src_masks = ~dst_bg, ~src_bg                               # trajectory_inference.py:175: the object, not the background
    # (items whose vehicle has left the frame: keep one pixel so that the crop geometry downstream stays defined, like the
    # reference's bare `except: break` would simply end that vehicle's trajectory)
    empty = ~dst_masks.flatten(1).any(1)
    dst_masks[empty, H // 2, W // 2] = True
    ev["sketches"][1].record()
    if args.icn_window:
        ev["icn_windows"][0].record()
        windows = icn_windows(dst_masks, (H, W))
        ev["icn_windows"][1].record()
        res = warp(windows)
    if args.device_geometry:
        ev["crop_geometry"][0].record()
        geom = crop_geometry(dst_masks, (H, W), frame_index=torch.as_tensor(step_of_item, device=dev).to(torch.int32))
        ev["crop_geometry"][1].record()
    central = torch.randint(0, 256, (N, 256, 256, 3), device=dev, dtype=torch.uint8)
    # 3. ICN inputs
    ev["icn_inputs"][0].record()
    if args.device_geometry:
        gen_in, _ = get_icn_inputs_batch(res.warped, dst_normals, None, central, geometry=geom)
    else:
        gen_in, crop_infos = get_icn_inputs_batch(res.warped, dst_normals, dst_masks, central)
    ev["icn_inputs"][1].record()
    # 4. ICN
    ev["icn"][0].record()
    icn_img = torch.cat([icn(gen_in[i:i + args.chunk]) for i in range(0, N, args.chunk)])
    ev["icn"][1].record()
    # 5. VUNet: appearance once per vehicle, shape path per item
    ev["vunet_inputs"][0].record()
    x_src, _, _ = pack_vunet_inputs_batch(frames_dev.unsqueeze(0), [0] * V, ~src_masks, src_normals, src_normals)
    if args.device_geometry:
        _, y_all, _ = pack_vunet_inputs_batch(frames_dev.unsqueeze(0), torch.zeros(N, dtype=torch.int32, device=dev), ~dst_masks, dst_normals,
                                              dst_normals, geometry=geom)
    else:
        _, y_all, _ = pack_vunet_inputs_batch(frames_dev.unsqueeze(0), [0] * N, ~dst_masks, dst_normals, dst_normals)
    ev["vunet_inputs"][1].record()
    ev["vunet"][0].record()
    with torch.no_grad():
        e = vunet.engine()
        outs_e, skips_e = e.enc_up(x_src)
        mu, _ = e.enc_down(outs_e, skips_e)
        mu_api = [e.to_nchw(a) for a in mu]
        vun = []
        for i in range(0, N, args.chunk):
            sel = vi[i:i + args.chunk]
            g = [e.g_from_api(m[sel].contiguous()) for m in mu_api]
            od, sd = e.dec_up(y_all[i:i + args.chunk])
            vun.append(e.dec_down(od, sd, g)[0])
        vun_img = torch.cat(vun)
    ev["vunet"][1].record()
    # 6. paste both generators' crops into their result frames
    ev["paste"][0].record()
    frames_icn = frames_dev.unsqueeze(0).repeat(S, 1, 1, 1)
    frames_vun = frames_icn.clone()
    if args.device_geometry:
        # items stay in (vehicle, step) order: inside a frame that is vehicle order, so the same item wins where masks overlap
        plan = PastePlan.from_geometry(geom, dst_masks)
        paste_back_packed(frames_icn, to_image_batch(icn_img, from_LAB=True), plan)
        paste_back_packed(frames_vun, to_image_batch(vun_img), plan)
        ev["paste"][1].record()
        torch.cuda.synchronize()
        return {k: a.elapsed_time(b) for k, (a, b) in ev.items()}, res, frames_icn, frames_vun
    order = np.argsort(step_of_item, kind="stable")                    # vehicles in selection order inside every frame
    infos_l = [crop_infos[i] for i in order]
    fidx = [int(step_of_item[i]) for i in order]
    oi = torch.as_tensor(order, device=dev)
    masks_o = dst_masks[oi]
    paste_back_batch(frames_icn, to_image_batch(icn_img, from_LAB=True)[oi].contiguous(), masks_o, infos_l, fidx)
    paste_back_batch(frames_vun, to_image_batch(vun_img)[oi].contiguous(), masks_o, infos_l, fidx)
    ev["paste"][1].record()
    torch.cuda.synchronize()
    return {k: a.elapsed_time(b) for k, (a, b) in ev.items()}, res, frames_icn, frames_vun


clip()                                                                  # warm-up (weight repack, allocator, table upload)
torch.cuda.synchronize()
runs = []
for _ in range(args.reps):                                              # host-side glue (CPU Sampler noise, Python) varies: report the best of a few
    mask_bbox_passes.clear()
    n0 = _lib.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    stages, res, f_icn, f_vun = clip()
    e1.record()
    torch.cuda.synchronize()
    runs.append((e0.elapsed_time(e1), e0.elapsed_time(e1), stages, _lib.kernel_launches() - n0))
runs.sort(key=lambda r: r[0])
_, total, stages, n_launch = runs[0]
path_ms = total
out = {"workload": f"BASELINE config 5: {V} vehicles x {S} future steps on {W}x{H} frames, {N} (vehicle, step) items, both generators, paste-back into {S} frames each",
       "icn_window": args.icn_window, "device_geometry": args.device_geometry, "items": N, "mask_bbox_passes": mask_bbox_passes, "ms_total": total, "ms_path": path_ms, "items_per_s": N / path_ms * 1e3, "stages_ms": stages,
       "gpu_launches": n_launch, "reps": args.reps, "ms_path_all_reps": [r[0] for r in runs],
       "refused_items": int((res.plane_j[:, 0] == -2).sum().item()),
       "items_with_out_of_frame_keypoints": int(((dst_kp_last < 0) | (dst_kp_last >= torch.tensor([W, H], device=dev))).any(-1).any(-1).sum().item()),
       "written_planes_per_item": float((res.plane_j >= 0).float().sum().item()) / N,
       "changed_pixels": {"icn_frames": int((f_icn != frames_dev).any(-1).sum().item()), "vunet_frames": int((f_vun != frames_dev).any(-1).sum().item())},
       "sha1": {"frames_icn": hashlib.sha1(f_icn.cpu().numpy().tobytes()).hexdigest(), "frames_vun": hashlib.sha1(f_vun.cpu().numpy().tobytes()).hexdigest()},
       "note": "one process, one B200, everything between the scene description and the composited frames on the device; stage times are "
               "CUDA-event brackets around the public calls (incl. their Python glue); 'sketches' is the device rasteriser standing in for the "
               "reference's Open3D window (render_open3d.get_rendered) and is part of ms_path", "data": "synthetic"}
print(json.dumps(out))
if args.out:
    open(args.out, "w").write(json.dumps(out) + "\n")
