"""The warp + ICN-input stages of the whole-frame trajectory chain in its two forms, on one GPU:

  full      fused warp of whole frames (B x 5 x H x W x 3 planes)     -> get_icn_inputs_batch(planes)
  windowed  icn_windows(masks) -> fused warp of the ICN crop windows  -> get_icn_inputs_batch(WindowedPlanes)

Items are (vehicle, future step) pairs from the trajectory kinematics as in scripts/bench_clip.py (30 vehicles x 20 steps = 600
items), on one source frame per vehicle read through src_index in both forms, so that only the output layout differs.  The two
forms alternate in one process for --rounds rounds each; every stage is bracketed by CUDA events.  Reported per frame size: ms per
stage (median and all rounds), bytes of planes written (from shapes: 5*w*h*3 per item against 5*H*W*3), the peak of
torch.cuda.max_memory_allocated over one call of each form, the share of k_plane_masks in the warp call's kernel time (torch.profiler,
a separate pass after the timed rounds), and that gen_in is byte-identical between the forms.  The device name and power limit
come from nvidia-smi in the same run.
usage: python scripts/bench_icn_window.py [--vehicles 30] [--steps 20] [--rounds 5] [--sizes 720x1280,1080x1920] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from future_urban_scene_generation_b200 import synth, kinematics
from future_urban_scene_generation_b200.warp_learn import warp_batch
from future_urban_scene_generation_b200.frame_ops import get_icn_inputs_batch, icn_windows

ap = argparse.ArgumentParser()
ap.add_argument("--vehicles", type=int, default=30)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--sizes", default="720x1280,1080x1920")
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_icn_window.py needs a CUDA device")
dev = torch.device("cuda")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        line = q.stdout.strip().splitlines()[torch.cuda.current_device()]
        name, power = (s.strip() for s in line.split(","))
        return {"name": name, "power_limit": power}
    except Exception as e:                                     # the numbers stay valid; say what could not be read
        return {"name": torch.cuda.get_device_name(), "power_limit": f"not read ({e.__class__.__name__})"}


def scene(H, W):
    """Per-item warp arguments, source frames, destination masks / normals and central crops, all on the device."""
    V, S = args.vehicles, args.steps
    N = V * S
    cases = []
    for v in range(V):
        c = synth.make_trajectory_case(v, steps=S, h=H, w=W)
        f = 1650.0 * W / 1920.0                                # bench_clip's focal length at 1080p, scaled with the frame
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
    warp_args = (torch.as_tensor(src_kp, device=dev)[vi], dst_kp, torch.as_tensor(K, device=dev)[vi], torch.as_tensor(E, device=dev)[vi],
                 torch.as_tensor(E, device=dev)[vi], torch.as_tensor(kp3d, device=dev)[vi])
    frames = torch.randint(0, 256, (V, H, W, 3), generator=torch.Generator(device=dev).manual_seed(1), device=dev, dtype=torch.uint8)
    # destination silhouettes: an ellipse in the keypoints' bounding box (bench_clip's stand-in), never empty
    kp = dst_kp.float()
    yy, xx = torch.arange(H, device=dev, dtype=torch.float32).view(1, H, 1), torch.arange(W, device=dev, dtype=torch.float32).view(1, 1, W)
    x0, x1, y0, y1 = kp[:, :, 0].min(1).values, kp[:, :, 0].max(1).values, kp[:, :, 1].min(1).values, kp[:, :, 1].max(1).values
    cx, cy = ((x0 + x1) / 2).clamp(20, W - 20).view(-1, 1, 1), ((y0 + y1) / 2).clamp(20, H - 20).view(-1, 1, 1)
    rx, ry = ((x1 - x0) / 2 + 6).clamp(8, W / 3).view(-1, 1, 1), ((y1 - y0) / 2 + 6).clamp(8, H / 3).view(-1, 1, 1)
    masks = ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0
    g = torch.Generator(device=dev).manual_seed(2)
    normals = torch.randint(1, 256, (N, H, W, 3), generator=g, device=dev, dtype=torch.uint8) * masks.unsqueeze(-1).to(torch.uint8)
    central = torch.randint(0, 256, (N, 256, 256, 3), generator=g, device=dev, dtype=torch.uint8)
    return dict(N=N, frames=frames, idx=torch.as_tensor(veh, device=dev), warp_args=warp_args, moved=moved, masks=masks, normals=normals,
                central=central)


def run(sc, windowed):
    """One pass of the stages; returns ({stage: ms}, gen_in, the warp result)."""
    names = ("icn_windows", "warp", "icn_pack") if windowed else ("warp", "icn_pack")
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in names}
    window = None
    if windowed:
        ev["icn_windows"][0].record()
        window = icn_windows(sc["masks"], tuple(sc["frames"].shape[1:3]))
        ev["icn_windows"][1].record()
    ev["warp"][0].record()
    res = warp_batch(sc["frames"], *sc["warp_args"], kp3d_dst=sc["moved"], src_index=sc["idx"], window=window)
    ev["warp"][1].record()
    ev["icn_pack"][0].record()
    gen_in, _ = get_icn_inputs_batch(res.warped, sc["normals"], sc["masks"], sc["central"])
    ev["icn_pack"][1].record()
    torch.cuda.synchronize()
    return {k: a.elapsed_time(b) for k, (a, b) in ev.items()}, gen_in, res


def plane_masks_share(sc, windowed):
    """k_plane_masks' share of the kernel time of one warp call (torch.profiler, CUDA activities)."""
    from torch.profiler import profile, ProfilerActivity
    window = icn_windows(sc["masks"], tuple(sc["frames"].shape[1:3])) if windowed else None
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        warp_batch(sc["frames"], *sc["warp_args"], kp3d_dst=sc["moved"], src_index=sc["idx"], window=window)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and e.key.startswith(("void fusg::", "fusg::")):
            per[e.key] = per.get(e.key, 0.0) + t
    total = sum(per.values())
    masks = sum(v for k, v in per.items() if "k_plane_masks" in k)
    return {"k_plane_masks_us": masks, "warp_kernels_us": total, "share": masks / total if total else None,
            "kernels_us": {k.split("(")[0].replace("void ", ""): v for k, v in per.items()}}


result = {"gpu": gpu_info(), "items": args.vehicles * args.steps, "rounds": args.rounds, "sizes": []}
for hw in args.sizes.split(","):
    H, W = (int(v) for v in hw.split("x"))
    sc = scene(H, W)
    N = sc["N"]
    # warm-up of both forms (module load, allocator, Lab tables), then one call each under a fresh memory peak
    peaks = {}
    for windowed in (False, True):
        run(sc, windowed)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        _, gi, res = run(sc, windowed)
        peaks["windowed" if windowed else "full"] = torch.cuda.max_memory_allocated() - base
        if windowed:
            rect = res.warped.rect
            gen_win = gi
        else:
            gen_full = gi
        del res
    assert torch.equal(gen_full.view(torch.int32), gen_win.view(torch.int32)), "gen_in differs between the forms"
    del gen_full, gen_win
    times = {"full": [], "windowed": []}
    for _ in range(args.rounds):                               # alternate the forms: both see the same state of the shared machine
        for windowed in (False, True):
            st, gi, res = run(sc, windowed)
            times["windowed" if windowed else "full"].append(st)
            del gi, res
    summary = {}
    for form, rounds in times.items():
        keys = rounds[0].keys()
        summary[form] = {k: {"median_ms": statistics.median(r[k] for r in rounds), "all_ms": [r[k] for r in rounds]} for k in keys}
        summary[form]["sum_median_ms"] = sum(summary[form][k]["median_ms"] for k in keys)
    bytes_full = N * 5 * H * W * 3
    bytes_win = int((5 * rect[:, 2].astype(np.int64) * rect[:, 3] * 3).sum())
    result["sizes"].append({
        "frame_hw": [H, W], "items": N,
        "ms": summary,
        "planes_bytes_written": {"full": bytes_full, "windowed": bytes_win, "ratio_full_over_windowed": bytes_full / bytes_win},
        "window_px": {"mean_w": float(rect[:, 2].mean()), "mean_h": float(rect[:, 3].mean()), "max_h": int(rect[:, 3].max())},
        "peak_memory_bytes": {**peaks, "ratio_full_over_windowed": peaks["full"] / peaks["windowed"]},
        "k_plane_masks": {"full": plane_masks_share(sc, False), "windowed": plane_masks_share(sc, True)},
        "gen_in_identical": True})
    del sc
    torch.cuda.empty_cache()
result["note"] = ("ms per stage are CUDA-event brackets around the public calls, Python glue included; icn_windows synchronises (one "
                  "device->host copy of the bboxes); peak memory is max_memory_allocated over one call of the form above what the inputs "
                  "already held; data: synthetic")
print(json.dumps(result))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    open(args.out, "w").write(json.dumps(result, indent=1) + "\n")
