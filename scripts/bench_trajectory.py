#!/usr/bin/env python
"""Throughput of the trajectory form (pipeline.TrajectoryPipeline) next to the per-item full forward (NovelViewPipeline) on the
same items, in one process, the two run alternately.

Workload: one step = B = 64 items = V = 8 vehicles x 8 future steps, synthetic 256x256 crops (synth), random-init weights,
host inputs as pinned uint8 buffers.  TrajectoryPipeline gets the per-vehicle source crops and appearance images once
(`set_vehicles`, outside the timed loops; its own time is reported as set_vehicles_ms) and per item the warp inputs and the
uint8 destination sketch; NovelViewPipeline gets, per item, the source crop and all three uint8 images (what bench.py ships).
Depth and warm-up follow bench.py: device-resident loop (graph replays only, inputs and noise already in HBM) with 2 slots,
end-to-end loop (H2D of the inputs, Sampler noise on the CPU generator, crops + flags D2H) with 3 slots on one stream.

  python scripts/bench_trajectory.py [--steps 50] [--warmup 3] [--reps 3]

Prints one JSON line: per pipeline the median over `reps` repetitions and the (min, max) spread.  Writes nothing."""
import argparse
import collections
import json
import os
import statistics
import subprocess
import sys
import time
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from future_urban_scene_generation_b200 import synth
from future_urban_scene_generation_b200.pipeline import NovelViewPipeline, TrajectoryPipeline
from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res

ap = argparse.ArgumentParser()
ap.add_argument("--vehicles", type=int, default=8)
ap.add_argument("--steps-per-vehicle", type=int, default=8)
ap.add_argument("--steps", type=int, default=50, help="timed pipeline steps per loop")
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()

if not torch.cuda.is_available():
    raise SystemExit("bench_trajectory.py: no CUDA device; the B200 path has no CPU fallback")
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
V, S = args.vehicles, args.steps_per_vehicle
B = V * S


def pinned(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


# ---- items: vehicle v, future step s -> item v * S + s
veh = np.repeat(np.arange(V), S).astype(np.int32)
wb = synth.make_warp_batch(0, B, crops=False)
src_v = np.stack([synth.make_crop(10_000 + v) for v in range(V)])
mk_v, ns_v, _ = synth.make_vunet_inputs_u8(10_000, V)
_, _, nd = synth.make_vunet_inputs_u8(0, B)
warp_in = {k: pinned(v) for k, v in wb.items()}
traj_vehicles = {"src": pinned(src_v), "x_mask_u8": pinned(mk_v), "x_normal_u8": pinned(ns_v)}
traj_host = dict(warp_in, vehicle=pinned(veh), y_normal_u8=pinned(nd))
nv_host = dict(warp_in, src=pinned(src_v[veh]), x_mask_u8=pinned(mk_v[veh]), x_normal_u8=pinned(ns_v[veh]), y_normal_u8=pinned(nd))


def nbytes(d):
    return sum(t.numel() * t.element_size() for t in d.values())


torch.manual_seed(0)
model = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).to(dev).eval()
model.engine()


def run_steps(pipe, n, resident, host):
    pending, last = collections.deque(), None
    for _ in range(n):
        last = pipe.submit(host, resident=resident)
        pending.append(last)
        if len(pending) >= pipe.depth and not resident:
            pipe.result(pending.popleft())
    if resident:
        pipe.wait(last)
    else:
        while pending:
            pipe.result(pending.popleft())
    return last


def timed(pipe, n, resident, host, first_stream, last_stream_of):
    """Device events on the first / last stream, cross-checked with the host clock around work that ends in a synchronise."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(first_stream)
    last = run_steps(pipe, n, resident, host)
    e1.record(last_stream_of(last))
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    return max(e0.elapsed_time(e1), wall)


def make(kind, depth, **kw):
    if kind == "trajectory":
        p = TrajectoryPipeline(model, max_vehicles=V, depth=depth, **kw)
        p.set_vehicles(traj_vehicles)
        return p, traj_host
    return NovelViewPipeline(model, depth=depth, **kw), nv_host


warm = max(3, args.warmup)
pipes = {}
for kind in ("trajectory", "novel_view"):
    r, host = make(kind, 2)
    run_steps(r, warm, False, host)
    e, _ = make(kind, 3, shared_stream=True)
    run_steps(e, max(2, warm), False, host)
    pipes[kind] = (r, e, host)

res = {k: collections.defaultdict(list) for k in pipes}
for rep in range(args.reps):
    for kind, (r, e, host) in pipes.items():                    # alternate the two pipelines inside every repetition
        ms = timed(r, args.steps, True, host, r.slots[r.n % r.depth].stream, lambda t, r=r: r.slots[t % r.depth].stream)
        res[kind]["resident_ms_per_step"].append(ms / args.steps)
        ms = timed(e, args.steps, False, host, e.copy_stream, lambda t, e=e: e.out_stream)
        res[kind]["e2e_ms_per_step"].append(ms / args.steps)
    # the per-vehicle encode the trajectory loops leave out: one set_vehicles of V vehicles (host clock, ends in a synchronise)
    r = pipes["trajectory"][0]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r.set_vehicles(traj_vehicles)
    torch.cuda.synchronize()
    res["trajectory"]["set_vehicles_ms"].append((time.perf_counter() - t0) * 1e3)


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


out = {}
for kind, (r, e, host) in pipes.items():
    d = res[kind]
    noise = sum(t.numel() * t.element_size() for t in r.slots[0].noise_stage)
    o = {"resident_items_per_s": summary([B / (ms * 1e-3) for ms in d["resident_ms_per_step"]]),
         "e2e_items_per_s": summary([B / (ms * 1e-3) for ms in d["e2e_ms_per_step"]]),
         "resident_ms_per_step": summary(d["resident_ms_per_step"]), "e2e_ms_per_step": summary(d["e2e_ms_per_step"]),
         "launches_per_step": r.launches_per_step(), "h2d_bytes_per_item": nbytes(host) / B, "noise_bytes_per_item": noise / B}
    if "set_vehicles_ms" in d:
        o["set_vehicles_ms"] = summary(d["set_vehicles_ms"])
        o["vehicle_bytes_per_set"] = nbytes(traj_vehicles)
    out[kind] = o

try:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip()
except Exception as ex:                                          # the reading is part of the result; say so when it is missing
    q = f"unavailable: {ex}"
line = {"metric": "trajectory items/s (warp + VUNet shape path per (vehicle, step) item)", "unit": "items/s",
        "items_per_step": B, "vehicles": V, "steps_per_vehicle": S, "steps": args.steps, "warmup": warm, "reps": args.reps,
        "gpu": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": q,
        "trajectory": out["trajectory"], "novel_view": out["novel_view"],
        "speedup_resident": out["trajectory"]["resident_items_per_s"]["median"] / out["novel_view"]["resident_items_per_s"]["median"],
        "speedup_e2e": out["trajectory"]["e2e_items_per_s"]["median"] / out["novel_view"]["e2e_items_per_s"]["median"],
        "note": "trajectory: appearance encoded once per vehicle (set_vehicles, outside the timed loops), decoded with the cached "
                "means as traj_test does; novel_view: NovelViewPipeline, a full forward per item (appearance re-encoded, sampled z)"}
print(json.dumps(line), flush=True)
