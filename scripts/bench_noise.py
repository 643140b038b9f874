#!/usr/bin/env python
"""Host vs device Sampler noise (pipeline noise="host" / "device") in both graph pipelines, in one process, run alternately.

Workload: B = 64 items per step (NovelViewPipeline: 64 crops, 10 draws, 1,310,720 normals; TrajectoryPipeline: 8 vehicles x
8 steps, 8 draws, 655,360 normals), synthetic 256x256 crops, random-init weights, pinned uint8 host inputs, as
scripts/bench_trajectory.py.  Per pipeline and noise mode:
  e2e_ms_per_step       end-to-end loop (H2D, replay, D2H; 3 slots on one stream), device events / host clock;
  resident_ms_per_step  graph replays only (2 slots): the step with the relayouts (host) or the generation branch (device);
  submit_cpu_ms         thread CPU time of the submitting thread per submit in the e2e loop (host mode: waiting for the
                        noise prefetch thread is not CPU time of this thread, the prefetch thread's is reported apart);
and the generation kernels alone (fusg_randn_mt19937 over the step's draws, NHWC), device events over many launches.

  python scripts/bench_noise.py [--steps 50] [--warmup 3] [--reps 3]

Prints one JSON line.  Writes nothing."""
import argparse
import collections
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from future_urban_scene_generation_b200 import noise, synth
from future_urban_scene_generation_b200.pipeline import NovelViewPipeline, TrajectoryPipeline, _GraphPipeline
from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=50, help="timed pipeline steps per loop")
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()

if not torch.cuda.is_available():
    raise SystemExit("bench_noise.py: no CUDA device; the B200 path has no CPU fallback")
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
V, S = 8, 8
B = V * S


def pinned(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


veh = np.repeat(np.arange(V), S).astype(np.int32)
wb = synth.make_warp_batch(0, B, crops=False)
src_v = np.stack([synth.make_crop(10_000 + v) for v in range(V)])
mk_v, ns_v, _ = synth.make_vunet_inputs_u8(10_000, V)
_, _, nd = synth.make_vunet_inputs_u8(0, B)
warp_in = {k: pinned(v) for k, v in wb.items()}
traj_vehicles = {"src": pinned(src_v), "x_mask_u8": pinned(mk_v), "x_normal_u8": pinned(ns_v)}
traj_host = dict(warp_in, vehicle=pinned(veh), y_normal_u8=pinned(nd))
nv_host = dict(warp_in, src=pinned(src_v[veh]), x_mask_u8=pinned(mk_v[veh]), x_normal_u8=pinned(ns_v[veh]), y_normal_u8=pinned(nd))

torch.manual_seed(0)
model = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).to(dev).eval()
model.engine()

# CPU time of the host-mode prefetch threads (they run torch.randn off the submitting thread)
_prefetch_cpu = [0.0]
_orig_draw = _GraphPipeline._draw_noise


def _counted_draw(self, slot, generator=None):
    t0 = time.thread_time()
    try:
        return _orig_draw(self, slot, generator)
    finally:
        if threading.current_thread() is not threading.main_thread():
            _prefetch_cpu[0] += time.thread_time() - t0


_GraphPipeline._draw_noise = _counted_draw


def run_steps(pipe, n, resident, host, cpu=None):
    pending, last = collections.deque(), None
    for _ in range(n):
        t0 = time.thread_time()
        last = pipe.submit(host, resident=resident)
        if cpu is not None:
            cpu.append(time.thread_time() - t0)
        pending.append(last)
        if len(pending) >= pipe.depth and not resident:
            pipe.result(pending.popleft())
    if resident:
        pipe.wait(last)
    else:
        while pending:
            pipe.result(pending.popleft())
    return last


def timed(pipe, n, resident, host, first_stream, last_stream_of, cpu=None):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(first_stream)
    last = run_steps(pipe, n, resident, host, cpu)
    e1.record(last_stream_of(last))
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    return max(e0.elapsed_time(e1), wall)


def make(kind, depth, mode, **kw):
    if kind == "trajectory":
        p = TrajectoryPipeline(model, max_vehicles=V, depth=depth, noise=mode, **kw)
        p.set_vehicles(traj_vehicles)
        return p, traj_host
    return NovelViewPipeline(model, depth=depth, noise=mode, **kw), nv_host


warm = max(3, args.warmup)
pipes = {}
for kind in ("novel_view", "trajectory"):
    for mode in ("host", "device"):
        r, host = make(kind, 2, mode)
        run_steps(r, warm, False, host)
        e, _ = make(kind, 3, mode, shared_stream=True)
        run_steps(e, max(2, warm), False, host)
        pipes[(kind, mode)] = (r, e, host)

res = {k: collections.defaultdict(list) for k in pipes}
for rep in range(args.reps):
    for key, (r, e, host) in pipes.items():                      # alternate all four inside every repetition
        ms = timed(r, args.steps, True, host, r.slots[r.n % r.depth].stream, lambda t, r=r: r.slots[t % r.depth].stream)
        res[key]["resident_ms_per_step"].append(ms / args.steps)
        cpu = []
        _prefetch_cpu[0] = 0.0
        ms = timed(e, args.steps, False, host, e.copy_stream, lambda t, e=e: e.out_stream, cpu)
        res[key]["e2e_ms_per_step"].append(ms / args.steps)
        res[key]["submit_cpu_ms"].append(1e3 * sum(cpu) / len(cpu))
        res[key]["prefetch_thread_cpu_ms_per_step"].append(1e3 * _prefetch_cpu[0] / args.steps)

# the generation kernels alone, on the step's draws (NHWC), device events over many launches
gen = {}
for kind, shapes in (("novel_view", [(B, 128, 4, 4), (B, 128, 8, 8)] + [(B, 128, 2, 2)] * 4 + [(B, 128, 4, 4)] * 4),
                     ("trajectory", [(B, 128, 2, 2)] * 4 + [(B, 128, 4, 4)] * 4)):
    outs = [torch.empty((b, h, w, c), dtype=torch.float32, device=dev) for b, c, h, w in shapes]
    plan = noise.DrawPlan(outs, shapes, True, dev)
    g = torch.Generator()
    g.manual_seed(1)
    plan.take(g)
    plan.upload()
    for _ in range(5):
        plan.launch()
    n = 200
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        plan.launch()
    e1.record()
    torch.cuda.synchronize()
    t0 = time.thread_time()
    for _ in range(n):
        plan.take(g)
    host_take = (time.thread_time() - t0) / n * 1e3
    t0 = time.thread_time()
    for s in shapes:
        torch.randn(*s, generator=g)
    host_randn = (time.thread_time() - t0) * 1e3
    gen[kind] = {"normals": plan.words, "kernel_ms": e0.elapsed_time(e1) / n, "host_take_cpu_ms": host_take,
                 "host_torch_randn_cpu_ms": host_randn}


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


out = {}
for (kind, mode), (r, e, host) in pipes.items():
    d = res[(kind, mode)]
    out.setdefault(kind, {})[mode] = {k: summary(v) for k, v in d.items()}
    out[kind][mode]["launches_per_step"] = r.launches_per_step()
for kind in out:
    out[kind]["generation"] = gen[kind]
    out[kind]["e2e_speedup_device_over_host"] = (out[kind]["host"]["e2e_ms_per_step"]["median"] /
                                                 out[kind]["device"]["e2e_ms_per_step"]["median"])
    out[kind]["resident_step_delta_ms_device_minus_host"] = (out[kind]["device"]["resident_ms_per_step"]["median"] -
                                                            out[kind]["host"]["resident_ms_per_step"]["median"])

try:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip()
except Exception as ex:
    q = f"unavailable: {ex}"
line = {"metric": "Sampler noise: host torch.randn vs device generation, B = 64 per step", "unit": "ms",
        "items_per_step": B, "steps": args.steps, "warmup": warm, "reps": args.reps,
        "gpu": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": q,
        "cpu_capability": torch.backends.cpu.get_cpu_capability(), **out}
print(json.dumps(line), flush=True)
