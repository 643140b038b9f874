#!/usr/bin/env python
"""bench.py -- novel-view completion (fused planar warp + VUNet bf16 forward) throughput on B200.

Metric (BASELINE.json): vehicle crops/s through warp + VUNet at N GPUs, plus the roofline fraction of
the dominant kernel, next to the reference algorithm's CPU path timed on this box's host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (one rank per GPU under torchrun)
  python bench.py ... --dump-outputs DIR                         also write the last timed step's outputs to DIR/*.npy
  python bench.py --impl reference ...                           CPU arm: the oracle port of the reference path

One "step" = one pass of the hot path over one batch of synthetic crops (BASELINE config 2: 64 crops
per GPU; at 8 GPUs BASELINE config 4: 4096 crops = 512 per rank in 8 micro-batches of 64):
fusg_warp_fused, Vunet_fix_res.forward, to_image, and -- when N > 1 -- ONE NCCL all-gather of the
step's completed uint8 crops (the only collective; crops are sharded contiguously by rank, weak
scaling).  Prints ONE JSON line on rank 0.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vehicle crops/s novel-view completion (warp+VUNet)"
UNIT = "crops/s"
WARP_BYTES_PER_CROP = 256 * 256 * 3 * 6            # read the crop once + write 5 planes (SURVEY.md §8d)
VUNET_FLOPS_PER_CROP = 76_271_321_088              # 112 convs, 2*MACs (SURVEY.md §8d)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median over the busy samples (idle samples before the first launch sit at low clocks)
        busy = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path (test infrastructure used as the timed baseline)
# ------------------------------------------------------------------------------------------------
def _cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _import_reference():
    """The reference's own modules, when its tree is reachable (the build container has /root/reference; the GPU box
    does not -- reference sources are never copied into this repo).  Returns None when it is not importable."""
    for root in ("/root/reference", os.path.join(ROOT, "baseline", "_ref")):
        if os.path.isdir(os.path.join(root, "warp_learn")) and os.path.isdir(os.path.join(root, "vunet")):
            os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
            if root not in sys.path:
                sys.path.append(root)
            try:
                import warnings
                warnings.simplefilter("ignore")
                from warp_learn.online_visibility import compute_visibility, pascal_texture_planes
                from warp_learn.planes_utils import get_planes, warp_unwarp_planes
                from vunet.models import Vunet_fix_res
                return {"root": root, "compute_visibility": compute_visibility, "pascal_texture_planes": pascal_texture_planes,
                        "get_planes": get_planes, "warp_unwarp_planes": warp_unwarp_planes, "Vunet_fix_res": Vunet_fix_res}
            except Exception:
                return None
    return None


def cpu_reference_run(steps, warmup, crops_per_step=1):
    """Times the reference's CPU path on BASELINE config 1 (batch 1, --device cpu), all host threads.
    kind "reference": the reference's own modules (compute_visibility x2 + get_planes x2 + warp_unwarp_planes through
    cv2, Vunet_fix_res.forward through torch) when its tree is importable; kind "port" otherwise: oracle/warp_oracle.c
    (scalar C, 1 thread) + oracle/vunet_oracle.py (torch fp32, all host threads)."""
    import numpy as np
    import torch
    from future_urban_scene_generation_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = _import_reference()
    if ref is not None:
        from argparse import Namespace
        import cv2
        torch.manual_seed(0)
        net = ref["Vunet_fix_res"](Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).eval()
        kind, cv_threads = "reference", cv2.getNumThreads()
    else:
        from oracle import warp_oracle as WO, vunet_oracle as VO
        sd = VO.make_state_dict(0)
        kind, cv_threads = "port", None
    t_warp, t_vunet = [], []
    for s in range(warmup + steps):
        tw = tv = 0.0
        for c in range(crops_per_step):
            idx = s * crops_per_step + c
            p = synth.make_pose_pair(idx)
            img = synth.make_crop(idx)
            x, y = synth.make_vunet_inputs(idx, 1)
            x, y = torch.from_numpy(x), torch.from_numpy(y)
            t0 = time.perf_counter()
            if ref is not None:
                kp3d = {k: p["kp3d"][i] for i, k in enumerate(synth.KP_NAMES)}
                ks = {k: p["kp2d_src"][i] for i, k in enumerate(synth.KP_NAMES)}
                kd = {k: p["kp2d_dst"][i] for i, k in enumerate(synth.KP_NAMES)}
                vs = ref["compute_visibility"](p["E_src"], p["K"], kp3d, 256, 256)
                vd = ref["compute_visibility"](p["E_dst"], p["K"], kp3d, 256, 256)
                sp, skp, sv = ref["get_planes"](img, ks, 'car', vs)
                dp, dkp, dv = ref["get_planes"](img, kd, 'car', vd)
                ref["warp_unwarp_planes"](sp, skp, dkp, sv, dv, 'car', ref["pascal_texture_planes"])
            else:
                WO.warp_fused(img, p["src_kp"], p["dst_kp"], p["K"], p["E_src"], p["E_dst"], p["kp3d"])
            t1 = time.perf_counter()
            with torch.no_grad():
                if ref is not None:
                    net(y, x)
                else:
                    VO.forward(sd, y, x)
            t2 = time.perf_counter()
            tw += t1 - t0
            tv += t2 - t1
        if s >= warmup:
            t_warp.append(tw)
            t_vunet.append(tv)
    total = sum(t_warp) + sum(t_vunet)
    n = steps * crops_per_step
    if ref is not None:
        how = (f"the reference's own modules ({ref['root']}): cv2 warp half {1e3 * sum(t_warp) / n:.1f} ms/crop (cv2 threads {cv_threads}) + "
               f"Vunet_fix_res.forward fp32 {sum(t_vunet) / n:.3f} s/crop (torch threads {torch.get_num_threads()})")
    else:
        how = (f"C oracle warp {1e3 * sum(t_warp) / n:.1f} ms/crop (1 thread) + torch fp32 VUNet oracle {sum(t_vunet) / n:.3f} s/crop "
               f"({torch.get_num_threads()} threads); reference tree not present on this box")
    return {"value": n / total, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{n} crops, batch 1 (BASELINE config 1): {how}; os.cpu_count()={cores}, CPU {_cpu_model()}",
            "ms_per_step": 1e3 * total / steps}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, max(1, args.warmup))
    line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": "1 synthetic 256x256 vehicle crop per step: warp (visibility x2, homographies, masked warp) + VUNet fp32 forward, CPU"},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def pin_to_gpu_numa(torch, rank, world):
    """Binds this rank's threads (main, noise prefetch, torch intra-op) to its share of the CPUs of the NUMA node its
    GPU hangs off, BEFORE any pinned staging buffer is allocated (first touch puts the pages on that node).  Without this
    eight ranks each start os.cpu_count() intra-op threads for the Sampler noise and trample each other."""
    def gpu_node(i):
        try:
            pr = torch.cuda.get_device_properties(i)
            bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            return int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        except Exception:
            return -1

    def cpulist(node):
        try:
            txt = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
            out = []
            for part in txt.split(","):
                lo, _, hi = part.partition("-")
                out.extend(range(int(lo), int(hi or lo) + 1))
            return out
        except Exception:
            return []
    try:
        allowed = sorted(os.sched_getaffinity(0))
        nodes = [gpu_node(i) for i in range(world)]
        mine = nodes[rank]
        pool = [c for c in cpulist(mine) if c in allowed] if mine >= 0 else []
        peers = [r for r in range(world) if nodes[r] == mine] if pool else list(range(world))
        if not pool:
            pool = allowed
        k = peers.index(rank)
        share = pool[k * len(pool) // len(peers):(k + 1) * len(pool) // len(peers)] or pool
        os.sched_setaffinity(0, share)
        torch.set_num_threads(max(1, min(len(share), 8)))
        return {"numa_node": mine, "cpus": len(share), "torch_threads": torch.get_num_threads()}
    except Exception as exc:                                  # affinity is an optimisation, never a reason to fail
        return {"numa_node": None, "error": str(exc)[:80]}


def run_ours(args):
    from argparse import Namespace
    import numpy as np
    import torch
    import torch.distributed as dist
    from future_urban_scene_generation_b200 import synth, _lib
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200.parallel import shard_range, gather_crops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity = pin_to_gpu_numa(torch, local_rank, world)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version/info lines must not land on stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)
    # BASELINE config 2: 64 crops per GPU per step; config 4 (8 GPUs): 4096 crops per step = 512 per rank, processed as
    # 8 micro-batches of 64 (the same kernels, graphs and per-GPU work per crop as every other N -> weak scaling holds)
    # with ONE all-gather of the 805 MB of completed crops per step.
    B = args.micro_batch
    CPR = args.crops_per_rank if args.crops_per_rank else (512 if world == 8 else 64)
    if CPR % B:
        raise SystemExit("--crops-per-rank must be a multiple of --micro-batch")
    M = CPR // B
    peaks = _peaks()

    # ---- model: random-init weights of the reference architecture (checkpoints are not available offline)
    torch.manual_seed(0)
    model = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).to(dev).eval()
    eng = model.engine()

    # ---- synthetic inputs for this rank's contiguous shard of crops (SURVEY.md §8d generators), one dict per micro-batch
    first, last = shard_range(world * CPR, rank, world)
    assert last - first == CPR

    def pinned(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    host_u8, host_f32 = [], []
    for mb in range(M):
        f0 = first + mb * B
        wb = {k: pinned(v) for k, v in synth.make_warp_batch(f0, B).items()}
        mk, nsrc, ndst = synth.make_vunet_inputs_u8(f0, B)
        # the form the reference holds before to_tensor (trajectory_inference.py:215-220): three uint8 images per crop
        host_u8.append(dict(wb, x_mask_u8=pinned(mk), x_normal_u8=pinned(nsrc), y_normal_u8=pinned(ndst)))
        if M == 1:
            xs, ys = synth.make_vunet_inputs(f0, B)
            host_f32.append(dict(wb, x=pinned(xs), y=pinned(ys)))
    h2d_bytes_u8 = M * sum(v.numel() * v.element_size() for v in host_u8[0].values())

    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    gather = (lambda c: gather_crops(c, world * CPR)) if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def reduce_max(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def run_steps(pipe, n, resident, host):
        """n steps of M micro-batches.  depth-1 submits stay in flight behind the one being issued; in the end-to-end
        form every micro-batch's outputs are read on the host."""
        pending, last = collections.deque(), None
        for _ in range(n):
            for mb in range(M):
                last = pipe.submit(host[mb], resident=resident)
                pending.append(last)
                if len(pending) >= pipe.depth and not resident:
                    pipe.result(pending.popleft())         # an earlier micro-batch's outputs are on the host
        if resident:
            pipe.wait(last)
        else:
            while pending:
                pipe.result(pending.popleft())
        if gather is not None:
            pipe.wait_gather()                             # the last step's all-gather belongs to the timed region
        return last

    def timed(pipe, n, resident, host, first_stream, last_stream_of):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(first_stream)
        last_t = run_steps(pipe, n, resident, host)
        e1.record(last_stream_of(last_t))
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        # several streams are in flight: bracket with device events and cross-check with the host clock
        ms = reduce_max(max(e0.elapsed_time(e1), wall if (n * M >= 20 or not resident) else 0.0))
        barrier()
        return ms, last_t

    # ---- device-resident loop: inputs and noise already in HBM, graph replays only ----------------
    # The public batched API: NovelViewPipeline (CUDA-graph replay of the launches of a micro-batch, two in flight).
    pipe = NovelViewPipeline(model, depth=2, gather_fn=gather, micro_batches_per_step=M)
    torch.manual_seed(1)
    warm = max(3, args.warmup)
    last_ticket = run_steps(pipe, max(warm, (3 + M - 1) // M), resident=False, host=host_u8)
    launches_per_mb = pipe.launches_per_step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, last_ticket = timed(pipe, args.steps, True, host_u8, pipe.slots[pipe.n % pipe.depth].stream, lambda t: pipe.slots[t % pipe.depth].stream)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pipe, last_ticket, min(M, pipe.depth))
    launches = launches_per_mb * M * args.steps
    ms_per_step = ms_total / args.steps
    value = world * CPR / (ms_per_step * 1e-3)
    del pipe

    # ---- end-to-end loop (the headline): every micro-batch copies its own pinned uint8 inputs H2D, draws the Sampler
    # noise on the CPU generator (reference semantics), and lands its completed crops + flags in host memory, inside
    # the timed region.  One compute stream shared by the slots: with host copies in the loop, graphs that overlap only
    # partially slow each other down (measured 11.8 vs 14.2 ms/step, scripts/e2e_probe.py).
    e2e_steps = args.steps

    def e2e_run(host, **kw):
        pp = NovelViewPipeline(model, depth=3, shared_stream=True, gather_fn=gather, micro_batches_per_step=M, **kw)
        lt = run_steps(pp, max(2, (5 + M - 1) // M), resident=False, host=host)
        d2h = M * pp.d2h_bytes(lt)
        ms, _ = timed(pp, e2e_steps, False, host, pp.copy_stream, lambda t: pp.out_stream)
        return world * CPR / (ms / e2e_steps * 1e-3), ms / e2e_steps, d2h
    e2e_value, e2e_ms_step, d2h_bytes = e2e_run(host_u8)
    extra = {}
    if M == 1 and not args.headline_only:
        # the same loop with the warped planes also copied back to the host (round-1 contract) ...
        v, ms, d2h = e2e_run(host_u8, return_warped=True)
        extra["e2e_u8_with_planes"] = {"value": v, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes_u8, "d2h_bytes_per_step": d2h, "ms_per_step": ms,
                                       "note": "as e2e, plus the (B,5,256,256,3) warped planes D2H (the reference never reads them on the host)"}
        # ... and with the VUNet inputs shipped as fp32 NCHW tensors (36 instead of 9 bytes per pixel)
        v, ms, d2h = e2e_run(host_f32, return_warped=True)
        extra["e2e_fp32"] = {"value": v, "unit": UNIT, "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host_f32[0].values()),
                             "d2h_bytes_per_step": d2h, "ms_per_step": ms,
                             "note": "round-1 headline form: x / y_tilde as fp32 NCHW host tensors, warped planes copied back"}

    # ---- per-launch roofline pass (CUDA events around every conv launch, on the launching stream)
    roof = warp_roof = None
    if rank == 0:
        xs, ys = synth.make_vunet_inputs(first, B)
        devin = {k: v.to(dev) for k, v in host_u8[0].items()}
        devin["x"], devin["y"] = torch.from_numpy(xs).to(dev), torch.from_numpy(ys).to(dev)
        noise_bank = {}

        def staged_noise(b, c, h, w):
            key = (b, c, h, w, staged_noise.i)
            staged_noise.i += 1
            if key not in noise_bank:
                noise_bank[key] = torch.randn((b, h, w, c), device=dev)
            return noise_bank[key]
        staged_noise.i = 0
        eng.noise_provider = staged_noise
        eng.profile = []
        model.fork_branches = False            # per-launch timing: one stream, no kernel overlaps another
        for _ in range(2):
            staged_noise.i = 0
            # park the stream behind a ~40 ms spin so the host enqueues the whole forward ahead of the GPU: the event
            # pairs then bracket kernel time, not host launch gaps (the narrow layers run 10-20 us, a launch costs ~15)
            torch.cuda._sleep(int(0.040 * 1.9e9))
            model(devin["y"], devin["x"])
        torch.cuda.synchronize()
        model.fork_branches = True
        recs = eng.profile
        eng.profile = None
        eng.noise_provider = None
        agg = {}
        for path, impl, flops, e0, e1 in recs:
            a = agg.setdefault(impl, [0.0, 0.0, 0])
            a[0] += flops
            a[1] += e0.elapsed_time(e1) * 1e-3
            a[2] += 1
        # every convolution launch of the forward counts (the 110 tcgen05 launches AND the two streaming first-layer NiNs,
        # impl 3, which hold 0.15 % of the FLOPs): FLOP-weighted over all 112 convs, the conservative reading
        tc = [sum(a[0] for a in agg.values()), sum(a[1] for a in agg.values()), sum(a[2] for a in agg.values())]
        tc_only = agg.get(1, [0.0, 1e-9, 0])
        achieved = tc[0] / tc[1] / 1e12
        peak = peaks["bf16_tflops_sustained"]
        traffic, traffic_src = None, None
        for name in ("r2_conv_traffic_summary.json", "r1_conv_traffic_summary.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath) and B == 64:
                tj = json.load(open(tpath))
                traffic, traffic_src = tj["avg_traffic_bytes_per_launch"], tj["source"]
                break
        roof = {"bound": "tensor", "kernel": "k_conv_tc (tcgen05 implicit-GEMM conv; all 112 conv launches of a forward are summed)", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "k_conv_tc_only": {"achieved": tc_only[0] / tc_only[1] / 1e12, "frac": tc_only[0] / tc_only[1] / 1e12 / peak, "launches_per_step": tc_only[2] // 2},
                "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes per launch (dram read+write, ncu; B=64)", "traffic_source": traffic_src, "peak_source": peaks["source"] + ", sustained bf16",
                "launches_per_step": tc[2] // 2, "avg_launch_ms": 1e3 * tc[1] / max(1, tc[2]),
                "algorithmic_flops_per_step": tc[0] / 2, "share_of_vunet_time": tc[1] / max(1e-9, sum(a[1] for a in agg.values()))}
        # fused warp path alone (HBM bound) at this micro-batch ...
        wk = ("src", "src_kp", "dst_kp", "K", "E_src", "E_dst", "kp3d")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            warp_batch(*(devin[k] for k in wk), device=dev)
        reps = 20
        e0.record()
        for _ in range(reps):
            warp_batch(*(devin[k] for k in wk), device=dev)
        e1.record()
        torch.cuda.synchronize()
        wsec = e0.elapsed_time(e1) * 1e-3 / reps
        wgbs = B * WARP_BYTES_PER_CROP / wsec / 1e9
        wtraffic = None
        wt = os.path.join(ROOT, "profiles", "r2_warp_traffic_summary.json")
        if os.path.exists(wt):
            wtraffic = json.load(open(wt))
        warp_roof = {"bound": "hbm", "kernel": "fusg_warp_fused", "achieved": wgbs, "peak": peaks["hbm_gbs"],
                     "unit": "GB/s", "frac": wgbs / peaks["hbm_gbs"], "crops": B, "ms": wsec * 1e3, "traffic": wtraffic,
                     "note": f"{B} crops only ({B * WARP_BYTES_PER_CROP / 1e6:.0f} MB < L2, latency-bound); see large_batch"}
        # ... and at an HBM-sized batch: this rank's crops tiled to 4096 (4.8 GB of algorithmic traffic);
        # BASELINE config 3 proper (16k crops) is scripts/bench_warp.py
        try:
            BL = 4096
            rep = (BL + B - 1) // B
            big = {k: devin[k].repeat((rep,) + (1,) * (devin[k].dim() - 1))[:BL].contiguous() for k in wk}
            for _ in range(2):
                rb = warp_batch(*(big[k] for k in wk), device=dev)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                rb = warp_batch(*(big[k] for k in wk), device=dev)
            e1.record()
            torch.cuda.synchronize()
            bsec = e0.elapsed_time(e1) * 1e-3 / 3
            bgbs = BL * WARP_BYTES_PER_CROP / bsec / 1e9
            warp_roof["large_batch"] = {"crops": BL, "ms": bsec * 1e3, "achieved": bgbs, "unit": "GB/s", "frac": bgbs / peaks["hbm_gbs"]}
            del big, rb
            torch.cuda.empty_cache()
            # 5/6 of this path's algorithmic bytes are writes and a pure write stream does not reach the copy bandwidth:
            # measured on the spot for the record (torch fill_ of 1 GiB); `frac` above stays against the copy peak
            probe = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
            probe.fill_(0)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                probe.fill_(0)
            e1.record()
            torch.cuda.synchronize()
            warp_roof["write_stream_GBps"] = probe.numel() * 5 / (e0.elapsed_time(e1) * 1e-3) / 1e9
            del probe
            torch.cuda.empty_cache()
        except RuntimeError as exc:                       # e.g. not enough free memory: report, do not fail the bench
            warp_roof["large_batch"] = {"skipped": str(exc)[:120]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))          # the CPU arm gets every host core
        except Exception:
            pass
        cpu = cpu_reference_run(steps=8, warmup=1)
        cpu.pop("ms_per_step", None)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"{CPR} synthetic 256x256 vehicle crops per GPU per step" + (f" in {M} micro-batches of {B}" if M > 1 else "") +
                                   ": fused planar warp (5 CAD planes) + VUNet bf16 forward, random-init weights (BASELINE config " +
                                   ("4: 4096 crops per step, 512 per rank" if world * CPR == 4096 else "2") + ")" +
                                   (", one NCCL all-gather of the completed uint8 crops per step" if world > 1 else ""),
                       "crops_per_gpu": CPR, "micro_batch": B, "global_crops_per_step": world * CPR, "parallelism": f"crop-sharded dp{world}",
                       "gathered_bytes_per_step": world * CPR * 256 * 256 * 3 if world > 1 else 0,
                       "l2": "per-micro-batch activations (>5 GB) exceed the 126 MB L2; no explicit flush",
                       "launch": "one CUDA-graph replay per micro-batch (gpu_launches counts the kernels inside the graphs)" +
                                 (" + one NCCL all-gather per step on its own stream, overlapping the next step" if world > 1 else ""),
                       "host_affinity": affinity},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes_u8, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms_step, "steps": e2e_steps,
                    "note": "NovelViewPipeline.submit/result: pinned host inputs in the form the reference holds them before to_tensor "
                            "(uint8 crop + three uint8 sketch images, trajectory_inference.py:215-220) -> H2D, to_tensor/flip/concat on the "
                            "device, Sampler noise drawn on the CPU generator (reference semantics), CUDA-graph replay, completed uint8 crops "
                            "+ plane_j + visibility flags D2H; 3 slots in flight, all inside the timed region.  The warped planes stay in HBM "
                            "(they feed get_icn_inputs on the device); e2e_u8_with_planes / e2e_fp32 time the round-1 forms"},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
            "roofline_warp": warp_roof,
            "vunet_tflops_whole_forward": world * CPR * VUNET_FLOPS_PER_CROP / (ms_per_step * 1e-3) / 1e12,
            "cpu_baseline": cpu,
        }
        line.update(extra)
        if world == 1 and not args.no_icn and not args.headline_only:
            line["icn_generator"] = icn_info(torch, synth, B, dev)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, pipe, last_ticket, n_tickets):
    """Writes what the timed loop computed in its last step -- the device outputs of its last `n_tickets` submits (all a
    pipeline of that depth still holds), crop axis first, concatenated in submit order -- as <out_dir>/<name>.npy, float32
    (float64 where float32 would not be exact).  Together they stay under DUMP_BYTES: smallest first, an array larger than
    an equal share of what is left keeps only a sample of its crops, the first k of a permutation seeded with 0, in crop
    order -- the same crops on every run, so two builds can be compared output for output."""
    import numpy as np
    import torch
    outs = [pipe.device_outputs(t) for t in range(last_ticket - n_tickets + 1, last_ticket + 1)]
    arrays = {}
    for k, v in outs[-1].items():
        v = v if k == "crops_all" else torch.cat([o[k] for o in outs])      # crops_all: the whole step, all ranks
        wide = v.dtype in (torch.float64, torch.int32, torch.int64)
        arrays[k] = v.to(torch.float64 if wide else torch.float32).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES - 4096 * len(arrays)                                    # room for the .npy headers
    for i, (k, a) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].nbytes)):
        share = left // (len(arrays) - i)
        if a.nbytes > share:
            keep = max(1, share // (a.nbytes // a.shape[0]))
            a = a[np.sort(np.random.default_rng(0).permutation(a.shape[0])[:keep])]
        np.save(os.path.join(out_dir, f"{k}.npy"), a)
        left -= a.nbytes


def icn_info(torch, synth, B, dev):
    """Informational, outside every timed region of the headline metric: the ICN generator G_Resnet (SURVEY.md 8f-1, the consumer of
    the warped planes in the reference's data flow) on the same batch size -- crops/s and FLOP-weighted tensor throughput."""
    try:
        from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
        torch.manual_seed(0)
        g = G_Resnet(21).to(dev).eval()
        xi = torch.from_numpy(synth.make_icn_inputs(0, min(B, 8), 256)).to(dev)
        xi = xi.repeat((B + xi.shape[0] - 1) // xi.shape[0], 1, 1, 1)[:B].contiguous()
        for _ in range(3):
            g(xi)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            g(xi)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        flops = 130124087296.0                       # per 256x256 crop, 18 convolutions (oracle/icn_oracle.py: flops_per_crop)
        return {"crops_per_s": B / ms * 1e3, "ms_per_forward": ms, "crops": B, "tflops_whole_forward": B * flops / (ms * 1e-3) / 1e12,
                "dtype": "fp16 operands, fp32 accumulate", "note": "not part of `value`; details in profiles/r1_icn_bench.json"}
    except Exception as ex:                          # never let the informational block take the bench line down
        return {"error": f"{type(ex).__name__}: {ex}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--crops-per-rank", type=int, default=0, help="crops per GPU per step (default: 512 at 8 GPUs = BASELINE config 4, else 64)")
    ap.add_argument("--micro-batch", type=int, default=64, help="crops per graph replay (BASELINE config 2 batch)")
    ap.add_argument("--headline-only", action="store_true", help="skip the informational extra keys (e2e_fp32, ICN)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-icn", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl ours)")
    # stdout carries exactly one JSON line: libraries that write to fd 1 on their own (NCCL prints its version there
    # whatever NCCL_DEBUG_FILE says) are pointed at stderr for the whole run, and print() gets the real stdout back
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    real_stdout.flush()


if __name__ == "__main__":
    main()
