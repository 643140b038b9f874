"""Batched, software-pipelined front end of the hot path: host buffers in, host buffers out.

`NovelViewPipeline.submit(batch)` enqueues, for one batch of crops,
    H2D of the pinned inputs (copy stream)  ->  fused planar warp + VUNet forward + to_image
    (compute stream)  ->  D2H of the completed uint8 crops and warped planes (output stream)
and returns immediately; `result(ticket)` blocks until that batch's outputs are in host memory.
With `depth` batches in flight the copies of batch n+1 overlap the kernels of batch n.  Each item is
one full reference forward (`Vunet_fix_res.forward`: appearance encoded per item, decoded with the
sampled z).

`TrajectoryPipeline` is the form of the trajectory loop (traj_test, trajectory_inference.py:230-233,
:413-426): the appearance of each vehicle is encoded once (`set_vehicles`) and each submitted
(vehicle, step) item runs only the shape path, decoded with the vehicle's cached means -- the
reference's results at a quarter of the convolution work.

The ~125 kernel launches of one step are captured once per slot into a CUDA graph (static device
buffers) and replayed, so the host issues one launch per step instead of ~125.  Sampler noise is
drawn from the CPU default generator in the reference's order and shapes (vunet/layers.py:166) --
`torch.manual_seed` reproduces the reference's outputs.  With noise="host" (the default) torch.randn draws it on
the host and it is copied into the graph's static noise buffers before each replay; with noise="device" the graph
itself generates the same numbers from the generator's 2.5 KB start state (noise.py, csrc/noise.cu).
"""
import contextlib
import threading

import torch

from . import _lib
from . import noise as device_noise
from .frame_ops import gather_rows, u8_to_vunet_inputs, u8_to_vunet_y
from .warp_learn.batch import warp_batch
from .warp_learn.planes_utils import to_image_batch


class _Slot:
    """Static buffers + captured graph of one in-flight batch."""

    def __init__(self):
        self.graph = None
        self.inp = None          # device input buffers (static)
        self.noise = []          # device noise buffers in draw order, NHWC fp32 (what the Sampler epilogues read)
        self.noise_nchw = []     # device copies of the staging buffers, NCHW as drawn; re-laid out to `noise` inside the graph
        self.noise_shapes = []   # (B,C,H,W) per draw
        self.noise_stage = []    # pinned NCHW staging buffers (one per draw): torch.randn writes straight into them
        self.draws = None        # noise="device": the DrawPlan that generates `noise` inside the graph (no staging, no relayout)
        self.dev_out = None      # device outputs (static)
        self.out = None          # pinned host outputs
        self.done = None
        self.copied = None       # event: this slot's last H2D (inputs + noise) has been consumed from the pinned buffers
        self.launches = 0
        self.stream = None       # this slot's compute stream: the small-grid tail layers of one batch overlap the
                                 # full-grid layers of the next batch in flight
        self.prefetch = None     # (thread, state_before, result holder) of a background noise draw into noise_stage
        self.crops_all = None    # multi-GPU: the all-gathered completed crops of the last step, on the device
        self.wkey = None         # the engine's folded-weight key the graph was captured against


class _GraphPipeline:
    """What NovelViewPipeline and TrajectoryPipeline share: slots of static buffers with one captured graph each, the copy /
    compute / output streams, the background Sampler-noise draw, the side-stream warp branch and the multi-GPU exchange.
    A subclass supplies the two branches of one step on the slot's input buffers: `_warp(inp)` returns the WarpResult,
    `_decode(inp)` the VUNet output x_tilde."""

    def __init__(self, model, depth: int = 2, gather_fn=None, shared_stream: bool = False,
                 prefetch_noise: bool = True, return_warped: bool = False, micro_batches_per_step: int = 1,
                 noise: str = "host"):
        """noise: where the Sampler noise is made.  "host": torch.randn on the CPU generator, drawn ahead on a worker
        thread, uploaded and re-laid out to NHWC in the graph.  "device": the same numbers, bit for bit, generated inside
        the captured graph (noise.py); a submit only reads the CPU generator's state and advances it past the step's draws.
        Both leave the CPU generator in the same state and give the same outputs.
        return_warped: also copy the (B,5,256,256,3) warped planes back to the host (63 of 75 MB per 64 crops).  The
        reference never reads the planes on the host for their own sake -- they feed get_icn_inputs
        (trajectory_inference.py:175-182), which runs on the device here -- so the default keeps them in HBM
        (`device_outputs(ticket)["warped"]`).
        micro_batches_per_step: a step of the data-parallel job is M consecutive submits (BASELINE config 4: 512 crops per
        rank = 8 micro-batches of 64); the completed crops of a step are collected in one device buffer and `gather_fn`
        runs ONCE per step on it, on its own stream, overlapping the next step's kernels."""
        _lib.require_cuda()
        if noise not in ("host", "device"):
            raise ValueError(f"noise must be 'host' or 'device', got {noise!r}")
        self.model = model
        self.dev = next(model.parameters()).device
        self.depth = depth
        self.gather_fn = gather_fn        # optional device-side collective on the completed crops (parallel.gather_crops)
        self.prefetch_noise = prefetch_noise
        self.return_warped = return_warped
        self.mps = max(1, int(micro_batches_per_step))
        self.step_bufs = None             # two (M*B,256,256,3) u8 device buffers: the step being filled / being gathered
        self.comm_stream = torch.cuda.Stream(self.dev)
        self.gather_done = [None, None]   # event per step buffer: its all-gather has finished reading it
        self.crops_all = None             # the last all-gathered step, on the device (global crop order)
        self.copy_stream = torch.cuda.Stream(self.dev)
        self.out_stream = torch.cuda.Stream(self.dev)
        self.side_stream = torch.cuda.Stream(self.dev)
        self.noise = noise
        if noise == "device":
            device_noise.ensure_checked(self.dev)      # raises rather than give other numbers than torch.randn
            self.noise_stream = torch.cuda.Stream(self.dev)
        self.slots = [_Slot() for _ in range(depth)]
        one = torch.cuda.Stream(self.dev)
        for sl in self.slots:
            sl.stream = one if shared_stream else torch.cuda.Stream(self.dev)
        self.n = 0
        self.captures = 0                 # graphs captured so far (one per slot; again after a weight reload or a shape change)

    # ------------------------------------------------------------------ one step of device work
    #: SMs the persistent conv grids leave to the warp stage's solver warps while both run in one step (a persistent CTA
    #: that cannot be placed doubles its layer's time; measured 8.50 -> 8.15 ms per 64-crop step, profiles/r2_summary.md)
    SM_RESERVE = 4

    def _compute(self, inp):
        prev = _lib.lib().fusg_conv2d_set_sm_reserve(self.SM_RESERVE)      # baked into the captured launches' grids
        try:
            # the planar warp is a chain of small latency-bound kernels (visibility -> homographies -> gather) that does
            # not feed the VUNet of the same batch: fork it onto a side stream so it fills the SMs the narrow VUNet
            # layers leave idle, and join before the outputs are read (inside a graph this becomes a parallel branch)
            cur = torch.cuda.current_stream(self.dev)
            self.side_stream.wait_stream(cur)
            with torch.cuda.stream(self.side_stream):
                res = self._warp(inp)
            with torch.no_grad(), torch.cuda.device(self.dev):
                x_tilde = self._decode(inp)
            crops = to_image_batch(x_tilde)
            cur.wait_stream(self.side_stream)
            for t in (res.warped, res.plane_j, res.vis):
                t.record_stream(cur)
            return {"crops": crops, "warped": res.warped, "plane_j": res.plane_j, "vis": res.vis}
        finally:
            _lib.lib().fusg_conv2d_set_sm_reserve(prev)

    def _graph_key(self, eng):
        """What a captured graph depends on besides its input shapes: the device pointers of the folded weights."""
        return eng._wkey

    def _prepare_slot(self, slot: _Slot, batch: dict):
        """First use of a slot: allocate static buffers, run once eagerly (weight fold, function
        attributes, allocator warm-up), then capture the step into a graph."""
        eng = self.model.engine()
        slot.wkey = None                      # until the capture below succeeds: a failed preparation is redone next time
        slot.inp = {k: torch.empty(tuple(v.shape), dtype=v.dtype, device=self.dev) for k, v in batch.items()}
        for k, v in batch.items():
            slot.inp[k].copy_(v)
        shapes = []

        def recording_provider(b, c, h, w):
            shapes.append((b, c, h, w))
            return torch.zeros((b, h, w, c), dtype=torch.float32, device=self.dev)
        with eng.noise_from(recording_provider), torch.cuda.stream(slot.stream):
            self._compute(slot.inp)                                   # eager warm-up
        slot.stream.synchronize()
        slot.noise_shapes = list(shapes)
        slot.noise = [torch.zeros((b, h, w, c), dtype=torch.float32, device=self.dev) for b, c, h, w in shapes]
        if self.noise == "device":
            slot.draws = device_noise.DrawPlan(slot.noise, shapes, True, self.dev)
            slot.noise_nchw, slot.noise_stage = [], []
        else:
            slot.draws = None
            slot.noise_nchw = [torch.zeros((b, c, h, w), dtype=torch.float32, device=self.dev) for b, c, h, w in shapes]
            slot.noise_stage = [torch.empty((b, c, h, w), dtype=torch.float32).pin_memory() for b, c, h, w in shapes]
        it = iter(slot.noise)
        joined = []

        def static_provider(b, c, h, w):
            if slot.draws is not None and not joined:                 # the generation branch joins before the first Sampler
                torch.cuda.current_stream(self.dev).wait_stream(self.noise_stream)
                joined.append(True)
            return next(it)
        n0 = _lib.kernel_launches()
        slot.graph = torch.cuda.CUDAGraph()
        with eng.noise_from(static_provider), torch.cuda.graph(slot.graph, stream=slot.stream):
            if slot.draws is not None:
                self._fork_noise(slot)
            else:
                self._relayout_noise(slot)
            slot.dev_out = self._compute(slot.inp)
        self.captures += 1
        slot.launches = _lib.kernel_launches() - n0
        slot.wkey = self._graph_key(eng)

    def _relayout_noise(self, slot: _Slot):
        """NCHW (as the reference draws it) -> NHWC (as the Sampler epilogues read it), on the device, on the current
        stream: ten small launches at the head of the captured step instead of a strided copy on the host for every step."""
        L = _lib.lib()
        for src, dst, (b, c, h, w) in zip(slot.noise_nchw, slot.noise, slot.noise_shapes):
            _lib.check(L.fusg_nchw_to_nhwc(_lib.ptr(src), _lib.ptr(dst), b, c, h, w, c, 0, 1, _lib.stream_ptr(torch)), "fusg_nchw_to_nhwc(noise)")      # elu 0, dtype 1 = fp32

    def _fork_noise(self, slot: _Slot):
        """noise="device": the step's generation on its own branch, forked from the head of the captured step.  It needs
        nothing but the start state, so it runs beside enc_up / dec_up and the warp until the first Sampler joins it."""
        self.noise_stream.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.noise_stream):
            slot.draws.launch()

    def _draw_noise(self, slot: _Slot, generator=None):
        """CPU generator (default: the global one), reference order and shapes (NCHW, vunet/layers.py:166), drawn straight
        into the slot's pinned staging buffers."""
        if slot.copied is not None:
            slot.copied.synchronize()          # the previous H2D out of these staging buffers has long completed
        for stage, (b, c, h, w) in zip(slot.noise_stage, slot.noise_shapes):
            torch.randn(b, c, h, w, generator=generator, out=stage)

    # The Sampler noise of a step costs ~3.6 ms of host time at 64 crops (1.3 M normals on the CPU generator, which is
    # what the reference draws from: vunet/layers.py:166).  To keep it off the submit path, the noise of the NEXT use
    # of a slot is drawn on a worker thread from a CLONE of the global generator; `submit` adopts it only if the
    # global generator is still in the state the clone started from (nobody seeded it or drew from it in between) and
    # then advances the global generator to the clone's end state -- bit-identical to drawing in `submit`.
    def _start_prefetch(self, slot: _Slot):
        if not self.prefetch_noise or not slot.noise_stage:
            return
        state0 = torch.get_rng_state()
        holder = {}

        def work():
            g = torch.Generator()
            g.set_state(state0)
            self._draw_noise(slot, generator=g)
            holder["state1"] = g.get_state()
        th = threading.Thread(target=work, daemon=True)
        th.start()
        slot.prefetch = (th, state0, holder)

    def _take_noise(self, slot: _Slot):
        """Fill the slot's staging buffers with this step's noise (adopt the prefetched draw when it is valid) -- or, with
        noise="device", take the generator's start state for the graph and advance the generator past the step."""
        if slot.draws is not None:
            if slot.copied is not None:
                slot.copied.synchronize()      # the previous H2D out of the pinned start state has completed
            slot.draws.take()
            return
        pf, slot.prefetch = slot.prefetch, None
        if pf is not None:
            th, state0, holder = pf
            th.join()
            if "state1" in holder and torch.equal(torch.get_rng_state(), state0):
                torch.set_rng_state(holder["state1"])
                return
        self._draw_noise(slot)

    def _upload_noise(self, slot: _Slot):
        if slot.draws is not None:
            slot.draws.upload()
            return
        for buf, stage in zip(slot.noise_nchw, slot.noise_stage):
            buf.copy_(stage, non_blocking=True)

    # ------------------------------------------------------------------ public API
    def submit(self, batch: dict, resident: bool = False) -> int:
        """batch: pinned host tensors `x` (B,6,256,256) f32, `y` (B,3,256,256) f32 -- or, 4x smaller, the three uint8
        images they are made of, `x_mask_u8`, `x_normal_u8`, `y_normal_u8` (B,256,256,3), see frame_ops -- and the warp inputs
        `src` (B,256,256,3) u8, `src_kp`/`dst_kp` (B,12,2) i32, `K` (B,3,3), `E_src`/`E_dst` (B,3,4), `kp3d` (B,12,3) f64.
        resident=True skips the host copies (inputs / noise already in the slot; outputs stay on the device)."""
        ticket = self.n
        slot = self.slots[ticket % self.depth]
        eng = self.model.engine()             # folds the weights again if the parameters changed (load_state_dict, .to, ...)
        # a captured graph bakes in the device pointers of the folded weights: re-capture after a reload instead of
        # replaying over freed memory
        fresh = slot.inp is None or slot.wkey != self._graph_key(eng) or set(slot.inp) != set(batch) or \
            any(tuple(slot.inp[k].shape) != tuple(v.shape) for k, v in batch.items())
        if not resident and not fresh:
            self._take_noise(slot)                                    # host RNG work overlaps the batches still in flight
        if slot.done is not None:
            slot.done.synchronize()                                   # the slot's previous outputs were consumed
        if fresh:
            if slot.prefetch is not None:                             # a draw into the old staging buffers is in flight
                slot.prefetch[0].join()
                slot.prefetch = None
            self._prepare_slot(slot, batch)
            if not resident:
                self._take_noise(slot)
        if not resident:
            with torch.cuda.stream(self.copy_stream):
                for k, v in batch.items():
                    slot.inp[k].copy_(v, non_blocking=True)
                self._upload_noise(slot)
                copied = torch.cuda.Event()
                copied.record(self.copy_stream)
            slot.copied = copied
            slot.stream.wait_event(copied)
        with torch.cuda.stream(slot.stream):
            slot.graph.replay()
            dev_out = dict(slot.dev_out)
            if self.gather_fn is not None:
                # the exchange step: every rank gets all completed crops ON THE DEVICE (for a device-side paste-back,
                # frame_ops.paste_back_batch); the host copy below stays this rank's own shard
                self._collect_and_gather(slot, dev_out["crops"], ticket)
            computed = torch.cuda.Event()
            computed.record(slot.stream)
        if not self.return_warped:
            dev_out.pop("warped", None)
        if resident:
            slot.done = computed
            self.n += 1
            return ticket
        if slot.out is None or any(tuple(slot.out[k].shape) != tuple(v.shape) for k, v in dev_out.items()):
            slot.out = {k: torch.empty(tuple(v.shape), dtype=v.dtype).pin_memory() for k, v in dev_out.items()}
        with torch.cuda.stream(self.out_stream):
            self.out_stream.wait_event(computed)
            for k, v in dev_out.items():
                slot.out[k].copy_(v, non_blocking=True)
                v.record_stream(self.out_stream)
            slot.done = torch.cuda.Event()
            slot.done.record(self.out_stream)
        self.n += 1
        nxt = self.slots[self.n % self.depth]
        if not resident and nxt.inp is not None and nxt.prefetch is None:
            self._start_prefetch(nxt)                                 # the next step's noise, off the submit path
        return ticket

    def _collect_and_gather(self, slot: _Slot, crops, ticket: int):
        """Runs on slot.stream.  Micro-batch `ticket % M` of the current step lands in the step buffer; the last one of
        a step triggers the all-gather of the whole step on comm_stream."""
        M, B = self.mps, crops.shape[0]
        if self.step_bufs is None or self.step_bufs[0].shape[0] != M * B:
            self.step_bufs = [torch.empty((M * B,) + tuple(crops.shape[1:]), dtype=crops.dtype, device=self.dev) for _ in range(2)]
            self.gather_done = [None, None]
        step, mb = divmod(ticket, M)
        which = step % 2
        buf = self.step_bufs[which]
        if self.gather_done[which] is not None:
            slot.stream.wait_event(self.gather_done[which])          # the gather that last read this buffer (two steps ago) is done
        if M == 1:
            src = crops
        else:
            buf[mb * B:(mb + 1) * B].copy_(crops, non_blocking=True)
            src = buf
        if mb == M - 1:
            filled = torch.cuda.Event()
            filled.record(slot.stream)
            if M > 1:
                # other micro-batches of this step may have run on other slot streams
                for other in self.slots:
                    if other is not slot and other.stream is not slot.stream and other.done is not None:
                        self.comm_stream.wait_stream(other.stream)
            self.comm_stream.wait_event(filled)
            with torch.cuda.stream(self.comm_stream):
                self.crops_all = self.gather_fn(src)
                done = torch.cuda.Event()
                done.record(self.comm_stream)
            src.record_stream(self.comm_stream)
            self.gather_done[which] = done
            slot.crops_all = self.crops_all

    def wait_gather(self):
        """Blocks until the last issued all-gather has completed; returns the gathered crops (device)."""
        for ev in self.gather_done:
            if ev is not None:
                ev.synchronize()
        return self.crops_all

    def result(self, ticket: int) -> dict:
        """Host (pinned) outputs of a submitted batch: `crops` (B,256,256,3) u8 completed views, `plane_j`, `vis`
        (+ `warped` (B,5,256,256,3) u8 planes with return_warped=True).  Valid until `depth` more batches are submitted."""
        slot = self.slots[ticket % self.depth]
        slot.done.synchronize()
        pj = slot.out.get("plane_j")
        if pj is not None and bool((pj == -2).any()):                # never hand back silently-black planes
            from .warp_learn.batch import RefusedCrops
            raise RefusedCrops(torch.nonzero((pj == -2).any(dim=1)).flatten().tolist())
        return slot.out

    def wait(self, ticket: int):
        self.slots[ticket % self.depth].done.synchronize()

    def device_outputs(self, ticket: int) -> dict:
        sl = self.slots[ticket % self.depth]
        out = dict(sl.dev_out)
        if sl.crops_all is not None:
            out["crops_all"] = sl.crops_all
        return out

    def launches_per_step(self) -> int:
        return self.slots[0].launches

    def d2h_bytes(self, ticket: int) -> int:
        return sum(v.numel() * v.element_size() for v in self.slots[ticket % self.depth].out.values())


class NovelViewPipeline(_GraphPipeline):
    """One complete reference forward per item: warp + `Vunet_fix_res.forward(y, x)` (appearance encoded for every item,
    decoded with the sampled z) + to_image.  See submit() for the batch keys."""
    WARP_KEYS = ("src", "src_kp", "dst_kp", "K", "E_src", "E_dst", "kp3d")

    def _warp(self, inp):
        return warp_batch(*(inp[k] for k in self.WARP_KEYS), device=self.dev)

    def _decode(self, inp):
        if "x" in inp:
            x, y = inp["x"], inp["y"]
        else:                                   # uint8 form: to_tensor / flip / concat on the device (frame_ops.u8_to_vunet_inputs)
            x, y = u8_to_vunet_inputs(inp["x_mask_u8"], inp["x_normal_u8"], inp["y_normal_u8"])
        return self.model(y, x)[0]


class TrajectoryPipeline(_GraphPipeline):
    """The trajectory loop (traj_test, trajectory_inference.py:230-233 and :413-426): each vehicle's appearance is encoded
    ONCE (`set_vehicles`: enc_up -> enc_down -> the six nin_k convolutions on the means mu), and every submitted (vehicle,
    future step) item runs only the shape path -- warp of the vehicle's source crop, dec_up(y), dec_down with that vehicle's
    cached appearance -- which is what the reference computes per step (decoding with mu_app), at a quarter of the
    convolution work of a full forward.  Source crops and cached appearance live in static buffers for `max_vehicles`
    vehicles, so `set_vehicles` replaces them in place without recapturing the step graphs.

        pipe = TrajectoryPipeline(model, max_vehicles=8)
        pipe.set_vehicles({"src": src_u8, "x_mask_u8": m_u8, "x_normal_u8": n_u8})       # (V,256,256,3) each
        t = pipe.submit({"vehicle": veh_i32, "src_kp": ..., "dst_kp": ..., "K": ..., "E_src": ..., "E_dst": ..., "kp3d": ...,
                         "kp3d_dst": ..., "y_normal_u8": y_u8})
        crops = pipe.result(t)["crops"]
    """
    WARP_KEYS = ("src_kp", "dst_kp", "K", "E_src", "E_dst", "kp3d")
    AR_BLOCKS = ("shape_decoder_1", "shape_decoder_2")

    def __init__(self, model, max_vehicles: int, depth: int = 2, **kw):
        super().__init__(model, depth=depth, **kw)
        if int(max_vehicles) <= 0:
            raise ValueError("max_vehicles must be positive")
        self.max_vehicles = int(max_vehicles)
        self.n_vehicles = 0
        self.veh_src = None      # (max_vehicles,H,W,3) u8 source crops
        self.veh_gk = None       # six (max_vehicles,h,w,512) ELU(nin_k(mu)) tensors, engine dtype: n = 0 (h = 2) k = 0..2, then n = 1 (h = 4)
        self.veh_wkey = None     # the folded weights the cache was encoded with

    def _graph_key(self, eng):
        # the graphs read the per-vehicle buffers by address: a reallocation (other crop size / engine dtype) recaptures
        return eng._wkey, None if self.veh_src is None else tuple(t.data_ptr() for t in [self.veh_src] + self.veh_gk)

    # ------------------------------------------------------------------ per-vehicle state
    def set_vehicles(self, batch: dict):
        """batch: `src` (V,H,W,3) u8 source crops and the appearance input of each vehicle -- `x` (V,6,256,256) f32, or the two
        uint8 images it is made of, `x_mask_u8` and `x_normal_u8` (V,256,256,3); host or device tensors.  Waits for every
        batch in flight, encodes the appearance (draws enc_down's two Sampler tensors from the CPU generator, as the
        reference does at step 0) and copies it and the source crops into the static per-vehicle buffers."""
        src = batch.get("src")
        if src is None or ("x" not in batch and not ("x_mask_u8" in batch and "x_normal_u8" in batch)):
            raise ValueError("set_vehicles: needs `src` and either `x` or `x_mask_u8` + `x_normal_u8`")
        V = int(src.shape[0])
        if not 0 < V <= self.max_vehicles:
            raise ValueError(f"set_vehicles: {V} vehicles, this pipeline holds 1..{self.max_vehicles}")
        if src.dim() != 4 or src.shape[-1] != 3 or src.dtype != torch.uint8:
            raise ValueError("set_vehicles: src must be (V,H,W,3) uint8")
        xs = [batch[k] for k in (("x",) if "x" in batch else ("x_mask_u8", "x_normal_u8"))]
        if any(int(t.shape[0]) != V for t in xs):
            raise ValueError("set_vehicles: appearance inputs and src disagree on V")
        for sl in self.slots:                                         # nothing in flight reads the buffers any more
            if sl.done is not None:
                sl.done.synchronize()
        dev = self.dev
        with torch.no_grad(), torch.cuda.device(dev):
            eng = self.model.engine()
            xs = [t.to(dev, non_blocking=True) for t in xs]
            if len(xs) == 1:
                x = xs[0].float().contiguous()
            else:                                                     # the y it writes as well is not needed
                x, _ = u8_to_vunet_inputs(xs[0].contiguous(), xs[1].contiguous(), xs[1].contiguous())
            # noise="device": enc_down's two Sampler tensors are made on the device too
            with eng.noise_from(device_noise.device_provider(device=dev)) if self.noise == "device" else contextlib.nullcontext():
                gk = eng.encode_vehicles(x)
            shapes = [tuple(src.shape[1:])] + [tuple(t.shape[1:]) for t in gk]
            if self.veh_src is None or [tuple(t.shape[1:]) for t in [self.veh_src] + self.veh_gk] != shapes or \
                    self.veh_gk[0].dtype != gk[0].dtype:
                self.veh_src = torch.zeros((self.max_vehicles,) + shapes[0], dtype=torch.uint8, device=dev)
                self.veh_gk = [torch.zeros((self.max_vehicles,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev) for t in gk]
            self.veh_src[:V].copy_(src, non_blocking=True)
            for buf, t in zip(self.veh_gk, gk):
                buf[:V].copy_(t)
            ready = torch.cuda.Event()
            ready.record(torch.cuda.current_stream(dev))
        for sl in self.slots:                                         # the next steps start after the new appearance is in place
            sl.stream.wait_event(ready)
        self.n_vehicles = V
        self.veh_wkey = eng._wkey

    # ------------------------------------------------------------------ one step of device work
    def _warp(self, inp):
        return warp_batch(self.veh_src, *(inp[k] for k in self.WARP_KEYS), device=self.dev, kp3d_dst=inp.get("kp3d_dst"),
                          src_index=inp["vehicle"])

    def _decode(self, inp):
        y = inp["y"] if "y" in inp else u8_to_vunet_y(inp["y_normal_u8"])
        eng = self.model.engine()
        out_d, skips_d = eng.dec_up(y, raw_skips=False)                  # skips are consumed pre-activated only
        gk = [torch.empty((y.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=self.dev) for t in self.veh_gk]
        gather_rows(list(zip(self.veh_gk, gk)), inp["vehicle"])        # one launch: every item's cached appearance
        return eng.dec_down(out_d, skips_d, enc_gk=[gk[:3], gk[3:]])[0]

    # ------------------------------------------------------------------ public API
    def submit(self, batch: dict, resident: bool = False) -> int:
        """batch, per item: `vehicle` (B,) int32 index into the vehicles of the last set_vehicles; the warp inputs `src_kp` /
        `dst_kp` (B,12,2) i32, `K` (B,3,3), `E_src` / `E_dst` (B,3,4), `kp3d` (B,12,3) f64 and optionally `kp3d_dst` (B,12,3)
        (the moved keypoints, kinematics.step_keypoints_batch); `y` (B,3,256,256) f32 or `y_normal_u8` (B,256,256,3) u8.
        The source crop is the vehicle's (set_vehicles).  Outputs as NovelViewPipeline: crops, plane_j, vis (+ warped)."""
        if self.veh_src is None:
            raise ValueError("TrajectoryPipeline.submit: call set_vehicles first")
        if "src" in batch:
            raise ValueError("TrajectoryPipeline.submit: the source crops are per vehicle (set_vehicles), not per item")
        missing = [k for k in ("vehicle",) + self.WARP_KEYS if k not in batch]
        if missing or ("y" in batch) == ("y_normal_u8" in batch):
            raise ValueError(f"TrajectoryPipeline.submit: needs {missing or ''} and exactly one of `y` / `y_normal_u8`")
        veh = batch["vehicle"]
        veh = veh if isinstance(veh, torch.Tensor) else torch.as_tensor(veh)
        if veh.dim() != 1 or veh.dtype.is_floating_point or veh.numel() == 0:
            raise ValueError("TrajectoryPipeline.submit: vehicle must be a non-empty (B,) integer array")
        lo, hi = int(veh.min()), int(veh.max())
        if lo < 0 or hi >= self.n_vehicles:
            raise ValueError(f"TrajectoryPipeline.submit: vehicle index {lo if lo < 0 else hi} outside [0, {self.n_vehicles})")
        eng = self.model.engine()
        if eng._wkey != self.veh_wkey:
            raise ValueError("TrajectoryPipeline.submit: the weights changed since set_vehicles; call it again to re-encode")
        if veh.dtype != torch.int32:
            batch = dict(batch, vehicle=veh.to(torch.int32))
        return super().submit(batch, resident)
