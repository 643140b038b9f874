"""The batched public API (pipeline.NovelViewPipeline: H2D -> CUDA-graph replay -> D2H, two batches in
flight) returns exactly what the eager module calls return, for the reference's noise semantics."""
from argparse import Namespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_pipeline_matches_eager_and_oracle(cuda):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch, to_image
    from oracle import vunet_oracle as VO, warp_oracle as WO
    B = 3
    sd = VO.make_state_dict(0)
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True))
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    pipe = NovelViewPipeline(m, depth=2, return_warped=True)
    batches = []
    for s in range(4):
        wb = synth.make_warp_batch(10 * s, B)
        xs, ys = synth.make_vunet_inputs(10 * s, B)
        host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
        host["x"], host["y"] = torch.from_numpy(xs).pin_memory(), torch.from_numpy(ys).pin_memory()
        batches.append(host)
    # pipelined: four batches through two slots (first use of a slot = eager + capture, then replays)
    torch.manual_seed(11)
    tickets, outs = [], []
    for host in batches:
        t = pipe.submit(host)
        if tickets:
            r = pipe.result(tickets[-1])
            outs.append({k: v.clone() for k, v in r.items()})
        tickets.append(t)
    outs.append({k: v.clone() for k, v in pipe.result(tickets[-1]).items()})
    assert pipe.launches_per_step() > 100
    # eager, same CPU noise stream
    torch.manual_seed(11)
    for host, out in zip(batches, outs):
        res = warp_batch(host["src"], host["src_kp"], host["dst_kp"], host["K"], host["E_src"], host["E_dst"], host["kp3d"])
        x_tilde = m(host["y"].cuda(), host["x"].cuda())[0]
        crops = to_image_batch(x_tilde)
        assert torch.equal(out["crops"], crops.cpu())
        assert torch.equal(out["warped"], res.warped.cpu())
        assert torch.equal(out["plane_j"], res.plane_j.cpu()) and torch.equal(out["vis"], res.vis.cpu())
        # to_image_batch == the reference-style per-image to_image
        assert np.array_equal(crops[0].cpu().numpy(), to_image(x_tilde[0], from_LAB=False))
    # and against the oracle for the first batch (warp bit-exact, image within one grey level of bf16 tolerance)
    torch.manual_seed(11)
    host = batches[0]
    with torch.no_grad():
        ref = VO.forward(sd, host["y"], host["x"])[0]
    ref_u8 = np.stack([to_image(ref[i], from_LAB=False) for i in range(B)])
    diff = np.abs(outs[0]["crops"].numpy().astype(int) - ref_u8.astype(int))
    assert diff.max() <= 2          # 1e-2 on [-1,1] is 1.3 grey levels
    w0 = WO.warp_fused(host["src"][0].numpy(), host["src_kp"][0].numpy(), host["dst_kp"][0].numpy(), host["K"][0].numpy(),
                       host["E_src"][0].numpy(), host["E_dst"][0].numpy(), host["kp3d"][0].numpy())[0]
    assert np.array_equal(outs[0]["warped"][0].numpy(), w0)


def test_warped_planes_stay_on_device_by_default(cuda):
    """Default outputs on the host: completed crops + flags; the planes stay in HBM (device_outputs) for get_icn_inputs."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    B = 2
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).cuda().eval()
    wb = synth.make_warp_batch(3, B)
    mk, ns, nd = synth.make_vunet_inputs_u8(3, B)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
    host.update(x_mask_u8=torch.from_numpy(mk).pin_memory(), x_normal_u8=torch.from_numpy(ns).pin_memory(), y_normal_u8=torch.from_numpy(nd).pin_memory())
    pipe = NovelViewPipeline(m, depth=2)
    t = pipe.submit(host)
    out = pipe.result(t)
    assert set(out) == {"crops", "plane_j", "vis"}
    res = warp_batch(host["src"], host["src_kp"], host["dst_kp"], host["K"], host["E_src"], host["E_dst"], host["kp3d"])
    assert torch.equal(pipe.device_outputs(t)["warped"], res.warped)


def test_reloading_weights_after_capture_recaptures_the_graph(cuda):
    """A captured graph bakes in the pointers of the folded weights; load_state_dict after the first submit must lead to
    a re-capture (outputs of the NEW weights), not a replay over freed memory."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch
    from oracle import vunet_oracle as VO
    B = 2
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True))
    m.load_state_dict(VO.make_state_dict(0), strict=True)
    m = m.cuda().eval()
    wb = synth.make_warp_batch(5, B)
    xs, ys = synth.make_vunet_inputs(5, B)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
    host["x"], host["y"] = torch.from_numpy(xs).pin_memory(), torch.from_numpy(ys).pin_memory()
    pipe = NovelViewPipeline(m, depth=2)
    torch.manual_seed(3)
    first = [pipe.result(pipe.submit(host))["crops"].clone() for _ in range(3)]
    m.load_state_dict(VO.make_state_dict(1), strict=True)             # second checkpoint, same module
    torch.manual_seed(3)
    second = [pipe.result(pipe.submit(host))["crops"].clone() for _ in range(3)]
    torch.manual_seed(3)
    eager = [to_image_batch(m(host["y"].cuda(), host["x"].cuda())[0]).cpu() for _ in range(3)]
    for a, b, c in zip(first, second, eager):
        assert torch.equal(b, c)
        assert not torch.equal(a, b)


@pytest.mark.parametrize("kind", ["novel_view", "trajectory"])
def test_a_failed_first_submit_leaves_the_engine_as_it_found_it(cuda, monkeypatch, kind):
    """The model's engine is shared with every eager caller: a step that raises during its first submit (here in
    to_image_batch, after the VUNet forward drew its noise from the warm-up's zero provider) must not leave that provider
    or the SM reserve installed, and the pipeline must prepare the slot again on the next submit."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib, pipeline, synth
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch
    from oracle import vunet_oracle as VO
    B = 2
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True))
    m.load_state_dict(VO.make_state_dict(0), strict=True)
    m = m.cuda().eval()
    wb = synth.make_warp_batch(5, B)
    xs, ys = synth.make_vunet_inputs(5, B)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
    x, y = torch.from_numpy(xs).pin_memory(), torch.from_numpy(ys).pin_memory()
    host["y"] = y
    if kind == "novel_view":
        host["x"] = x
        pipe = pipeline.NovelViewPipeline(m, depth=1)
        vehicles = None
    else:
        vehicles = {"src": host.pop("src"), "x": x}                       # vehicle b is item b
        host["vehicle"] = torch.arange(B, dtype=torch.int32)
        pipe = pipeline.TrajectoryPipeline(m, max_vehicles=B, depth=1)

    def eager_x_tilde():
        with torch.no_grad():
            return m(y.cuda(), x.cuda())[0]

    def eager_crops():
        if vehicles is None:
            return to_image_batch(eager_x_tilde()).cpu()
        with torch.no_grad():                                            # set_vehicles, then one step, on the engine
            e = m.engine()
            mu, _ = e.enc_down(*e.enc_up(x.cuda()))
            od, sd = e.dec_up(y.cuda())
            return to_image_batch(e.dec_down(od, sd, [g.aux["s2d_elu"] for g in mu])[0]).cpu()

    torch.manual_seed(4)
    before = eager_x_tilde()

    def fail(*a, **k):
        raise RuntimeError("injected failure")
    with monkeypatch.context() as mp:
        mp.setattr(pipeline, "to_image_batch", fail)
        if vehicles is not None:
            pipe.set_vehicles(vehicles)
        with pytest.raises(RuntimeError, match="injected failure"):
            pipe.submit(host)
    torch.cuda.synchronize()
    assert m.engine().noise_provider is None
    assert _lib.lib().fusg_conv2d_set_sm_reserve(-1) == 0
    torch.manual_seed(4)
    assert torch.equal(eager_x_tilde(), before)
    torch.manual_seed(6)
    if vehicles is not None:
        pipe.set_vehicles(vehicles)
    crops = pipe.result(pipe.submit(host))["crops"].clone()
    assert pipe.captures == 1
    torch.manual_seed(6)
    assert torch.equal(crops, eager_crops())


def test_noise_prefetch_keeps_generator_semantics(cuda):
    """The background noise draw is adopted only when it is bit-identical to drawing inside submit(): same outputs as
    prefetch_noise=False for one seed, also when the caller reseeds or draws from the global generator between steps."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    B = 2
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).cuda().eval()
    wb = synth.make_warp_batch(3, B)
    xs, ys = synth.make_vunet_inputs(3, B)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
    host["x"], host["y"] = torch.from_numpy(xs).pin_memory(), torch.from_numpy(ys).pin_memory()

    def run(prefetch):
        pipe = NovelViewPipeline(m, depth=2, prefetch_noise=prefetch)
        torch.manual_seed(5)
        outs = []
        for step in range(6):
            if step == 3:
                torch.manual_seed(77)              # reseed between steps: a pending prefetch must be discarded
            if step == 4:
                torch.rand(3)                      # foreign draw from the global generator
            t = pipe.submit(host)
            outs.append(pipe.result(t)["crops"].clone())
        return outs, torch.get_rng_state()

    a, sa = run(True)
    b, sb = run(False)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert torch.equal(sa, sb)                     # the global generator ends in the same state
    assert not torch.equal(a[0], a[1])             # different noise every step


def test_pipeline_uint8_inputs_equal_float_inputs(cuda):
    """Shipping the three uint8 images (9 B/pixel) and doing to_tensor / flip / concat on the device gives the same
    completed crops as shipping the float tensors the reference builds on the host (36 B/pixel)."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.frame_ops import u8_to_vunet_inputs
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    B = 2
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)).cuda().eval()
    wb = synth.make_warp_batch(7, B)
    xs, ys = synth.make_vunet_inputs(7, B)
    mk, ns, nd = synth.make_vunet_inputs_u8(7, B)
    x, y = u8_to_vunet_inputs(torch.from_numpy(mk).cuda(), torch.from_numpy(ns).cuda(), torch.from_numpy(nd).cuda())
    assert torch.equal(x.cpu(), torch.from_numpy(xs)) and torch.equal(y.cpu(), torch.from_numpy(ys))
    base = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
    hf = dict(base, x=torch.from_numpy(xs).pin_memory(), y=torch.from_numpy(ys).pin_memory())
    hu = dict(base, x_mask_u8=torch.from_numpy(mk).pin_memory(), x_normal_u8=torch.from_numpy(ns).pin_memory(),
              y_normal_u8=torch.from_numpy(nd).pin_memory())
    outs = []
    for host in (hf, hu):
        pipe = NovelViewPipeline(m, depth=2)
        torch.manual_seed(2)
        r = [pipe.result(pipe.submit(host))["crops"].clone() for _ in range(3)]
        outs.append(r)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_config5_clip_script_runs_end_to_end(cuda):
    """scripts/bench_clip.py at toy size: kinematics -> whole-frame fused warp -> get_icn_inputs -> ICN, VUNet, Lab->BGR, paste-back of
    both generators -- every row of SURVEY.md section 8 chained on the device must keep composing."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "scripts", "bench_clip.py"), "--vehicles", "3", "--steps", "2", "--chunk", "4", "--reps", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["items"] == 6 and d["ms_path"] > 0
    assert d["changed_pixels"]["icn_frames"] > 0 and d["changed_pixels"]["vunet_frames"] > 0
    assert set(d["stages_ms"]) >= {"kinematics", "warp", "icn_inputs", "icn", "vunet", "paste"}


def test_icn_generator_non_power_of_two_frames_use_the_direct_kernel(cuda):
    """Frame sizes the tcgen05 tiling does not cover (not powers of two) are served by the CUDA-core kernel of the same library --
    same program, same tolerance; nothing silently differs."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
    from oracle import icn_oracle as IO
    sd = IO.make_state_dict(0)
    g = G_Resnet(21)
    g.load_state_dict(sd, strict=True)
    g = g.cuda().eval()
    x = torch.from_numpy(synth.make_icn_inputs(2, 1, 96)[:, :, :80, :])            # 80 x 96
    with torch.no_grad():
        want = IO.forward(sd, x)
    got = g(x.cuda())
    assert got.shape == want.shape and (got.cpu() - want).abs().max().item() <= 1e-2


def test_bench_step_parity_b64(cuda):
    """Exactly bench.py's step (BASELINE config 2: 64 crops, uint8 inputs, graph replay): completed crops against the
    fp32 torch oracle of the VUNet forward with the same CPU noise (bar: 1e-2 on [-1,1] = 1.3 grey levels -> <= 2 after
    the truncating uint8 conversion), warped planes / flags bit-exact against the C oracle of the warp half."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image
    from oracle import vunet_oracle as VO, warp_oracle as WO
    B = 64
    sd = VO.make_state_dict(0)
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True))
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    wb = synth.make_warp_batch(0, B)
    xs, ys = synth.make_vunet_inputs(0, B)
    mk, ns, nd = synth.make_vunet_inputs_u8(0, B)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
    host.update(x_mask_u8=torch.from_numpy(mk).pin_memory(), x_normal_u8=torch.from_numpy(ns).pin_memory(), y_normal_u8=torch.from_numpy(nd).pin_memory())
    pipe = NovelViewPipeline(m, depth=2, return_warped=True)
    pipe.result(pipe.submit(host))                       # eager pass + capture
    pipe.result(pipe.submit(host))
    torch.manual_seed(21)
    out = {k: v.clone() for k, v in pipe.result(pipe.submit(host)).items()}       # a graph REPLAY, like the bench's timed steps
    torch.manual_seed(21)
    with torch.no_grad():
        ref = VO.forward(sd, torch.from_numpy(ys), torch.from_numpy(xs))[0]
    ref_u8 = np.stack([to_image(ref[i], from_LAB=False) for i in range(B)])
    diff = np.abs(out["crops"].numpy().astype(int) - ref_u8.astype(int))
    assert diff.max() <= 2, diff.max()
    assert (diff > 1).mean() < 1e-3
    for i in range(B):
        w, vis, pj, _ = WO.warp_fused(wb["src"][i], wb["src_kp"][i], wb["dst_kp"][i], wb["K"][i], wb["E_src"][i], wb["E_dst"][i], wb["kp3d"][i])
        assert np.array_equal(out["warped"][i].numpy(), w), i
        assert np.array_equal(out["plane_j"][i].numpy(), pj) and np.array_equal(out["vis"][i].numpy(), vis[:2])


def _nccl_worker(rank, world, port, n_total, q):
    import os
    import torch
    import torch.distributed as dist
    from future_urban_scene_generation_b200.parallel import shard_range, gather_crops
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        g = torch.Generator().manual_seed(5)
        full = torch.randint(0, 256, (n_total, 64, 64, 3), dtype=torch.uint8, generator=g)
        b, e = shard_range(n_total, rank, world)
        out = gather_crops(full[b:e].cuda(), n_total)
        torch.cuda.synchronize()
        q.put((rank, bool(torch.equal(out.cpu(), full))))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n_total", [8, 7])
def test_gather_crops_nccl_world_2(cuda, n_total):
    """gather_crops over NCCL on two GPUs: global crop order, even and ragged shards.  Skips on a one-GPU box."""
    torch = cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29650 + n_total
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, n_total, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
    got = sorted(q.get(timeout=10) for _ in range(2))
    assert got == [(0, True), (1, True)]
