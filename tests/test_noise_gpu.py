"""Sampler noise made on the device (noise.py, csrc/noise.cu) against torch.randn on the CPU generator, bit for bit, and the
two graph pipelines with noise="device" against noise="host"."""
from argparse import Namespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ARGS = Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)


def sampler_shapes(B, form="forward"):
    enc = [(B, 128, 4, 4), (B, 128, 8, 8)]
    dec = [(B, 128, 2, 2)] * 4 + [(B, 128, 4, 4)] * 4
    return {"forward": enc + dec, "step": dec}[form]


def _bits_equal(torch, a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _check_draws(torch, shapes, layout, g):
    from future_urban_scene_generation_b200.noise import randn_cpu_exact
    ref_g = torch.Generator()
    ref_g.set_state(g.get_state())
    got = randn_cpu_exact(shapes, layout=layout, generator=g)
    ref = [torch.randn(*s, generator=ref_g) for s in shapes]
    assert torch.equal(g.get_state(), ref_g.get_state())          # set before the device has drawn anything
    for s, a, r in zip(shapes, got, ref):
        a = a.cpu()
        if layout == "nhwc":
            assert tuple(a.shape) == (s[0], s[2], s[3], s[1])
            a = a.permute(0, 3, 1, 2)
        assert _bits_equal(torch, a, r), (s, layout, float((a - r).abs().max()))


@pytest.mark.parametrize("B", [1, 5, 64])
@pytest.mark.parametrize("form", ["forward", "step"])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_device_draws_equal_torch_randn(cuda, B, form, layout):
    torch = cuda
    g = torch.Generator()
    g.manual_seed(B * 7 + len(form))
    torch.randn(B + 3, generator=g)                               # a start in the middle of a block
    _check_draws(torch, sampler_shapes(B, form), layout, g)


def test_a_chain_of_20_steps_on_the_global_generator(cuda):
    torch = cuda
    from future_urban_scene_generation_b200.noise import randn_cpu_exact
    torch.manual_seed(11)
    ref_g = torch.Generator()
    ref_g.set_state(torch.get_rng_state())
    outs, refs = [], []
    for k in range(20):
        shapes = sampler_shapes(64, "forward" if k % 2 else "step")
        outs.append(randn_cpu_exact(shapes, layout="nhwc"))      # enqueued back to back, compared at the end
        refs.append([torch.randn(*s, generator=ref_g) for s in shapes])
    assert torch.equal(torch.get_rng_state(), ref_g.get_state())
    for o, r in zip(outs, refs):
        for a, b in zip(o, r):
            assert _bits_equal(torch, a.cpu().permute(0, 3, 1, 2), b)


def test_into_given_outputs_and_on_a_side_stream(cuda):
    torch = cuda
    from future_urban_scene_generation_b200.noise import randn_cpu_exact
    shapes = [(3, 16, 4, 4), (2, 128, 8, 8)]
    out = [torch.full(s, float("nan"), device="cuda") for s in shapes]
    g = torch.Generator()
    g.manual_seed(5)
    ref_g = torch.Generator()
    ref_g.set_state(g.get_state())
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        got = randn_cpu_exact(shapes, generator=g, out=out)
    st.synchronize()
    assert all(a is b for a, b in zip(got, out))
    for a, s in zip(out, shapes):
        assert _bits_equal(torch, a.cpu(), torch.randn(*s, generator=ref_g))


def test_self_check_raises_on_a_wrong_expected_draw(cuda):
    torch = cuda
    from future_urban_scene_generation_b200 import noise, _lib
    noise.self_check("cuda:0")                                    # the real comparison passes
    g = torch.Generator()
    g.manual_seed(1)
    wrong = [torch.randn(2, 3, 8, 8, generator=g), torch.randn(1, 16, 5, 3, generator=g)]
    with pytest.raises(_lib.FusgError, match=torch.backends.cpu.get_cpu_capability()):
        noise.self_check("cuda:0", expected=wrong)


def test_engine_provider_equals_the_host_draw(cuda):
    torch = cuda
    from future_urban_scene_generation_b200 import noise, synth
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from oracle import vunet_oracle as VO
    m = Vunet_fix_res(ARGS)
    m.load_state_dict(VO.make_state_dict(0), strict=True)
    m = m.cuda().eval()
    x, y = (torch.from_numpy(t).cuda() for t in synth.make_vunet_inputs(2, 5))
    with torch.no_grad():
        torch.manual_seed(3)
        a = [t.clone() for t in m(y, x)[:1]]
        sa = torch.get_rng_state()
        torch.manual_seed(3)
        with m.engine().noise_from(noise.device_provider()):
            b = [t.clone() for t in m(y, x)[:1]]
        sb = torch.get_rng_state()
    assert m.engine().noise_provider is None
    assert torch.equal(a[0], b[0]) and torch.equal(sa, sb)


# ---------------------------------------------------------------------------------------------------------------- pipelines
def _model(torch, seed=0):
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from oracle import vunet_oracle as VO
    m = Vunet_fix_res(ARGS)
    m.load_state_dict(VO.make_state_dict(seed), strict=True)
    return m.cuda().eval()


def _nv_batches(torch, n, B):
    from future_urban_scene_generation_b200 import synth
    out = []
    for s in range(n):
        wb = synth.make_warp_batch(20 + s, B)
        xs, ys = synth.make_vunet_inputs(20 + s, B)
        h = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
        h["x"], h["y"] = torch.from_numpy(xs).pin_memory(), torch.from_numpy(ys).pin_memory()
        out.append(h)
    return out


def _drive(torch, pipe, batches, between, depth):
    """Submits with up to `depth` tickets in flight; between(k) runs before submit k (seeds, foreign draws, set_vehicles)."""
    outs, pending = [], []
    for k, h in enumerate(batches):
        between(k)
        if len(pending) == depth:
            outs.append({kk: v.clone() for kk, v in pipe.result(pending.pop(0)).items()})
        pending.append(pipe.submit(h))
    for t in pending:
        outs.append({kk: v.clone() for kk, v in pipe.result(t).items()})
    return outs, torch.get_rng_state()


def _assert_same_runs(torch, a, b):
    assert len(a[0]) == len(b[0])
    for x, y in zip(a[0], b[0]):
        assert set(x) == set(y)
        for k in x:
            assert torch.equal(x[k], y[k]), k
    assert torch.equal(a[1], b[1])


@pytest.mark.parametrize("depth", [2, 3])
def test_novel_view_pipeline_device_noise_equals_host_noise(cuda, depth):
    torch = cuda
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline
    m = _model(torch)
    batches = _nv_batches(torch, 7, 5)

    def between(k):
        if k == 3:
            torch.manual_seed(77)
        if k == 5:
            torch.randn(3)                                      # a user draw from the global generator between submits

    runs, launches = {}, {}
    for mode in ("host", "device"):
        pipe = NovelViewPipeline(m, depth=depth, return_warped=True, noise=mode)
        torch.manual_seed(5)
        runs[mode] = _drive(torch, pipe, batches, between, depth)
        launches[mode] = pipe.launches_per_step()
        if mode == "device":
            assert all(not sl.noise_stage and not sl.noise_nchw and sl.prefetch is None for sl in pipe.slots)
    _assert_same_runs(torch, runs["host"], runs["device"])
    print(f"NovelViewPipeline launches per step: host {launches['host']}, device {launches['device']}")
    assert launches["device"] == launches["host"] - 10 + 2   # ten relayouts out, the two generation kernels in


@pytest.mark.parametrize("depth", [2, 3])
def test_trajectory_pipeline_device_noise_equals_host_noise(cuda, depth):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import TrajectoryPipeline
    m = _model(torch)
    V, veh = 3, [0, 0, 1, 2, 2, 2, 1]
    steps = []
    for s in range(7):
        wb = synth.make_warp_batch(30 + 10 * s, len(veh), crops=False)
        h = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
        h["kp3d_dst"] = (h["kp3d"] * 1.02).pin_memory()
        h["y"] = torch.from_numpy(synth.make_vunet_inputs(30 + 10 * s, len(veh))[1]).pin_memory()
        h["vehicle"] = torch.tensor(veh, dtype=torch.int32).pin_memory()
        steps.append(h)

    def vehicles(seed):
        x, _ = synth.make_vunet_inputs(seed, V)
        src = np.stack([synth.make_crop(seed + v) for v in range(V)])
        return {"src": torch.from_numpy(src).pin_memory(), "x": torch.from_numpy(x).pin_memory()}
    runs, launches = {}, {}
    for mode in ("host", "device"):
        pipe = TrajectoryPipeline(m, max_vehicles=4, depth=depth, return_warped=True, noise=mode)
        torch.manual_seed(9)
        pipe.set_vehicles(vehicles(300))

        def between(k):
            if k == 2:
                torch.manual_seed(19)
            if k == 4:
                pipe.set_vehicles(vehicles(400))              # re-encodes: two more draws from the generator
            if k == 5:
                torch.rand(5)
        runs[mode] = _drive(torch, pipe, steps, between, depth)
        launches[mode] = pipe.launches_per_step()
    _assert_same_runs(torch, runs["host"], runs["device"])
    print(f"TrajectoryPipeline launches per step: host {launches['host']}, device {launches['device']}")
    assert launches["device"] == launches["host"] - 8 + 2
