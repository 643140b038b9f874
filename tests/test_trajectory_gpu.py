"""The trajectory form of the hot path: the indexed fused warp (one source image per vehicle), the per-item row gather, and
pipeline.TrajectoryPipeline (appearance encoded once per vehicle, shape path per (vehicle, step) item) against the engine
run eagerly, the fp32 oracle and the reference's generator semantics."""
from argparse import Namespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ARGS = Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)


def _model(seed=0):
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from oracle import vunet_oracle as VO
    m = Vunet_fix_res(ARGS)
    m.load_state_dict(VO.make_state_dict(seed), strict=True)
    return m.cuda().eval()


def _warp_pair(torch, src_v, idx, wb, kp3d_dst=None):
    """(indexed call, call on the expanded per-item source) -> both WarpResults, synchronised."""
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    args = (wb["src_kp"], wb["dst_kp"], wb["K"], wb["E_src"], wb["E_dst"], wb["kp3d"])
    src_d = torch.as_tensor(src_v).cuda()
    idx_d = torch.as_tensor(idx, dtype=torch.int32).cuda()
    a = warp_batch(src_d, *args, kp3d_dst=kp3d_dst, src_index=idx_d)
    b = warp_batch(src_d[idx_d.long()].contiguous(), *args, kp3d_dst=kp3d_dst)
    torch.cuda.synchronize()
    return a, b


def _assert_same(torch, a, b):
    assert torch.equal(a.warped, b.warped)
    assert torch.equal(a.vis, b.vis)
    assert torch.equal(a.plane_j, b.plane_j)
    assert torch.equal(a.H12.view(torch.int64), b.H12.view(torch.int64))


# ---------------------------------------------------------------------------------------------------------------- 1. warp
@pytest.mark.parametrize("case", ["in_frame", "full_height", "out_of_frame"])
@pytest.mark.parametrize("moved", [False, True])
def test_indexed_warp_is_bit_exact_crops(cuda, case, moved):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    B, V = 12, 5
    wb = synth.make_warp_batch(40, B, crops=False, out_of_frame=case == "out_of_frame")
    if case == "full_height":
        # stretch the source polygons vertically: a vehicle filling the crop needs the full-height (MAX_HW) source window
        kp = wb["src_kp"].astype(np.int64)
        kp[:, :, 1] = (kp[:, :, 1] - 128) * 2 + 128
        wb["src_kp"] = np.int32(kp)
        rows = np.clip(wb["src_kp"][:, :, 1], 0, 255)
        assert (rows.max(1) - rows.min(1) > 120).sum() >= 4
    src_v = np.stack([synth.make_crop(900 + v) for v in range(V)])
    idx = np.array([3, 0, 0, 4, 2, 2, 1, 3, 4, 0, 1, 2], np.int32)            # repeated, unsorted
    kd = torch.as_tensor(wb["kp3d"] * 1.03 + np.array([0.2, -0.1, 0.0])) if moved else None
    a, b = _warp_pair(torch, src_v, idx, wb, kd)
    _assert_same(torch, a, b)
    assert int((a.plane_j >= 0).sum()) > 0                                   # the case really warps something
    assert int(a.warped.count_nonzero()) > 0


@pytest.mark.parametrize("hw", [(300, 400), (720, 1280)])
def test_indexed_warp_is_bit_exact_whole_frames(cuda, hw):
    """The whole-frame path (frames > 256, k_warp_frame) on trajectory items: vehicles x steps from the kinematics."""
    torch = cuda
    from future_urban_scene_generation_b200 import kinematics as KM, synth
    H, W = hw
    V, S = 3, 4
    cases = [synth.make_trajectory_case(v, steps=S, h=H, w=W) for v in range(V)]
    for c in cases:                                          # a focal length that keeps the vehicle a fraction of the frame
        c["K"] = np.array([[1.3 * W, 0, W / 2.0], [0, 1.3 * W, H / 2.0], [0, 0, 1.0]])
    kp3d = np.stack([c["kp3d"] for c in cases])
    R, t, K = np.stack([c["R"] for c in cases]), np.stack([c["t"] for c in cases]), np.stack([c["K"] for c in cases])
    E = np.concatenate([R, t[:, :, None]], 2)
    src_kp = np.int32(np.stack([synth.project(K[v], np.vstack([E[v], [0, 0, 0, 1]]), kp3d[v]) for v in range(V)]))
    poses = [KM.trajectory_poses(c["meter_coords"]) for c in cases]
    veh = np.repeat(np.arange(V), S).astype(np.int32)
    moved, _, dst_kp = KM.step_keypoints_batch(kp3d, veh, np.concatenate([p[2] for p in poses]), np.concatenate([p[1] for p in poses]),
                                               R, t, K, H, W)
    order = np.array([5, 0, 11, 2, 2, 7, 1, 9, 4, 10, 3, 6, 8], np.int64)     # unsorted items, one repeated
    wb = dict(src_kp=src_kp[veh[order]], dst_kp=dst_kp[torch.as_tensor(order).cuda()], K=K[veh[order]], E_src=E[veh[order]],
              E_dst=E[veh[order]], kp3d=kp3d[veh[order]])
    frames = np.stack([np.random.default_rng(500 + v).integers(0, 256, (H, W, 3), dtype=np.uint8) for v in range(V)])
    for kd in (None, moved[torch.as_tensor(order).cuda()]):
        a, b = _warp_pair(torch, frames, veh[order], wb, kd)
        _assert_same(torch, a, b)
        assert int((a.plane_j >= 0).sum()) > 0


def test_indexed_warp_refuses_an_index_out_of_range(cuda):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.warp_learn import warp_batch, check_refused, RefusedCrops
    B, V = 6, 3
    wb = synth.make_warp_batch(60, B, crops=False)
    src_v = np.stack([synth.make_crop(950 + v) for v in range(V)])
    idx = np.array([2, 0, V, 1, 1, 0], np.int32)                              # item 2 names a source that does not exist
    args = (wb["src_kp"], wb["dst_kp"], wb["K"], wb["E_src"], wb["E_dst"], wb["kp3d"])
    with pytest.raises(ValueError):                                          # a host index is checked before the upload
        warp_batch(src_v, *args, src_index=idx)
    with pytest.raises(ValueError):
        warp_batch(src_v, *args, src_index=np.array([0, 1, 2, 0, -1, 0], np.int32))
    idx_d = torch.as_tensor(idx).cuda()                                      # on the device: the kernels refuse the item
    res = warp_batch(torch.as_tensor(src_v).cuda(), *args, src_index=idx_d)
    ok = np.array([0, 1, 3, 4, 5])
    ref = warp_batch(src_v[idx[ok]], *(a[ok] for a in args))
    torch.cuda.synchronize()
    pj = res.plane_j.cpu()
    assert (pj[2] == -2).all() and not (pj[ok] == -2).any()
    assert int(res.warped[2].count_nonzero()) == 0 and int(res.H12[2].abs().sum()) == 0
    assert torch.equal(res.warped[ok], ref.warped) and torch.equal(res.plane_j[ok], ref.plane_j)
    with pytest.raises(RefusedCrops) as ei:
        check_refused(res)
    assert ei.value.indices == [2]
    with pytest.raises(RefusedCrops):
        warp_batch(torch.as_tensor(src_v).cuda(), *args, src_index=idx_d, check=True)


# ---------------------------------------------------------------------------------------------------------------- 2. gather
def test_gather_rows_equals_torch_indexing(cuda):
    torch = cuda
    from future_urban_scene_generation_b200.frame_ops import gather_rows
    g = torch.Generator(device="cuda").manual_seed(3)
    B = 37
    srcs = [torch.randn((5, 2, 2, 512), device="cuda", generator=g).to(torch.bfloat16),
            torch.randn((5, 4, 4, 512), device="cuda", generator=g).to(torch.bfloat16),
            torch.randn((3, 16), device="cuda", generator=g),                            # 64-byte rows, fewer source rows
            torch.randint(0, 255, (7, 3, 16), device="cuda", generator=g, dtype=torch.uint8),   # 48-byte rows
            torch.randn((5, 128, 1024), device="cuda", generator=g)]                     # 512 KB rows: split over CTAs
    idx = torch.randint(0, 5, (B,), device="cuda", generator=g, dtype=torch.int32)
    idx[3], idx[9], idx[20] = -1, 5, 6                                                   # out of range for some or all segments
    dsts = [torch.full((B,) + tuple(s.shape[1:]), 7, dtype=s.dtype, device="cuda") for s in srcs]
    gather_rows(list(zip(srcs, dsts)), idx)
    torch.cuda.synchronize()
    for s, d in zip(srcs, dsts):
        n = s.shape[0]
        valid = (idx >= 0) & (idx < n)
        want = torch.zeros_like(d)
        want[valid] = s[idx[valid].long()]
        assert torch.equal(d, want)
    with pytest.raises(ValueError):
        gather_rows([(srcs[0], dsts[0])] * 9, idx)


# ---------------------------------------------------------------------------------------------------------------- 3..8 pipeline
VEH = [0, 0, 1, 2, 2, 2, 1]


def _vehicles(torch, V, seed=300):
    from future_urban_scene_generation_b200 import synth
    x, _ = synth.make_vunet_inputs(seed, V)
    src = np.stack([synth.make_crop(seed + v) for v in range(V)])
    return {"src": torch.from_numpy(src).pin_memory(), "x": torch.from_numpy(x).pin_memory()}


def _steps(torch, n, veh, seed=0, u8=False):
    from future_urban_scene_generation_b200 import synth
    B = len(veh)
    out = []
    for s in range(n):
        wb = synth.make_warp_batch(seed + 10 * s, B, crops=False)
        h = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in wb.items()}
        h["kp3d_dst"] = (h["kp3d"] * 1.02).pin_memory()
        if u8:
            h["y_normal_u8"] = torch.from_numpy(synth.make_vunet_inputs_u8(seed + 10 * s, B)[2]).pin_memory()
        else:
            h["y"] = torch.from_numpy(synth.make_vunet_inputs(seed + 10 * s, B)[1]).pin_memory()
        h["vehicle"] = torch.tensor(veh, dtype=torch.int32).pin_memory()
        out.append(h)
    return out


def _run_pipeline(pipe, steps):
    tickets, outs = [], []
    for h in steps:
        t = pipe.submit(h)
        if tickets:
            outs.append({k: v.clone() for k, v in pipe.result(tickets[-1]).items()})
        tickets.append(t)
    outs.append({k: v.clone() for k, v in pipe.result(tickets[-1]).items()})
    return outs


def _eager(torch, m, veh_inp, steps):
    """traj_test order on the engine: enc_up / enc_down once on the vehicles, then per step dec_up(y) and dec_down with
    the items' rows of ELU(S2D(mu)) -- the existing enc_g path, which runs the nin_k convolutions per item."""
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image_batch
    with torch.no_grad():
        e = m.engine()
        out_e, sk_e = e.enc_up(veh_inp["x"].cuda())
        mu_app, _ = e.enc_down(out_e, sk_e)
        crops = []
        for h in steps:
            v = h["vehicle"].cuda().long()
            od, sd = e.dec_up(h["y"].cuda())
            xt, _, _ = e.dec_down(od, sd, [mu.aux["s2d_elu"][v].contiguous() for mu in mu_app])
            crops.append(to_image_batch(xt).cpu())
    return crops


def _check_warp(torch, outs, veh_inp, steps):
    from future_urban_scene_generation_b200.warp_learn import warp_batch
    for h, o in zip(steps, outs):
        v = h["vehicle"].long()
        res = warp_batch(veh_inp["src"][v].contiguous(), h["src_kp"], h["dst_kp"], h["K"], h["E_src"], h["E_dst"], h["kp3d"],
                         kp3d_dst=h["kp3d_dst"])
        torch.cuda.synchronize()
        assert torch.equal(o["warped"], res.warped.cpu())
        assert torch.equal(o["plane_j"], res.plane_j.cpu()) and torch.equal(o["vis"], res.vis.cpu())


def test_pipeline_equals_the_engine_run_eagerly(cuda):
    torch = cuda
    from future_urban_scene_generation_b200.pipeline import TrajectoryPipeline
    m = _model(0)
    veh_inp = _vehicles(torch, 3)
    steps = _steps(torch, 4, VEH)
    pipe = TrajectoryPipeline(m, max_vehicles=4, depth=2, return_warped=True)
    torch.manual_seed(13)
    pipe.set_vehicles(veh_inp)
    outs = _run_pipeline(pipe, steps)
    torch.manual_seed(13)
    eager = _eager(torch, m, veh_inp, steps)
    for o, c in zip(outs, eager):
        assert torch.equal(o["crops"], c)
    assert not torch.equal(outs[0]["crops"], outs[1]["crops"])
    _check_warp(torch, outs, veh_inp, steps)


def test_pipeline_matches_the_reference_semantics(cuda):
    """Against the fp32 oracle in traj_test's order (forward_enc_up / forward_enc_down once, forward_dec_up /
    forward_dec_down(..., mu_app of the item's vehicle) per step), at the bar of test_bench_step_parity_b64."""
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import TrajectoryPipeline
    from future_urban_scene_generation_b200.warp_learn.planes_utils import to_image
    from oracle import vunet_oracle as VO, warp_oracle as WO

    def oracle_crops(sd, x_v, ys, vehs, seed):
        torch.manual_seed(seed)
        with torch.no_grad():
            out_e, sk_e = VO.forward_enc_up(sd, x_v)
            mu_r, _ = VO.forward_enc_down(sd, out_e, sk_e)
            res = []
            for y, v in zip(ys, vehs):
                od, sk = VO.forward_dec_up(sd, y)
                xt = VO.forward_dec_down(sd, od, sk, [mu[torch.as_tensor(v).long()] for mu in mu_r])[0]
                res.append(np.stack([to_image(xt[i], from_LAB=False) for i in range(xt.shape[0])]))
        return res

    def close(got, want):
        diff = np.abs(got.astype(int) - want.astype(int))
        assert diff.max() <= 2, diff.max()
        assert (diff > 1).mean() < 1e-3

    sd = VO.make_state_dict(0)
    m = _model(0)
    # the small case of test 3, fp32 inputs
    veh_inp = _vehicles(torch, 3)
    steps = _steps(torch, 4, VEH)
    pipe = TrajectoryPipeline(m, max_vehicles=3, depth=2)
    torch.manual_seed(17)
    pipe.set_vehicles(veh_inp)
    outs = _run_pipeline(pipe, steps)
    want = oracle_crops(sd, veh_inp["x"], [h["y"] for h in steps], [h["vehicle"] for h in steps], 17)
    for o, w in zip(outs, want):
        close(o["crops"].numpy(), w)
    # B = 64 from V = 8 vehicles, uint8 inputs, measured on a graph REPLAY
    V, B = 8, 64
    veh = np.random.default_rng(4).integers(0, V, B).astype(np.int32)
    mk, ns, _ = synth.make_vunet_inputs_u8(700, V)
    xs, _ = synth.make_vunet_inputs(700, V)
    src_v = np.stack([synth.make_crop(700 + v) for v in range(V)])
    vin = {"src": torch.from_numpy(src_v), "x_mask_u8": torch.from_numpy(mk), "x_normal_u8": torch.from_numpy(ns)}
    st = _steps(torch, 1, veh, seed=800, u8=True)[0]
    for k in ("kp3d_dst",):
        st.pop(k)
    _, ys = synth.make_vunet_inputs(800, B)
    pipe = TrajectoryPipeline(m, max_vehicles=V, depth=2, return_warped=True)
    torch.manual_seed(1)
    pipe.set_vehicles(vin)
    pipe.result(pipe.submit(st))                                             # eager pass + capture
    pipe.result(pipe.submit(st))
    torch.manual_seed(23)
    pipe.set_vehicles(vin)
    out = {k: v.clone() for k, v in pipe.result(pipe.submit(st)).items()}    # slot 0 again: a replay
    assert pipe.captures == 2
    want = oracle_crops(sd, torch.from_numpy(xs), [torch.from_numpy(ys)], [veh], 23)[0]
    close(out["crops"].numpy(), want)
    wb = {k: v.numpy() for k, v in st.items()}
    for i in range(B):
        w, vis, pj, _ = WO.warp_fused(src_v[veh[i]], wb["src_kp"][i], wb["dst_kp"][i], wb["K"][i], wb["E_src"][i], wb["E_dst"][i], wb["kp3d"][i])
        assert np.array_equal(out["warped"][i].numpy(), w), i
        assert np.array_equal(out["plane_j"][i].numpy(), pj) and np.array_equal(out["vis"][i].numpy(), vis[:2])


@pytest.mark.parametrize("prefetch", [True, False])
def test_generator_semantics_are_kept(cuda, prefetch):
    torch = cuda
    from future_urban_scene_generation_b200.pipeline import TrajectoryPipeline
    m = _model(0)
    V, B = 3, len(VEH)
    veh_inp = _vehicles(torch, V)
    steps = _steps(torch, 5, VEH)

    def expected(seed, k, reseed_at=None):
        torch.manual_seed(seed)
        torch.randn(V, 128, 4, 4)
        torch.randn(V, 128, 8, 8)
        for s in range(k):
            if s == reseed_at:
                torch.manual_seed(seed + 100)
            for _ in range(4):
                torch.randn(B, 128, 2, 2)
            for _ in range(4):
                torch.randn(B, 128, 4, 4)
        return torch.get_rng_state()

    for reseed_at in (None, 3):
        pipe = TrajectoryPipeline(m, max_vehicles=V, depth=2, prefetch_noise=prefetch)
        torch.manual_seed(9)
        pipe.set_vehicles(veh_inp)
        for s, h in enumerate(steps):
            if s == reseed_at:
                torch.manual_seed(109)
            pipe.result(pipe.submit(h))
        assert torch.equal(torch.get_rng_state(), expected(9, len(steps), reseed_at))


def test_appearance_swaps_without_recapture_and_reloads_recapture(cuda):
    torch = cuda
    from future_urban_scene_generation_b200.pipeline import TrajectoryPipeline
    from oracle import vunet_oracle as VO
    m = _model(0)
    steps = _steps(torch, 3, VEH)
    pipe = TrajectoryPipeline(m, max_vehicles=4, depth=2)
    torch.manual_seed(5)
    pipe.set_vehicles(_vehicles(torch, 3, seed=300))
    _run_pipeline(pipe, steps)
    assert pipe.captures == 2                                                # one graph per slot
    new = _vehicles(torch, 3, seed=400)
    torch.manual_seed(6)
    pipe.set_vehicles(new)
    outs = _run_pipeline(pipe, steps)
    assert pipe.captures == 2                                                # the appearance changed in place
    torch.manual_seed(6)
    for o, c in zip(outs, _eager(torch, m, new, steps)):
        assert torch.equal(o["crops"], c)
    # new weights: the cache is stale until set_vehicles runs again, and the graphs are captured anew
    m.load_state_dict(VO.make_state_dict(1), strict=True)
    with pytest.raises(ValueError):
        pipe.submit(steps[0])
    torch.manual_seed(7)
    pipe.set_vehicles(new)
    outs2 = _run_pipeline(pipe, steps)
    assert pipe.captures == 4
    torch.manual_seed(7)
    for o, o_old, c in zip(outs2, outs, _eager(torch, m, new, steps)):
        assert torch.equal(o["crops"], c)
        assert not torch.equal(o["crops"], o_old["crops"])


def test_the_trajectory_step_is_smaller(cuda):
    torch = cuda
    from future_urban_scene_generation_b200 import synth
    from future_urban_scene_generation_b200.pipeline import NovelViewPipeline, TrajectoryPipeline
    m = _model(0)
    B = len(VEH)
    tp = TrajectoryPipeline(m, max_vehicles=3, depth=1)
    tp.set_vehicles(_vehicles(torch, 3))
    h = _steps(torch, 1, VEH)[0]
    h.pop("kp3d_dst")
    tp.result(tp.submit(h))
    nv = NovelViewPipeline(m, depth=1)
    wb = synth.make_warp_batch(0, B)
    xs, ys = synth.make_vunet_inputs(0, B)
    hn = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in wb.items()}
    hn["x"], hn["y"] = torch.from_numpy(xs), torch.from_numpy(ys)
    nv.result(nv.submit(hn))
    assert nv.launches_per_step() - tp.launches_per_step() >= 36, (nv.launches_per_step(), tp.launches_per_step())


def test_input_errors_are_refused(cuda):
    torch = cuda
    from future_urban_scene_generation_b200.pipeline import TrajectoryPipeline
    m = _model(0)
    pipe = TrajectoryPipeline(m, max_vehicles=3, depth=2)
    steps = _steps(torch, 1, VEH)
    with pytest.raises(ValueError):
        pipe.submit(steps[0])                                                # no vehicles yet
    with pytest.raises(ValueError):
        pipe.set_vehicles(_vehicles(torch, 4))                               # V > max_vehicles
    pipe.set_vehicles(_vehicles(torch, 3))
    bad = dict(steps[0], vehicle=torch.tensor([0, 1, 2, 3, 0, 0, 0], dtype=torch.int32))
    n0 = pipe.n
    with pytest.raises(ValueError):
        pipe.submit(bad)
    with pytest.raises(ValueError):
        pipe.submit(dict(steps[0], vehicle=torch.tensor([0, -1, 2, 0, 0, 0, 0], dtype=torch.int32)))
    assert pipe.n == n0 and all(sl.inp is None for sl in pipe.slots)         # nothing was enqueued
    pipe.set_vehicles(_vehicles(torch, 2))                                   # fewer vehicles now: index 2 is out of range
    with pytest.raises(ValueError):
        pipe.submit(steps[0])
    assert all(sl.inp is None for sl in pipe.slots)
