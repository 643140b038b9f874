"""CPU suite, part 2: host logic and the C-ABI boundary (no compute calls without a GPU)."""
import ctypes
import hashlib
import json
import os
import re
from argparse import Namespace

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the original Python project (alexj94/future_urban_scene_generation), if one is at hand
REFERENCE = os.environ.get("FUSG_REFERENCE_DIR", "")


def test_library_exports_every_declared_symbol():
    from future_urban_scene_generation_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "fusg.h")).read()
    names = sorted(set(re.findall(r"\b(fusg_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 15
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), n
    L = _lib.lib()
    assert L.fusg_version() >= 100
    assert L.fusg_warp_workspace_bytes(3) == 3 * 5 * 9 * 8 + (4 + 6 * 3) * 4 + 3 * 5 * 56   # Minv | counters[4] | list6[2B] | list4[3B] | big_list[B] | PlaneRec[B,5]
    assert L.fusg_kernel_launches() >= 0


def test_ctypes_struct_matches_c_layout():
    from future_urban_scene_generation_b200 import _lib
    from future_urban_scene_generation_b200.vunet.engine import ConvDesc, ConvOut
    assert ctypes.sizeof(ConvOut) == 32
    assert ctypes.sizeof(ConvDesc) == _lib.lib().fusg_sizeof_conv_desc()


def test_argument_validation_without_gpu():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    assert L.fusg_warp_fused(None, None, None, None, None, None, None, None, None, None, None, None, 0, 1, 256, 256, None) == -1
    assert L.fusg_conv2d(None, None) == -1
    assert L.fusg_visibility(None, None, None, None, None, None, 1, 256, 256, None) == -1
    assert L.fusg_find_homography(None, None, 4, None, None, 1, None) == -1


def test_vunet_module_checkpoint_contract():
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from future_urban_scene_generation_b200._lib import FusgError
    m = Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True))
    sd = m.state_dict()
    keys = list(sd.keys())
    assert len(keys) == 336
    assert hashlib.sha1("\n".join(keys).encode()).hexdigest() == "6a36f5dfc3dc8ab32fb79a78d759d8d28e09d940"   # SURVEY.md §8a
    assert keys[:3] == ["app_encoder_1.nin.layers.1.conv.bias", "app_encoder_1.nin.layers.1.conv.weight_g", "app_encoder_1.nin.layers.1.conv.weight_v"]
    assert sd["shape_decoder_1.residual_0.layers.2.conv.weight_v"].shape == (512, 1024, 3, 3)
    assert sd["shape_decoder_6.conv.conv.weight_g"].shape == (3, 1, 1, 1)
    assert sum(v.numel() for v in sd.values()) == 45225158
    # weight_norm initialisation: g = ||v||
    v, g = sd["app_bottleneck.conv.weight_v"], sd["app_bottleneck.conv.weight_g"]
    assert torch.allclose(v.flatten(1).norm(dim=1), g.flatten())
    from oracle import vunet_oracle as VO
    res = m.load_state_dict(VO.make_state_dict(3), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    bad = dict(VO.make_state_dict(3))
    bad.pop("app_bottleneck.conv.bias")
    with pytest.raises(RuntimeError):
        m.load_state_dict(bad, strict=True)
    with pytest.raises(NotImplementedError):
        Vunet_fix_res(Namespace(up_mode='conv2d_t', w_norm=True, drop_prob=0.2, vunet_256=True))
    with pytest.raises(NotImplementedError):
        Vunet_fix_res(Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=False))
    # no CPU fallback: a CPU module refuses to run
    with pytest.raises(FusgError):
        m.eval()(torch.zeros(1, 3, 256, 256), torch.zeros(1, 6, 256, 256))
    # training mode (active Dropout2d) is refused, not silently different
    if torch.cuda.is_available():
        with pytest.raises(NotImplementedError):
            m.cuda().train()(torch.zeros(1, 3, 256, 256).cuda(), torch.zeros(1, 6, 256, 256).cuda())


def test_icn_module_checkpoint_contract():
    """SURVEY.md 8b: G_Resnet(21) keeps the reference's 40-key state_dict (order, shapes) and refuses to run on the CPU."""
    from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
    from future_urban_scene_generation_b200._lib import FusgError
    from oracle import icn_oracle as IO
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "icn_golden.json")))
    m = G_Resnet(21)
    sd = m.state_dict()
    keys = list(sd.keys())
    assert len(keys) == gold["n_keys"] == 40
    assert hashlib.sha1("\n".join(keys).encode()).hexdigest() == gold["key_sha1"]
    assert keys[0] == "enc_content.model.0.conv.weight" and keys[-1] == "dec.model.5.conv.bias"
    assert keys.index("dec.model.2.norm.gamma") < keys.index("dec.model.2.conv.weight")      # Conv2dBlock builds its norm first
    assert sd["dec.model.4.conv.weight"].shape == (64, 128, 5, 5) and sd["enc_content.model.2.conv.weight"].shape == (256, 128, 4, 4)
    assert sum(v.numel() for v in sd.values()) == gold["n_params"]
    assert float(sd["dec.model.2.norm.beta"].abs().max()) == 0.0 and 0.0 <= float(sd["dec.model.2.norm.gamma"].min())
    res = m.load_state_dict(IO.make_state_dict(3), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    bad = dict(IO.make_state_dict(3))
    bad.pop("dec.model.5.conv.bias")
    with pytest.raises(RuntimeError):
        m.load_state_dict(bad, strict=True)
    with pytest.raises(NotImplementedError):
        G_Resnet(21, norm='batch')
    with pytest.raises(FusgError):
        m.eval()(torch.zeros(1, 21, 64, 64))
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 21, 30, 30))


def test_kinematics_host_mirror():
    """trajectory_poses mirrors trajectory_inference.py:258-298: rotation always by theta, translation gated at +-20 degrees."""
    from future_urban_scene_generation_b200 import kinematics as KM
    mc = np.array([[0, 0], [1, 0], [2, 0], [3, 0.1], [4, 0.1], [5, 0.2]], np.float64)
    theta, tr, rot = KM.trajectory_poses(mc)
    assert theta.shape == (5,) and tr.shape == (5, 3) and rot.shape == (5, 3, 3) and rot.dtype == np.float32
    assert np.allclose(np.linalg.norm(tr, axis=1), np.linalg.norm(mc[1:] - mc[0], axis=1), rtol=1e-6)
    assert np.array_equal(rot[2], KM.z_rot(theta[2])) and np.all(tr[:, 2] == 0)
    # a hairpin: heading differs from the start heading by > 20 degrees -> translation along -y unrotated (z_rot(0))
    hair = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], np.float64)
    th, tr2, _ = KM.trajectory_poses(hair)
    assert abs(np.degrees(th[-1])) > 20 and tr2[-1, 0] == 0 and tr2[-1, 1] == -np.linalg.norm(hair[3] - hair[0])
    with pytest.raises(ValueError):
        KM.trajectory_poses(np.zeros((1, 2)))
    L = __import__("future_urban_scene_generation_b200._lib", fromlist=["lib"]).lib()
    assert L.fusg_step_keypoints(None, None, None, None, None, None, None, None, None, None, 1, 256, 256, None) == -1
    assert L.fusg_norm_stats(None, None, 1, 1, 8, 1, 0, None) == -1


def test_warp_mirror_surface_and_constants():
    from future_urban_scene_generation_b200.warp_learn import online_visibility as ov, planes_utils as pu
    assert list(ov.pascal_texture_planes['car'].keys()) == ['left', 'right', 'roof', 'front', 'back']
    assert [len(v) for v in ov.pascal_texture_planes['car'].values()] == [6, 6, 4, 4, 4]
    assert ov.pascal_texture_planes['chair'] == {}
    for fn in (ov.compute_visibility, pu.get_planes, pu.warp_unwarp_planes, pu.planes_to_torch, pu.to_image):
        assert callable(fn)
    # host-side pieces that need no GPU
    x = torch.linspace(-1.2, 1.2, 3 * 4 * 5).view(3, 4, 5)
    img = pu.to_image(x, from_LAB=False)
    want = np.clip((np.transpose(x.numpy(), (1, 2, 0)) + 1.) / 2 * 255, 0, 255).astype(np.uint8)
    assert img.dtype == np.uint8 and np.array_equal(img, want)
    planes = np.random.default_rng(0).integers(0, 256, (5, 8, 8, 3), dtype=np.uint8)
    t = pu.planes_to_torch(planes, to_LAB=False)
    assert t.shape == (5, 3, 8, 8) and t.dtype == torch.float32
    assert torch.allclose(t, (torch.from_numpy(np.transpose(np.float32(planes) / 255., (0, 3, 1, 2))) - 0.5) / 0.5)
    with pytest.raises(ValueError):
        ov._extrinsic34(np.ones((4, 4)))
    if not torch.cuda.is_available():
        from future_urban_scene_generation_b200._lib import FusgError
        with pytest.raises(FusgError):
            ov.compute_visibility(np.eye(4), np.eye(3), {k: np.zeros(3) for k in ov._KP_NAMES}, 256, 256)


def test_synthetic_inputs_are_deterministic_and_in_frame():
    from future_urban_scene_generation_b200 import synth
    a, b = synth.make_warp_batch(5, 6), synth.make_warp_batch(5, 6)
    for k in a:
        assert np.array_equal(a[k], b[k])
    assert a["src"].shape == (6, 256, 256, 3) and a["src_kp"].dtype == np.int32
    for k in ("src_kp", "dst_kp"):
        assert a[k].min() >= 0 and a[k].max() <= 255
    x, y = synth.make_vunet_inputs(0, 2)
    assert x.shape == (2, 6, 256, 256) and y.shape == (2, 3, 256, 256) and x.dtype == np.float32
    assert -1.0 <= x.min() and x.max() <= 1.0


def test_shard_range_partitions_contiguously():
    from future_urban_scene_generation_b200.parallel import shard_range
    for n in (0, 1, 7, 64, 4096, 4099):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for (b0, e0), (b1, e1) in zip(spans, spans[1:]):
                assert e0 == b1
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


def _gloo_worker(rank, world, port, n_total, q):
    import torch.distributed as dist
    from future_urban_scene_generation_b200.parallel import shard_range, gather_crops
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    full = torch.arange(n_total * 4 * 4 * 3, dtype=torch.int64).remainder(251).to(torch.uint8).view(n_total, 4, 4, 3)
    b, e = shard_range(n_total, rank, world)
    out = gather_crops(full[b:e].clone(), n_total)
    q.put((rank, bool(torch.equal(out, full))))
    dist.destroy_process_group()


@pytest.mark.parametrize("n_total", [8, 7])
def test_gather_crops_world_size_2_gloo(n_total):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 400) + n_total
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, n_total, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    res = dict(q.get(timeout=10) for _ in range(2))
    assert res == {0: True, 1: True}


def test_import_shim_serves_reference_import_sites():
    """INTEGRATION.md §1: with the shim first on sys.path the reference's own import statements
    resolve to the B200 modules (and, where the reference checkout is present, its untouched
    submodules keep resolving to the reference)."""
    import subprocess
    import sys
    shim = os.path.join(ROOT, "future_urban_scene_generation_b200", "shim")
    ref = REFERENCE
    code = (
        "import sys, warnings; warnings.filterwarnings('ignore');"
        f"sys.path[:0] = [{ROOT!r}, {shim!r}];"
        + (f"sys.path.append({ref!r});" if os.path.isdir(ref) else "")
        + "from vunet.models import Vunet_fix_res;"
        "from warp_learn.online_visibility import pascal_texture_planes, compute_visibility;"
        "from warp_learn.planes_utils import to_image, warp_unwarp_planes, get_planes, planes_to_torch;"
        "assert Vunet_fix_res.__module__.startswith('future_urban_scene_generation_b200');"
        "assert get_planes.__module__.startswith('future_urban_scene_generation_b200');"
        + "from warp_learn.models import G_Resnet;"
        "assert G_Resnet.__module__.startswith('future_urban_scene_generation_b200');"
        + "from warp_learn.models import get_icn_inputs;"
        "assert get_icn_inputs.__module__.startswith('future_urban_scene_generation_b200');"
        + ("from warp_learn.models import get_icn_inputs_reference, G_Resnet_reference, GANLoss; import warp_learn.models as wm;"
           f"assert get_icn_inputs_reference.__code__.co_filename.startswith({ref!r});"
           "assert wm.planes_to_torch.__module__.startswith('future_urban_scene_generation_b200');" if os.path.isdir(ref) else "")
        + "print('ok')")
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]


def test_reference_orchestrator_imports_through_the_shim():
    """The reference's own orchestrator module (`trajectory_inference.py`, unedited, from the checkout FUSG_REFERENCE_DIR
    names; skipped without one) imports with the shim first on sys.path: every hot-path name it binds -- get_icn_inputs,
    pascal_texture_planes, to_image, warp_unwarp_planes, and through the reference's own vehicle_utils:
    compute_visibility, get_planes, get_rendered (the Open3D window) -- resolves to the B200 modules.  open3d /
    matplotlib / skimage are stubbed.  (Running traj_test itself needs a GPU as well as the checkout.)"""
    import subprocess
    import sys
    ref = REFERENCE
    if not os.path.isdir(ref):
        pytest.skip("needs a checkout of the original project: set FUSG_REFERENCE_DIR")
    shim = os.path.join(ROOT, "future_urban_scene_generation_b200", "shim")
    code = r"""
import sys, types, warnings
warnings.filterwarnings('ignore')
sys.path[:0] = [%r, %r]
sys.path.append(%r)
def stub(name, **attrs):
    m = types.ModuleType(name); m.__dict__.update(attrs); sys.modules[name] = m; return m
o3d = stub('open3d')
o3d.geometry = stub('open3d.geometry', TriangleMesh=object)
o3d.utility = stub('open3d.utility', Vector3dVector=lambda a: a)
o3d.visualization = stub('open3d.visualization')
o3d.io = stub('open3d.io')
mpl = stub('matplotlib'); mpl.pyplot = stub('matplotlib.pyplot'); mpl.cm = stub('matplotlib.cm'); mpl.colors = stub('matplotlib.colors')
sk = stub('skimage'); sk.feature = stub('skimage.feature', canny=None); sk.color = stub('skimage.color', rgb2gray=None)
import trajectory_inference as ti
ours = 'future_urban_scene_generation_b200'
for name in ('get_icn_inputs', 'to_image', 'warp_unwarp_planes'):
    assert getattr(ti, name).__module__.startswith(ours), name
import warp_learn.online_visibility as ov
assert ti.pascal_texture_planes is ov.pascal_texture_planes and ov.__name__ and ov.compute_visibility.__module__.startswith(ours)
g = ti.get_vehicle_information.__globals__                      # the REFERENCE's vehicle_utils, served through the shim package path
assert ti.get_vehicle_information.__code__.co_filename.startswith(%r)
for name in ('compute_visibility', 'get_planes', 'get_rendered'):
    assert g[name].__module__.startswith(ours), name
print('ok')
""" % (ROOT, shim, ref, ref)
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-3000:]
