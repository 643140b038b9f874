"""The CPU side of the device Sampler noise: the numpy restatement of torch.randn (oracle/noise_oracle.py) against torch
itself, the generator state layout, the host advance fusg_mt19937_advance and argument checks."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import noise_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sampler_shapes(B, form="forward"):
    """The Sampler draws in the reference's order: enc_down's two, then dec_down's 4 + 4 (auto-regressive blocks)."""
    enc = [(B, 128, 4, 4), (B, 128, 8, 8)]
    dec = [(B, 128, 2, 2)] * 4 + [(B, 128, 4, 4)] * 4
    return {"forward": enc + dec, "enc": enc, "step": dec}[form]


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _check_against_torch(g, shapes):
    s0 = g.get_state()
    ref = [torch.randn(*s, generator=g).numpy() for s in shapes]
    got, s1 = O.randn(shapes, s0)
    for s, a, b in zip(shapes, got, ref):
        assert _same_bits(a, b), s
    assert torch.equal(s1, g.get_state())


def test_oracle_equals_torch_randn_over_100_seeds():
    for seed in range(100):
        g = torch.Generator()
        g.manual_seed(seed)
        _check_against_torch(g, sampler_shapes(1))


@pytest.mark.parametrize("B", [1, 5, 64])
def test_oracle_equals_torch_randn_at_every_sampler_shape(B):
    g = torch.Generator()
    g.manual_seed(1000 + B)
    _check_against_torch(g, sampler_shapes(B, "forward") + sampler_shapes(B, "step"))


def test_oracle_starts_mid_block():
    for odd in (1, 7, 33, 623, 625, 1000):         # odd-sized earlier draws leave the position anywhere in a block
        g = torch.Generator()
        g.manual_seed(odd)
        torch.randn(odd, generator=g)
        _check_against_torch(g, [(2, 16, 3, 3), (1, 128, 4, 4)])


_CAPABILITY_SCRIPT = r"""
import sys, torch, numpy as np
sys.path.insert(0, sys.argv[1])
from oracle import noise_oracle as O
bad = 0
for seed in range(8):
    g = torch.Generator(); g.manual_seed(seed); torch.randn(5 + seed, generator=g)
    s0 = g.get_state()
    shapes = [(5, 128, 4, 4), (5, 128, 8, 8), (3, 16, 7, 9)]
    ref = [torch.randn(*s, generator=g).numpy() for s in shapes]
    got, s1 = O.randn(shapes, s0)
    bad += sum(int((a.view(np.uint32) != b.view(np.uint32)).sum()) for a, b in zip(got, ref))
    bad += int(not torch.equal(s1, g.get_state()))
print(torch.backends.cpu.get_cpu_capability(), bad)
"""


@pytest.mark.parametrize("capability", [None, "avx2"])
def test_oracle_equals_torch_under_each_cpu_capability(capability):
    env = dict(os.environ)
    env.pop("ATEN_CPU_CAPABILITY", None)
    if capability:
        env["ATEN_CPU_CAPABILITY"] = capability
    out = subprocess.run([sys.executable, "-c", _CAPABILITY_SCRIPT, ROOT], env=env, capture_output=True, text=True, check=True)
    cap, bad = out.stdout.split()
    if capability:
        assert cap.lower() == capability
    assert bad == "0", out.stdout


def test_transform_on_both_ends_of_the_uniform_range():
    """u = 0 (u1 = 1, log 0) and u = 1 - 2^-24 (the smallest u1, the largest theta) as torch makes them: a generator
    state whose next words temper to 0 and to 0xFFFFFF is hard to reach, so check the transform's own invariants."""
    u = np.array([0.0] * 8 + [0.0] * 8 + [1 - 2.0 ** -24] * 8 + [1 - 2.0 ** -24] * 8, np.float32)
    out = O.box_muller(u)
    assert np.all(np.isfinite(out))
    assert np.all(out[:16] == 0) and not np.signbit(out[:16]).any()    # radius 0; -0 becomes +0 through fmadd(n, 1, 0)
    assert np.abs(out[16:]).max() < 6.0


def test_state_parse_and_build_round_trip():
    g = torch.Generator()
    g.manual_seed(42)
    torch.randn(3, generator=g)                     # < 16 elements: torch caches a double normal sample in the state
    s = g.get_state()
    words, left, nxt = O.parse_state(s)
    assert len(bytes(s.numpy())) == O.STATE_BYTES
    assert torch.equal(O.build_state(s, words, left, nxt), s)
    w2, l2, n2 = O.advance(words, left, nxt, 777)
    g2 = torch.Generator()
    g2.set_state(O.build_state(s, w2, l2, n2))      # torch accepts the built state, and it is where 777 words of
    torch.rand(777, generator=g)                    # torch's own fp32 uniforms (one word each) leave the generator
    assert torch.equal(g2.get_state(), g.get_state())


def test_seeded_state_layout():
    g = torch.Generator()
    g.manual_seed(1)
    words, left, nxt = O.parse_state(g.get_state())
    assert list(words[:3]) == [1, 1812433254, 3713160357] and (left, nxt) == (1, 0)
    torch.randn(32, generator=g)
    assert O.parse_state(g.get_state())[1:] == (593, 32)


def test_host_advance_equals_the_oracle():
    from future_urban_scene_generation_b200 import noise as N
    g = torch.Generator()
    g.manual_seed(3)
    torch.randn(45, generator=g)
    words, left, nxt = N.parse_state(g.get_state())
    for n in (0, 1, left - 2, left - 1, left, 624, 625, 5000, 1310720 + 7):   # the last crosses ~2100 twists
        a = N.advance(words, left, nxt, n)
        b = O.advance(words, left, nxt, n)
        assert np.array_equal(a[0], b[0]) and a[1:] == b[1:], n
    w1, l1, n1 = N.advance(*N.advance(words, left, nxt, 1000), 2345)
    w2, l2, n2 = N.advance(words, left, nxt, 3345)
    assert np.array_equal(w1, w2) and (l1, n1) == (l2, n2)


def test_host_advance_refuses_a_position_torch_never_reaches():
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    s = np.zeros(624, np.uint32)
    o = np.zeros(624, np.uint32)
    lo, no = ctypes.c_int(), ctypes.c_longlong()
    for left, nxt, n in ((0, 0, 1), (625, 0, 1), (10, 620, 1), (5, 1, -1)):
        assert L.fusg_mt19937_advance(s.ctypes.data, left, nxt, n, o.ctypes.data, ctypes.byref(lo), ctypes.byref(no)) == -1


def test_bad_shapes_raise_value_error():
    from future_urban_scene_generation_b200 import noise as N
    for shapes in ([(1, 1, 2, 4)], [(1, 3, 5, 1)], [(2, 128, 4)], [(0, 128, 4, 4)], [], [(1, 16, 1, 1)] * 17):
        with pytest.raises(ValueError):
            N.randn_cpu_exact(shapes)
    for shapes in ([(1, 1, 2, 4)], [(1, 3, 5, 1)]):
        with pytest.raises(ValueError):
            O.check_shapes(shapes)
    with pytest.raises(ValueError):
        N.randn_cpu_exact([(1, 16, 1, 1)], layout="nhcw")


def test_entry_point_validates_its_arguments():
    from future_urban_scene_generation_b200 import _lib, noise as N
    L = _lib.lib()
    assert L.fusg_sizeof_randn_draw() == ctypes.sizeof(N.RandnDraw) == 32
    fake = ctypes.c_void_p(0x100000)

    def table(*shapes, nhwc=0, out=0x100000):
        t = (N.RandnDraw * len(shapes))()
        for e, (b, c, h, w) in zip(t, shapes):
            e.out, e.b, e.c, e.h, e.w, e.nhwc = out, b, c, h, w, nhwc
        return t
    assert L.fusg_randn_mt19937(fake, table((1, 3, 5, 1)), 1, None) == -2          # numel 15
    assert L.fusg_randn_mt19937(fake, table((1, 8, 3, 1)), 1, None) == -2          # numel 24: not a multiple of 16
    assert L.fusg_randn_mt19937(fake, table((1, 16, 1, 1), nhwc=2), 1, None) == -1
    assert L.fusg_randn_mt19937(fake, table((1, 16, 1, 1), out=0x100002), 1, None) == -1   # misaligned output
    assert L.fusg_randn_mt19937(fake, table((0, 16, 1, 1)), 1, None) == -1
    assert L.fusg_randn_mt19937(fake, table(*[(1, 16, 1, 1)] * 17), 17, None) == -1
    assert L.fusg_randn_mt19937(None, table((1, 16, 1, 1)), 1, None) == -1
