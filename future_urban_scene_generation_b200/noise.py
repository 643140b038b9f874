"""The VUNet Sampler noise drawn on the device, bit-identical to `torch.randn` on torch's CPU generator.

The reference draws each Sampler's noise with `torch.randn(b, c, h, w)` on the CPU default generator (vunet/layers.py:166),
in eval mode too.  `randn_cpu_exact` gives the same tensors -- and leaves the generator in the same state -- with the
normals made by csrc/noise.cu on the GPU: the host only reads the 624-word MT19937 state, ships 2.5 KB and advances the
generator past the draw (`fusg_mt19937_advance`, twists only).  It covers what the Sampler shapes need: contiguous fp32
draws with numel a positive multiple of 16, mean 0, std 1 (DESIGN.md §4.8).

    eps, = randn_cpu_exact([(B, 128, 8, 8)], layout="nhwc")       # == torch.randn(B, 128, 8, 8).permute(0, 2, 3, 1)
    with engine.noise_from(device_provider()):                    # eager engine calls draw their noise this way
        ...

The first draw on each device checks itself against `torch.randn` on a copy of a generator and raises `FusgError` if the
two differ; there is no silent fall-back to the host draw.
"""
import ctypes as C
import threading

import numpy as np
import torch

from . import _lib

MT_N = 624
STATE_BYTES = 5056            # CPUGeneratorImpl::get_state: u64 seed, i32 left, i32 seeded, u64 next, u64 words[624], ...
MAX_DRAWS = 16                # FUSG_RANDN_MAX_DRAWS
LAYOUTS = ("nchw", "nhwc")


class RandnDraw(C.Structure):
    """fusg_randn_draw (include/fusg.h)."""
    _fields_ = [("out", C.c_void_p), ("b", C.c_int32), ("c", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("nhwc", C.c_int32), ("reserved", C.c_int32)]


def check_shapes(shapes):
    """[(b, c, h, w), ...] -> list of int 4-tuples; ValueError for what torch would draw another way."""
    shapes = [tuple(int(d) for d in s) for s in shapes]
    if not 0 < len(shapes) <= MAX_DRAWS:
        raise ValueError(f"randn_cpu_exact: 1..{MAX_DRAWS} draws per call, got {len(shapes)}")
    for s in shapes:
        if len(s) != 4 or min(s) <= 0:
            raise ValueError(f"randn_cpu_exact: draw shape {s} is not a positive (b, c, h, w)")
        n = s[0] * s[1] * s[2] * s[3]
        if n < 16 or n % 16:
            raise ValueError(f"randn_cpu_exact: draw {s} has numel {n}; only positive multiples of 16 are covered "
                             "(torch.randn takes another path for the others)")
    return shapes


def _layout_shape(s, nhwc):
    b, c, h, w = s
    return (b, h, w, c) if nhwc else (b, c, h, w)


def parse_state(state):
    """5056-byte generator state -> (words u32[624], left, next)."""
    b = state.numpy().tobytes()
    if len(b) != STATE_BYTES:
        raise _lib.FusgError(f"CPU generator state is {len(b)} bytes, this module knows the {STATE_BYTES}-byte layout")
    left = int(np.frombuffer(b, np.int32, 1, 8)[0])
    nxt = int(np.frombuffer(b, np.uint64, 1, 16)[0])
    return np.frombuffer(b, np.uint64, MT_N, 24).astype(np.uint32), left, nxt


def advance(words, left, nxt, n):
    """Position n words after (words, left, next), on the host: (words, left, next)."""
    src = np.ascontiguousarray(words, dtype=np.uint32)
    out = np.empty(MT_N, np.uint32)
    lo, no = C.c_int(), C.c_longlong()
    _lib.check(_lib.lib().fusg_mt19937_advance(src.ctypes.data, int(left), int(nxt), int(n), out.ctypes.data, C.byref(lo),
                                               C.byref(no)), "fusg_mt19937_advance")
    return out, lo.value, no.value


def _with_position(state, words, left, nxt):
    """`state` with its MT19937 words and position replaced; seed and cached normal samples kept."""
    s = state.clone()
    v = s.numpy()
    v[8:12] = np.frombuffer(np.int32(left).tobytes(), np.uint8)
    v[16:24] = np.frombuffer(np.uint64(nxt).tobytes(), np.uint8)
    v[24:24 + 8 * MT_N] = np.frombuffer(words.astype(np.uint64).tobytes(), np.uint8)
    return s


class DrawPlan:
    """A fixed list of draws into fixed device tensors: what one step of a captured graph generates.

    `take(generator)` (host) copies the generator's position into a pinned start buffer and advances the generator past
    the draws, as torch.randn would; `upload()` copies that start state to the device on the current stream; `launch()`
    enqueues the generation on the current stream, reading the device start state -- so a graph that captured `launch()`
    draws fresh noise on every replay after a `take` + `upload`."""

    def __init__(self, outs, shapes, nhwc, device):
        shapes = check_shapes(shapes)
        if len(outs) != len(shapes):
            raise ValueError("DrawPlan: one output tensor per draw")
        for t, s in zip(outs, shapes):
            if (t.dtype != torch.float32 or not t.is_cuda or not t.is_contiguous() or t.device != torch.device(device)
                    or tuple(t.shape) != _layout_shape(s, nhwc)):
                raise ValueError(f"DrawPlan: output for draw {s} must be a contiguous fp32 {_layout_shape(s, nhwc)} tensor on {device}")
        self.outs = list(outs)
        self.words = sum(s[0] * s[1] * s[2] * s[3] for s in shapes)
        self.table = (RandnDraw * len(shapes))()
        for e, t, (b, c, h, w) in zip(self.table, outs, shapes):
            e.out, e.b, e.c, e.h, e.w, e.nhwc = t.data_ptr(), b, c, h, w, int(nhwc)
        self.start_host = torch.empty(MT_N + 2, dtype=torch.int32).pin_memory()
        self.start_dev = torch.zeros(MT_N + 2, dtype=torch.int32, device=device)      # until an upload: left = 0, NaN noise

    def take(self, generator=None):
        g = torch.default_generator if generator is None else generator
        state = g.get_state()
        words, left, nxt = parse_state(state)
        v = self.start_host.numpy().view(np.uint32)
        v[:MT_N] = words
        v[MT_N], v[MT_N + 1] = left, nxt
        g.set_state(_with_position(state, *advance(words, left, nxt, self.words)))

    def upload(self):
        self.start_dev.copy_(self.start_host, non_blocking=True)

    def launch(self):
        _lib.check(_lib.lib().fusg_randn_mt19937(_lib.ptr(self.start_dev), self.table, len(self.table), _lib.stream_ptr(torch)),
                   "fusg_randn_mt19937")


def _randn(shapes, nhwc, generator, device, out):
    with torch.cuda.device(device):
        if out is None:
            out = [torch.empty(_layout_shape(s, nhwc), dtype=torch.float32, device=device) for s in shapes]
        plan = DrawPlan(out, shapes, nhwc, device)
        plan.take(generator)
        plan.upload()
        plan.launch()
    return list(out)


_checked = set()
_check_lock = threading.Lock()


def self_check(device, expected=None):
    """Draws two small tensors (mid-block start, both layouts) on `device` and compares them bit for bit, and the generator
    state after them, with `torch.randn` on a copy of the same generator -- or with `expected`, a list of the two NCHW
    tensors, which lets a test hand it a wrong draw.  Raises FusgError on any difference."""
    device = torch.device(device)
    g = torch.Generator()
    g.manual_seed(20240607)
    torch.randn(37, generator=g)                                 # a start in the middle of a 624-word block
    shapes = [(2, 3, 8, 8), (1, 16, 5, 3)]
    ref_g = torch.Generator()
    ref_g.set_state(g.get_state())
    ref = [torch.randn(*s, generator=ref_g) for s in shapes]
    if expected is None:
        expected = ref
    bad = []
    for nhwc in (False, True):
        gd = torch.Generator()
        gd.set_state(g.get_state())
        got = [t.cpu() for t in _randn(shapes, nhwc, gd, device, None)]
        for s, t, e in zip(shapes, got, expected):
            t = t.permute(0, 3, 1, 2) if nhwc else t
            if not torch.equal(t.contiguous().view(torch.int32), e.contiguous().view(torch.int32)):
                bad.append(f"{LAYOUTS[nhwc]} draw {s}")
        if not torch.equal(gd.get_state(), ref_g.get_state()):
            bad.append(f"generator state after the {LAYOUTS[nhwc]} draws")
    if bad:
        raise _lib.FusgError(
            f"device Sampler noise on {device} differs from torch.randn on this host ({', '.join(bad)}); torch's CPU "
            f"capability here is {torch.backends.cpu.get_cpu_capability()!r}.  Use the host noise (noise='host').")


def ensure_checked(device):
    """self_check once per process and device."""
    device = torch.device(device)
    with _check_lock:
        if device not in _checked:
            self_check(device)
            _checked.add(device)


def _device(device):
    if device is None:
        _lib.require_cuda()
        return torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if device.type != "cuda":
        raise ValueError(f"randn_cpu_exact: device must be a CUDA device, got {device}")
    return torch.device("cuda", torch.cuda.current_device() if device.index is None else device.index)


def randn_cpu_exact(shapes, layout="nchw", generator=None, device=None, out=None):
    """`[torch.randn(*s, generator=generator) for s in shapes]`, made on `device` (default: the current CUDA device) in
    `layout` "nchw" (as torch.randn) or "nhwc" (as the Sampler epilogues read it), into `out` if given.  The generator
    (default: the global CPU generator) ends where torch.randn would leave it, before the device has drawn anything.
    The draws are enqueued on the device's current stream."""
    if layout not in LAYOUTS:
        raise ValueError(f"randn_cpu_exact: layout must be one of {LAYOUTS}, got {layout!r}")
    shapes = check_shapes(shapes)
    device = _device(device)
    ensure_checked(device)
    return _randn(shapes, layout == "nhwc", generator, device, out)


def device_provider(generator=None, device=None):
    """A noise provider for `VunetEngine.noise_from`: each Sampler's (B, C, H, W) draw made on the device, NHWC."""
    def provide(b, c, h, w):
        return randn_cpu_exact([(b, c, h, w)], layout="nhwc", generator=generator, device=device)[0]
    return provide
