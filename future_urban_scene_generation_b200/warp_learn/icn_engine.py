"""Execution engine of the ICN generator forward on libfusg.so (SURVEY.md section 8f-1).

The network of warp_learn/models.py:128-208 (reference: ContentEncoder -> ResBlocks -> Decoder) is run as a flat
sequence of launches on NHWC activations:

    conv      fusg_conv2d with pad_mode = 1: the ReflectionPad2d of every Conv2dBlock (models.py:43-44,86) is *stored* in
              the input tensor's own border, so the implicit-GEMM kernel reads it with plain in-bounds TMA boxes
              (7x7, 4x4 stride 2, 3x3, 5x5; bias in the epilogue, tanh for the last block)
    stats     fusg_norm_stats + fusg_norm_finalize: InstanceNorm2d / the reference's LayerNorm (models.py:15-35,55-58)
              as per-(sample, channel) scale / shift pairs
    apply     fusg_norm_apply: normalise + ReLU + ResBlock residual (models.py:98-102) + nearest 2x upsample
              (models.py:138-147) + the reflection border of the NEXT convolution, one pass over the tensor

dtype 'fp16' is the product path: tcgen05 kernels (power-of-two frame sizes) on fp16 activations / weights with fp32
accumulation.  Every activation of this network is InstanceNorm / LayerNorm-bounded, so fp16's range is ample, and its
11-bit significand keeps the 18-layer stack at ~2e-3 max-abs from the fp32 reference, where bf16 operands alone put a
floor of ~1.1e-2 under it (tests/test_icn_gpu.py; same tensor-core rate).  dtype 'bf16' runs the identical program on
bf16; dtype 'fp32' runs it on the CUDA-core direct kernel (verification build, <= 1e-4).
"""
import ctypes as C

from .. import _lib
from ..vunet.engine import ConvDesc, DT_BF16, DT_F32, IMPL_AUTO, IMPL_TC, IMPL_DIRECT

DT_F16 = 2

EPS = 1e-5


def _pad16(c):
    return (c + 15) // 16 * 16


class Padded:
    """NHWC device tensor [B, H + 2*border, W + 2*border, C] holding an H x W image plus its reflection border."""
    __slots__ = ("t", "H", "W", "C", "border")

    def __init__(self, t, H, W, C_, border):
        self.t, self.H, self.W, self.C, self.border = t, H, W, C_, border


class IcnEngine:
    def __init__(self, module, dtype="fp16", impl="auto"):
        assert dtype in ("fp16", "bf16", "fp32")
        self.m = module
        self.dtype = dtype
        self.impl = {"auto": IMPL_AUTO, "tcgen05": IMPL_TC, "direct": IMPL_DIRECT}[impl]
        self._wkey = None
        self._w = {}
        self.launches = 0
        self.profile = None        # list -> (name, kind, flops_or_bytes, start event, end event)

    # ------------------------------------------------------------------ plumbing
    @property
    def torch(self):
        return _lib.require_cuda()

    @property
    def tdtype(self):
        torch = self.torch
        return {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}[self.dtype]

    @property
    def cdtype(self):
        return {"fp16": DT_F16, "bf16": DT_BF16, "fp32": DT_F32}[self.dtype]

    def device(self):
        return next(self.m.parameters()).device

    def _stream(self):
        return _lib.stream_ptr(self.torch)

    def _empty(self, *shape, dtype=None):
        return self.torch.empty(shape, dtype=dtype or self.tdtype, device=self.device())

    def _timed(self, name, kind, amount, fn):
        prof = self.profile
        if prof is None:
            fn()
        else:
            torch = self.torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            prof.append((name, kind, amount, e0, e1))
        self.launches += 1

    # ------------------------------------------------------------------ weights
    def prepare_weights(self, force=False):
        """[cout][cin][k][k] fp32 -> [cout_pad][k*k][cin_pad] in the activation dtype, once per (re)load."""
        key = tuple((p.data_ptr(), p._version) for p in self.m.parameters())
        if not force and key == self._wkey:
            return
        torch = self.torch
        dev = self.device()
        if dev.type != "cuda":
            raise _lib.FusgError("G_Resnet: parameters are not on a CUDA device; the B200 path has no CPU fallback (call .to('cuda'))")
        self._w = {}
        self._kwide = {}
        for path, blk in self.m.blocks.items():
            w = blk.conv.weight.detach().float()
            cout, cin, k, _ = w.shape
            cin_pad = 32 if cin < 32 else cin          # the 21-channel input: one 64-byte swizzle span
            # K of a narrow-input layer is widened to 64 (TMA zero-fills beyond the 32 stored channels, fusg_conv_desc.cphys0):
            # twice the tensor work, but a 64-channel k-block is what the sliding-window A tiles need -- one row-segment load
            # per (tile, ky) instead of a load per tap (49 for the 7x7 first layer)
            kwide = 64 if cin_pad == 32 and k >= 5 else cin_pad
            cout_pad = _pad16(cout)
            wp = torch.zeros((cout_pad, k * k, kwide), dtype=torch.float32, device=dev)
            wp[:cout, :, :cin] = w.permute(0, 2, 3, 1).reshape(cout, k * k, cin)
            bias = torch.zeros((cout_pad,), dtype=torch.float32, device=dev)
            bias[:cout] = blk.conv.bias.detach().float()
            gamma = beta = None
            if blk.norm is not None:
                gamma, beta = blk.norm.gamma.detach().float().contiguous(), blk.norm.beta.detach().float().contiguous()
            self._w[path] = (wp.to(self.tdtype).contiguous(), bias, cout, cout_pad, cin, cin_pad, k, gamma, beta)
            self._kwide[path] = kwide
        self._wkey = key

    # ------------------------------------------------------------------ launches
    def to_padded(self, x_nchw, border, cpad=None):
        """Foreign NCHW fp32 tensor -> reflection-bordered NHWC activation."""
        t = x_nchw.detach()
        if t.device != self.device():
            t = t.to(self.device())
        t = t.float().contiguous()
        B, Cn, H, W = t.shape
        cp = cpad or Cn
        out = self._empty(B, H + 2 * border, W + 2 * border, cp)
        L = _lib.lib()
        self._timed("nchw_to_nhwc_reflect", "bytes", t.numel() * 4 + out.numel() * out.element_size(),
                    lambda: _lib.check(L.fusg_nchw_to_nhwc_reflect(_lib.ptr(t), _lib.ptr(out), B, Cn, H, W, cp, border, self.cdtype,
                                                                   self._stream()), "fusg_nchw_to_nhwc_reflect"))
        return Padded(out, H, W, cp, border)

    def conv(self, path, x, stride, pad, out=None, tanh_nchw=None):
        """One convolution of a Conv2dBlock on the bordered input `x`; returns the raw NHWC output [B,Ho,Wo,cout]
        (or writes tanh(conv) as NCHW fp32 into `tanh_nchw`)."""
        w, bias, cout, cout_pad, cin, cin_pad, k, _, _ = self._w[path]
        assert x.C == cin_pad and x.border >= pad, (path, x.C, cin_pad, x.border, pad)
        B = x.t.shape[0]
        Ho, Wo = (x.H + 2 * pad - k) // stride + 1, (x.W + 2 * pad - k) // stride + 1
        d = ConvDesc()
        d.in0 = x.t.data_ptr()
        d.c0, d.pitch0 = x.C, x.C
        if self._kwide.get(path, x.C) > x.C:               # weights are 64 channels wide, the activation stores 32
            d.c0, d.cphys0 = self._kwide[path], x.C
        d.B, d.H, d.W = B, x.H, x.W
        d.ksize, d.stride = k, stride
        d.pad_mode, d.pad, d.border = 1, pad, x.border
        d.weight, d.bias = w.data_ptr(), bias.data_ptr()
        d.cout, d.cout_pad = cout, cout_pad
        if tanh_nchw is not None:
            d.outs[0].ptr = tanh_nchw.data_ptr()
            d.outs[0].elu, d.outs[0].layout = 2, 1
            res = tanh_nchw
        else:
            assert cout == cout_pad
            res = self._empty(B, Ho, Wo, cout)
            d.outs[0].ptr = res.data_ptr()
        d.dtype = self.cdtype
        d.impl = self.impl if self.dtype != "fp32" else IMPL_DIRECT
        L = _lib.lib()
        self._timed(path, "flops", 2.0 * B * Ho * Wo * cout * cin * k * k,
                    lambda: _lib.check(L.fusg_conv2d(C.byref(d), self._stream()), f"fusg_conv2d({path})"))
        return res, Ho, Wo

    def norm(self, name, raw, H, W, kind, gamma=None, beta=None, residual=None, relu=True, up=1, border=1):
        """InstanceNorm ('inst') / LayerNorm ('ln') of the raw conv output + activation (+ residual) (+ upsample), written as
        the bordered input of the next convolution."""
        torch = self.torch
        B, Cn = raw.shape[0], raw.shape[-1]
        HW = H * W
        nsplit = max(1, min(64, HW // 512))
        partial = self._empty(B * nsplit * Cn * 2 + B * Cn, dtype=torch.float32)      # (sum, sumsq) of the shifted values per split + the shifts
        ss = self._empty(B, Cn, 2, dtype=torch.float32)
        L = _lib.lib()
        esz = raw.element_size()
        self._timed(name + ".stats", "bytes", raw.numel() * esz,
                    lambda: _lib.check(L.fusg_norm_stats(_lib.ptr(raw), _lib.ptr(partial), B, HW, Cn, nsplit, self.cdtype, self._stream()),
                                       "fusg_norm_stats"))
        self._timed(name + ".finalize", "bytes", partial.numel() * 4,
                    lambda: _lib.check(L.fusg_norm_finalize(_lib.ptr(partial), _lib.ptr(gamma), _lib.ptr(beta), _lib.ptr(ss), B, HW, Cn, nsplit,
                                                            0 if kind == "inst" else 1, EPS, self._stream()), "fusg_norm_finalize"))
        out = self._empty(B, up * H + 2 * border, up * W + 2 * border, Cn)
        rb = 0
        if residual is not None:
            assert (residual.H, residual.W, residual.C) == (H, W, Cn)
            rb = residual.border
        self._timed(name + ".apply", "bytes", (raw.numel() * (2 if residual is not None else 1) + out.numel()) * esz,
                    lambda: _lib.check(L.fusg_norm_apply(_lib.ptr(raw), _lib.ptr(ss), _lib.ptr(residual.t) if residual is not None else None, rb,
                                                         _lib.ptr(out), B, H, W, Cn, 1 if relu else 0, up, border, self.cdtype, self._stream()),
                                       "fusg_norm_apply"))
        return Padded(out, up * H, up * W, Cn, border)

    # ------------------------------------------------------------------ the network
    def _block(self, path, x, stride, pad, kind, relu=True, residual=None, up=1, border=1):
        raw, Ho, Wo = self.conv(path, x, stride, pad)
        _, _, _, _, _, _, _, gamma, beta = self._w[path]
        return self.norm(path, raw, Ho, Wo, kind, gamma, beta, residual=residual, relu=relu, up=up, border=border)

    def _res_blocks(self, prefix, x, n_res, last_up=1, last_border=1):
        """ResBlocks (models.py:94-125) on a border-1 activation; the last block may upsample / re-border its sum."""
        for r in range(n_res):
            h = self._block(f"{prefix}.model.{r}.model.0", x, 1, 1, "inst", relu=True, border=1)
            last = r == n_res - 1
            x = self._block(f"{prefix}.model.{r}.model.1", h, 1, 1, "inst", relu=False, residual=x,
                            up=last_up if last else 1, border=last_border if last else 1)
        return x

    def encode(self, image_nchw, last_up=1, last_border=1):
        """ContentEncoder (models.py:128-149) -> bordered content activation."""
        m = self.m
        x = self.to_padded(image_nchw, 3, cpad=self._w["enc_content.model.0"][5])
        x = self._block("enc_content.model.0", x, 1, 3, "inst", border=1)
        for i in range(m.n_down):
            x = self._block(f"enc_content.model.{1 + i}", x, 2, 1, "inst", border=1)
        return self._res_blocks(f"enc_content.model.{1 + m.n_down}", x, m.n_res, last_up, last_border)

    def decode(self, content):
        """Decoder (models.py:164-188) on a border-1 content activation -> NCHW fp32 image."""
        m = self.m
        torch = self.torch
        x = self._res_blocks("dec.model.0", content, m.n_res, last_up=2, last_border=2)
        for i in range(m.n_down):
            last = i == m.n_down - 1
            x = self._block(f"dec.model.{2 + 2 * i}", x, 1, 2, "ln", up=1 if last else 2, border=3 if last else 2)
        B = x.t.shape[0]
        out = self._empty(B, m.output_nc, x.H, x.W, dtype=torch.float32)
        self.conv(f"dec.model.{1 + 2 * m.n_down}", x, 1, 3, tanh_nchw=out)
        return out

    def forward(self, image_nchw):
        return self.decode(self.encode(image_nchw))

    def content_to_nchw(self, c):
        b = c.border
        return c.t[:, b:b + c.H, b:b + c.W, :].permute(0, 3, 1, 2).float().contiguous()
