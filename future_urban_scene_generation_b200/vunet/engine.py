"""Execution engine of the VUNet forward on libfusg.so (include/fusg.h: fusg_conv2d).

The network of vunet/models.py:191-484 (reference) is run as a flat sequence of fused
convolution launches on NHWC activations.  Every tensor exists as `raw` and/or `elu` copy,
because the reference applies ELU to the *input* of most convolutions (pre-activation,
vunet/layers.py:98-102) while the operands reach the tensor cores straight from TMA: the producer
kernel's epilogue writes the activated copy once instead.

dtype 'bf16' is the product path (tcgen05 kernels); dtype 'fp32' is the verification build
(north_star: <=1e-4), which runs the same program on the CUDA-core direct kernel.
"""
import contextlib
import ctypes as C

from .. import _lib

DT_BF16, DT_F32 = 0, 1
IMPL_AUTO, IMPL_TC, IMPL_DIRECT = 0, 1, 2
PLAIN, D2S, S2D, D2S_BLOCK, UNPAIR = 0, 1, 2, 3, 4
MAX_OUTS = 6


class ConvOut(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("source", C.c_int32), ("elu", C.c_int32), ("layout", C.c_int32),
                ("mode", C.c_int32), ("blk", C.c_int32), ("reserved", C.c_int32)]


FUSED_NIN = ("app_encoder_1.nin.layers.1", "app_encoder_1.residual_0.layers.2")


class ConvDesc(C.Structure):
    _fields_ = [("in0", C.c_void_p), ("in1", C.c_void_p), ("c0", C.c_int32), ("c1", C.c_int32),
                ("pitch0", C.c_int32), ("pitch1", C.c_int32), ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("ksize", C.c_int32), ("stride", C.c_int32), ("weight", C.c_void_p), ("bias", C.c_void_p),
                ("cout", C.c_int32), ("cout_pad", C.c_int32), ("residual", C.c_void_p), ("noise", C.c_void_p),
                ("outs", ConvOut * MAX_OUTS), ("dtype", C.c_int32), ("impl", C.c_int32), ("zero_kblocks", C.c_uint64),
                ("pad_mode", C.c_int32), ("pad", C.c_int32), ("border", C.c_int32), ("cphys0", C.c_int32), ("cphys1", C.c_int32),
                ("cin_real", C.c_int32)]


class Act:
    """An activation: NHWC device tensors `raw` / `elu` (either may be None), C channels of a
    buffer whose pixel pitch is `pitch`, channel offset already applied to the data pointer."""
    __slots__ = ("raw", "elu", "C", "H", "W", "pitch", "off", "f32", "aux", "cphys")

    def __init__(self, C_, H, W, raw=None, elu=None, pitch=None, off=0, f32=None):
        self.raw, self.elu, self.C, self.H, self.W = raw, elu, C_, H, W
        self.pitch = pitch if pitch is not None else C_
        self.off = off
        self.f32 = f32          # optional NCHW fp32 API copy
        self.aux = {}
        self.cphys = None       # channels the buffer really holds when fewer than C (the rest read as zero: fusg_conv_desc.cphys)

    def slice(self, c0, c):
        a = Act(c, self.H, self.W, self.raw, self.elu, self.pitch, self.off + c0)
        return a


def _pad16(c):
    return (c + 15) // 16 * 16


class OutSpec:
    """What one output slot of a conv launch should produce."""
    __slots__ = ("source", "elu", "layout", "mode", "blk", "tensor")

    def __init__(self, source=0, elu=0, layout=0, mode=PLAIN, blk=0, tensor=None):
        self.source, self.elu, self.layout, self.mode, self.blk, self.tensor = source, elu, layout, mode, blk, tensor


class VunetEngine:
    def __init__(self, module, dtype="bf16", impl="auto"):
        self.m = module
        self.dtype = dtype
        self.impl = {"auto": IMPL_AUTO, "tcgen05": IMPL_TC, "direct": IMPL_DIRECT}[impl]
        self._wkey = None
        self._w = {}
        self._wp = {}                  # pixel-pair packed weights of the narrow stride-1 layers
        self._wfused = {}              # combined weights of fused layer pairs (see prepare_weights)
        self.launches = 0
        self.profile = None            # list -> per-launch (path, impl, flops, start, end) CUDA-event records
        self.noise_provider = None     # callable(B,C,H,W) -> NHWC fp32 device tensor; None = CPU torch.randn (reference semantics)

    # ------------------------------------------------------------------ plumbing
    @property
    def torch(self):
        return _lib.require_cuda()

    @property
    def tdtype(self):
        return self.torch.bfloat16 if self.dtype == "bf16" else self.torch.float32

    @property
    def cdtype(self):
        return DT_BF16 if self.dtype == "bf16" else DT_F32

    def device(self):
        return next(self.m.parameters()).device

    def _stream(self):
        return _lib.stream_ptr(self.torch)

    def _empty(self, *shape, dtype=None):
        return self.torch.empty(shape, dtype=dtype or self.tdtype, device=self.device())

    def record_stream(self, act, stream):
        """Marks every tensor of an activation as in use on `stream` (torch's caching allocator)."""
        for t in (act.raw, act.elu, act.f32) + tuple(v for v in act.aux.values() if hasattr(v, "record_stream")):
            if t is not None and t.is_cuda:
                t.record_stream(stream)

    # ------------------------------------------------------------------ weights
    def _weights_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.m.parameters())

    def prepare_weights(self, force=False):
        """weight_norm fold + repack (layers.py:29-31), once per (re)load of the parameters."""
        key = self._weights_key()
        if not force and key == self._wkey:
            return
        torch = self.torch
        dev = self.device()
        if dev.type != "cuda":
            raise _lib.FusgError("Vunet_fix_res: parameters are not on a CUDA device; the B200 path has no CPU fallback "
                                 "(call .to('cuda'))")
        L = _lib.lib()
        self._w = {}
        self._wp = {}
        with torch.cuda.device(dev):
            for path, conv in self.m.convs.items():
                cout, cin, k = conv.cout, conv.cin, conv.k
                cin_pad = 32 if cin < 16 else cin            # the two RGB-ish first layers are padded to one 64B swizzle span
                if path == FUSED_NIN[0] and self.dtype == "bf16":
                    cin_pad = 64                             # its input doubles as a 64-channel operand of the fused residual
                cout_pad = _pad16(cout)
                w = torch.empty((cout_pad, k * k, cin_pad), dtype=self.tdtype, device=dev)
                bias = torch.zeros((cout_pad,), dtype=torch.float32, device=dev)
                bias[:cout] = conv.bias.detach().float()
                v = conv.weight_v.detach().float().contiguous()
                g = conv.weight_g.detach().float().contiguous()
                _lib.check(L.fusg_fold_weightnorm(_lib.ptr(v), _lib.ptr(g), _lib.ptr(w), cout, cin, k, cout_pad, cin_pad,
                                                  self.cdtype, self._stream()), "fusg_fold_weightnorm")
                self.launches += 1
                self._w[path] = (w, bias, cout, cout_pad, cin_pad, k)
                if self.dtype == "bf16" and cout in (32, 3) and cin in (32, 64):
                    # narrow layer: also fold a pixel-pair packed copy (inputs are one or two 32-channel tensors)
                    c0, c1 = 32, cin - 32
                    cp2 = _pad16(2 * cout)
                    wp = torch.empty((cp2, k * k, 2 * cin), dtype=self.tdtype, device=dev)
                    bp = torch.empty((cp2,), dtype=torch.float32, device=dev)
                    braw = conv.bias.detach().float().contiguous()
                    _lib.check(L.fusg_fold_weightnorm_paired(_lib.ptr(v), _lib.ptr(g), _lib.ptr(braw), _lib.ptr(wp), _lib.ptr(bp), cout, c0, c1, k,
                                                             cp2, self.cdtype, self._stream()), "fusg_fold_weightnorm_paired")
                    self.launches += 1
                    self._wp[path] = (wp, bp, 2 * cout, cp2, 2 * cin, k)
            # NiN folded into the first residual of the appearance encoder: x0 + conv3x3(ELU(x0)) with x0 = NiN(ELU(in))
            # becomes one convolution over [ELU(x0) | ELU(in)] whose weights for the second input are the NiN's at the
            # centre tap and zero elsewhere -- the tensor core adds the residual, so x0 itself is never written or read
            # (2.1 GB of HBM traffic per 64-crop forward); the kernel skips the all-zero k-blocks (zero_kblocks hint)
            self._wfused = {}
            if self.dtype == "bf16":
                nin_p, res_p = FUSED_NIN
                wn, bn, cout, cout_pad, cinp_n, _ = self._w[nin_p]
                wr, br, _, _, cinp_r, k = self._w[res_p]
                wc = torch.zeros((cout_pad, k * k, cinp_r + cinp_n), dtype=self.tdtype, device=dev)
                wc[:, :, :cinp_r] = wr
                wc[:, (k * k) // 2, cinp_r:] = wn[:, 0, :]
                chunks = (cinp_r + cinp_n) // 64
                zero = 0
                for tap in range(k * k):
                    if tap != (k * k) // 2:
                        for c in range(cinp_r // 64, chunks):
                            zero |= 1 << (tap * chunks + c)
                self._wfused[res_p] = (wc, (br + bn).contiguous(), cout, cout_pad, cinp_r + cinp_n, k, zero)
        self._wkey = key

    # ------------------------------------------------------------------ one conv launch
    def conv(self, path, srcs, stride=1, residual=None, noise=None, outs=(), B=None, fused=False):
        """srcs: list of (Act, 'raw'|'elu') -- one or two inputs concatenated along channels.
        outs: list of OutSpec with .tensor set.  Returns nothing (outputs are written in place)."""
        d = ConvDesc()
        if fused:
            w, bias, cout, cout_pad, cin_pad, k, d.zero_kblocks = self._wfused[path]
        else:
            w, bias, cout, cout_pad, cin_pad, k = self._w[path]
        a0, which0 = srcs[0]
        # pixel-pair packing: [B,H,W,32] viewed as [B,H,W/2,64] (same bytes) for narrow stride-1 layers
        pair = (not fused and path in self._wp and stride == 1 and noise is None and a0.W >= 64 and a0.W % 2 == 0
                and all(a.C == 32 and a.pitch == 32 and a.off == 0 for a, _ in srcs) and all(o.mode == PLAIN for o in outs))
        if pair:
            w, bias, cout, cout_pad, cin_pad, k = self._wp[path]
        pm = 2 if pair else 1
        t0 = getattr(a0, which0)
        assert t0 is not None, f"{path}: input 0 has no '{which0}' copy"
        esz = t0.element_size()
        d.in0 = t0.data_ptr() + a0.off * esz
        d.c0, d.pitch0 = a0.C * pm, a0.pitch * pm
        d.cphys0 = a0.cphys or 0
        if a0.cphys and len(srcs) == 1 and path in self.m.convs:
            d.cin_real = self.m.convs[path].cin            # a network input stored 16 wide: lets AUTO pick the streaming 1x1 kernel
        ctot = a0.C * pm
        keep = [t0]
        if len(srcs) > 1:
            a1, which1 = srcs[1]
            t1 = getattr(a1, which1)
            assert t1 is not None, f"{path}: input 1 has no '{which1}' copy"
            assert (a1.H, a1.W) == (a0.H, a0.W)
            d.in1 = t1.data_ptr() + a1.off * esz
            d.c1, d.pitch1 = a1.C * pm, a1.pitch * pm
            d.cphys1 = a1.cphys or 0
            ctot += a1.C * pm
            keep.append(t1)
        assert ctot == cin_pad, f"{path}: channels {ctot} != weight cin {cin_pad}"
        d.B, d.H, d.W = B, a0.H, a0.W // pm
        d.ksize, d.stride = k, stride
        d.weight, d.bias = w.data_ptr(), bias.data_ptr()
        d.cout, d.cout_pad = cout, cout_pad
        if residual is not None:
            assert residual.raw is not None and residual.pitch == residual.C and residual.off == 0 and residual.C * pm == cout
            d.residual = residual.raw.data_ptr()
        if noise is not None:
            d.noise = noise.data_ptr()
        assert 0 < len(outs) <= MAX_OUTS
        for i, o in enumerate(outs):
            d.outs[i].ptr = o.tensor.data_ptr()
            d.outs[i].source, d.outs[i].elu, d.outs[i].layout = o.source, o.elu, o.layout
            d.outs[i].mode, d.outs[i].blk = o.mode, o.blk
            if pair and o.layout == 1:
                d.outs[i].mode = UNPAIR
        d.dtype = self.cdtype
        d.impl = self.impl if self.dtype == "bf16" else IMPL_DIRECT
        prof = self.profile
        if prof is not None:
            torch = self.torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            impl = d.impl if d.impl != IMPL_AUTO else _lib.lib().fusg_conv2d_select(C.byref(d))
            Ho, Wo = (a0.H - 1) // stride + 1, (a0.W - 1) // stride + 1
            e0.record()
        rc = _lib.lib().fusg_conv2d(C.byref(d), self._stream())
        _lib.check(rc, f"fusg_conv2d({path})")
        if prof is not None:
            e1.record()
            # algorithmic FLOPs of the reference conv (real channels, SURVEY.md §8d)
            conv = self.m.convs[path]
            prof.append((path, impl, 2.0 * B * Ho * Wo * conv.cout * conv.cin * k * k, e0, e1))
        self.launches += 1

    # ------------------------------------------------------------------ helpers building Acts
    def _act(self, B, Cn, H, W, raw=True, elu=True):
        return Act(Cn, H, W, raw=self._empty(B, H, W, Cn) if raw else None, elu=self._empty(B, H, W, Cn) if elu else None)

    def _plain_outs(self, act):
        outs = []
        if act.raw is not None:
            outs.append(OutSpec(tensor=act.raw))
        if act.elu is not None:
            outs.append(OutSpec(elu=1, tensor=act.elu))
        return outs

    def from_nchw(self, t, elu_only=False, cpad=None, cphys=None):
        """Foreign NCHW fp32 tensor -> Act (raw + elu, or only the ELU copy).  cphys: store only this many channels
        (>= the tensor's, multiple of 8) although the Act is `cpad` channels wide for the convolutions that read it -- the
        kernels zero-extend (fusg_conv_desc.cphys0/1), so the padding never exists in HBM."""
        torch = self.torch
        t = t.detach()
        if t.device != self.device():
            t = t.to(self.device())
        t = t.float().contiguous()
        B, Cn, H, W = t.shape
        cp = cpad or Cn
        L = _lib.lib()
        act = Act(cp, H, W)
        if cphys is not None and cphys < cp:
            assert cphys >= Cn and cphys % 8 == 0
            act.pitch = act.cphys = cphys
            cp = cphys
        if not elu_only:
            act.raw = self._empty(B, H, W, cp)
            _lib.check(L.fusg_nchw_to_nhwc(_lib.ptr(t), _lib.ptr(act.raw), B, Cn, H, W, cp, 0, self.cdtype, self._stream()), "nchw_to_nhwc")
            self.launches += 1
        act.elu = self._empty(B, H, W, cp)
        _lib.check(L.fusg_nchw_to_nhwc(_lib.ptr(t), _lib.ptr(act.elu), B, Cn, H, W, cp, 1, self.cdtype, self._stream()), "nchw_to_nhwc")
        self.launches += 1
        act.aux["keep"] = t
        return act

    def to_nchw(self, act, which="raw"):
        """Act -> NCHW fp32 torch tensor (API-visible), remembering the Act for zero-cost chaining."""
        if act.f32 is not None and which == "raw":
            out = act.f32
        else:
            src = getattr(act, which)
            B = src.shape[0]
            out = self._empty(B, act.C, act.H, act.W, dtype=self.torch.float32)
            _lib.check(_lib.lib().fusg_nhwc_to_nchw(C.c_void_p(src.data_ptr() + act.off * src.element_size()), _lib.ptr(out), B, act.C,
                                                    act.H, act.W, act.pitch, self.cdtype, self._stream()), "nhwc_to_nchw")
            self.launches += 1
        out._fusg_act = (act, out._version)
        return out

    def as_act(self, t, need_raw=True):
        """API tensor -> Act: the attached engine-native activation if the tensor is untouched,
        else a conversion of its values."""
        tag = getattr(t, "_fusg_act", None)
        if tag is not None and tag[1] == t._version and (tag[0].raw is not None or not need_raw) and tag[0].elu is not None:
            return tag[0]
        return self.from_nchw(t, elu_only=not need_raw)

    def _ensure_elu(self, act):
        if act.elu is None:
            act.elu = self.torch.empty_like(act.raw)
            assert act.pitch == act.C and act.off == 0
            _lib.check(_lib.lib().fusg_elu(_lib.ptr(act.raw), _lib.ptr(act.elu), act.raw.numel(), self.cdtype, self._stream()), "fusg_elu")
            self.launches += 1
        return act

    def draw_noise(self, B, Cn, H, W):
        """Sampler noise (layers.py:166): torch.randn on the CPU default generator, in the reference's
        order and NCHW shape; shipped to the device as NHWC fp32 for the conv epilogue."""
        if self.noise_provider is not None:
            return self.noise_provider(B, Cn, H, W)
        torch = self.torch
        eps = torch.randn(B, Cn, H, W)
        # NHWC copy in pinned memory (caching host allocator: reuse is ordered after the async copy)
        stage = torch.empty((B, H, W, Cn), dtype=torch.float32, pin_memory=True)
        stage.copy_(eps.permute(0, 2, 3, 1))
        return stage.to(self.device(), non_blocking=True)

    @contextlib.contextmanager
    def noise_from(self, provider):
        """Draws the Sampler noise from `provider` inside the block.  The engine is shared by every user of its model, so
        the previous provider is put back however the block ends."""
        prev, self.noise_provider = self.noise_provider, provider
        try:
            yield
        finally:
            self.noise_provider = prev

    # ------------------------------------------------------------------ blocks
    def residual(self, path, x, skip=None, B=None, raw=True, elu=True, out_mode=PLAIN):
        """Residual (layers.py:83-105): x + conv3x3(elu(cat[x, skip])), optionally written SpaceToDepth'ed."""
        cout = self._w[path + ".layers.2"][2]
        if out_mode == S2D:
            out = self._act(B, 4 * cout, x.H // 2, x.W // 2, raw, elu)
        else:
            out = self._act(B, cout, x.H, x.W, raw, elu)
        srcs = [(x, "elu")] + ([(skip, "elu")] if skip is not None else [])
        outs = self._plain_outs(out)
        for o in outs:
            o.mode = out_mode
        self.conv(path + ".layers.2", srcs, residual=x, outs=outs, B=B)
        return out

    def nin(self, path, srcs, B, raw=True, elu=True):
        """NiN (layers.py:42-58): conv1x1(elu(x)); srcs = Acts whose ELU copies are concatenated."""
        cout = self._w[path + ".layers.1"][2]
        out = self._act(B, cout, srcs[0].H, srcs[0].W, raw, elu)
        self.conv(path + ".layers.1", [(s, "elu") for s in srcs], outs=self._plain_outs(out), B=B)
        return out

    def down_block(self, path, x, B, last_elu=False):
        """DownBlock (models.py:92-114) -> (x, [skip0, skip1])."""
        cout = self._w[path + ".down.down"][2]
        d = self._act(B, cout, x.H // 2, x.W // 2)
        self.conv(path + ".down.down", [(x, "raw")], stride=2, outs=self._plain_outs(d), B=B)
        s0 = self.residual(path + ".residual_0", d, B=B)
        s1 = self.residual(path + ".residual_1", s0, B=B, elu=last_elu)
        return s1, [s0, s1]

    def init_block(self, path, x_elu, B, last_elu=False):
        """InitBlock (models.py:141-163); x_elu already holds ELU(x) padded to the weight's cin."""
        cout = self._w[path + ".nin.layers.1"][2]
        if path + ".residual_0.layers.2" in self._wfused:
            # fused form: only ELU(NiN(x)) is materialised; the residual term is recomputed by the tensor core
            h = self._act(B, cout, x_elu.H, x_elu.W, raw=False, elu=True)
            self.conv(path + ".nin.layers.1", [(x_elu, "elu")], outs=self._plain_outs(h), B=B)
            s0 = self._act(B, cout, x_elu.H, x_elu.W)
            self.conv(path + ".residual_0.layers.2", [(h, "elu"), (x_elu, "elu")], outs=self._plain_outs(s0), B=B, fused=True)
            s1 = self.residual(path + ".residual_1", s0, B=B, elu=last_elu)
            return s1, [s0, s1]
        h = self._act(B, cout, x_elu.H, x_elu.W)
        self.conv(path + ".nin.layers.1", [(x_elu, "elu")], outs=self._plain_outs(h), B=B)
        s0 = self.residual(path + ".residual_0", h, B=B)
        s1 = self.residual(path + ".residual_1", s0, B=B, elu=last_elu)
        return s1, [s0, s1]

    def upsample(self, path, x, B, raw=True, elu=True):
        """UpSample 'subpixel' (layers.py:121-152): DepthToSpace(conv3x3(x -> 4*cout))."""
        c4 = self._w[path + ".depth4x"][2]
        out = self._act(B, c4 // 4, 2 * x.H, 2 * x.W, raw, elu)
        outs = self._plain_outs(out)
        for o in outs:
            o.mode = D2S
        self.conv(path + ".depth4x", [(x, "raw")], outs=outs, B=B)
        return out

    def sampler_plain(self, path, x, B, want_s2d=True):
        """Sampler (layers.py:158-170) of the appearance decoder: returns Acts (mu, z) carrying fp32
        NCHW API copies, z.raw, and SpaceToDepth'ed ELU copies for the auto-regressive blocks."""
        torch = self.torch
        cout = self._w[path + ".conv"][2]
        H, W = x.H, x.W
        eps = self.draw_noise(B, cout, H, W)
        mu = Act(cout, H, W, f32=self._empty(B, cout, H, W, dtype=torch.float32))
        z = Act(cout, H, W, raw=self._empty(B, H, W, cout), f32=self._empty(B, cout, H, W, dtype=torch.float32))
        outs = [OutSpec(layout=1, tensor=mu.f32), OutSpec(source=1, layout=1, tensor=z.f32), OutSpec(source=1, tensor=z.raw)]
        if want_s2d:
            mu.aux["s2d_elu"] = self._empty(B, H // 2, W // 2, 4 * cout)
            z.aux["s2d_elu"] = self._empty(B, H // 2, W // 2, 4 * cout)
            outs += [OutSpec(elu=1, mode=S2D, tensor=mu.aux["s2d_elu"]), OutSpec(source=1, elu=1, mode=S2D, tensor=z.aux["s2d_elu"])]
        self.conv(path + ".conv", [(x, "raw")], noise=eps, outs=outs, B=B)
        z.aux["eps"] = eps
        return mu, z

    def ar_block(self, path, x, skip_a, B, g_s2d_elu=None, gk=None):
        """AutoRegressiveBlock (models.py:17-89).  g_s2d_elu: (B,h/2,w/2,512) ELU(SpaceToDepth(enc_down_mu))
        or None.  gk: three (B,h,w,512) tensors ELU(nin_k(g)), k = 0..2, computed beforehand (encode_vehicles): the
        block then skips its three nin_k launches.  Returns (x, mu Act with .f32, z Act with .f32 and .elu)."""
        torch = self.torch
        x = self.residual(path + ".residual_init", x, skip_a, B=B)
        x_ = self.residual(path + ".residual_s2d", x, B=B, out_mode=S2D)
        h, w = x_.H, x_.W
        if gk is not None:
            assert len(gk) == 3 and all(tuple(t.shape) == (B, h, w, 512) for t in gk), f"{path}: gk must be three (B,{h},{w},512) tensors"
            gk = [Act(512, h, w, elu=t) for t in gk]
        elif g_s2d_elu is not None:
            g = Act(512, h, w, elu=g_s2d_elu)
            gk = [self.nin(f"{path}.nin_{k}", [g.slice(128 * k, 128)], B, raw=False) for k in range(3)]
        mu = Act(128, 2 * h, 2 * w, f32=self._empty(B, 128, 2 * h, 2 * w, dtype=torch.float32))
        z = Act(128, 2 * h, 2 * w, elu=self._empty(B, 2 * h, 2 * w, 128), f32=self._empty(B, 128, 2 * h, 2 * w, dtype=torch.float32))
        for k in range(4):
            eps = self.draw_noise(B, 128, h, w)
            outs = [OutSpec(layout=1, mode=D2S_BLOCK, blk=k, tensor=mu.f32),
                    OutSpec(source=1, layout=1, mode=D2S_BLOCK, blk=k, tensor=z.f32),
                    OutSpec(source=1, elu=1, mode=D2S_BLOCK, blk=k, tensor=z.elu)]
            zk = None
            if gk is None and k < 3:
                zk = Act(128, h, w, elu=self._empty(B, h, w, 128))
                outs.append(OutSpec(source=1, elu=1, tensor=zk.elu))
            self.conv(f"{path}.sampler_{k}.conv", [(x_, "raw")], noise=eps, outs=outs, B=B)
            z.aux[f"eps{k}"] = eps
            if k < 3:
                skip = gk[k] if gk is not None else self.nin(f"{path}.nin_{k}", [zk], B, raw=False)
                x_ = self.residual(f"{path}.residual_{k}", x_, skip, B=B)
        return x, mu, z

    def up_block(self, path, x, skip_a, skip_b, B):
        """UpBlock (models.py:117-138)."""
        x = self.residual(path + ".residual_0", x, skip_a, B=B)
        x = self.residual(path + ".residual_1", x, skip_b, B=B, elu=False)
        return self.upsample(path + ".up", x, B)

    # ------------------------------------------------------------------ the four sub-forwards
    def enc_up(self, x_nchw):
        """models.py:333-353 -> (outputs [Act,Act], skips [Act,Act])."""
        B = x_nchw.shape[0]
        # the 6- / 3-channel network inputs are stored 16 channels wide; TMA zero-fills the rest of their 64- / 32-channel K block
        xin = self.from_nchw(x_nchw, elu_only=True, cpad=self._w["app_encoder_1.nin.layers.1"][4], cphys=16)
        x, _ = self.init_block("app_encoder_1", xin, B)
        for name in ("app_encoder_1_a", "app_encoder_1_b", "app_encoder_1_c", "app_encoder_2"):
            x, _ = self.down_block(name, x, B)
        x, _ = self.down_block("app_encoder_3", x, B, last_elu=True)
        skips = [self.nin("app_skip_3_c", [x], B)]
        x, sl = self.down_block("app_encoder_4", x, B, last_elu=True)
        outputs = [sl[-2], x]
        skips.append(self.nin("app_skip_4_c", [x], B))
        return outputs, skips

    def enc_down(self, outputs, skips):
        """models.py:390-408 -> (mu [Act,Act], z [Act,Act])."""
        o_r0, o_x = outputs
        B = o_x.raw.shape[0]
        xb = self._act(B, 128, o_x.H, o_x.W)
        self.conv("app_bottleneck", [(o_x, "raw")], outs=self._plain_outs(xb), B=B)
        xa = self.residual("app_decoder_1_a", xb, skips[-1], B=B)
        mu0, z0 = self.sampler_plain("app_decoder_1_b", xa, B)
        x_ = self._act(B, 128, xa.H, xa.W, raw=False)
        self.conv("app_decoder_1_c", [(o_r0, "raw"), (z0, "raw")], outs=self._plain_outs(x_), B=B)
        xd = self.residual("app_decoder_1_d", xa, x_, B=B, elu=False)
        xe = self.upsample("app_decoder_1_e", xd, B)
        xf = self.residual("app_decoder_2_a", xe, B=B, elu=False)
        mu1, z1 = self.sampler_plain("app_decoder_2_b", xf, B)
        return [mu0, mu1], [z0, z1]

    def encode_vehicles(self, x_nchw):
        """The appearance side of the trajectory loop, once per vehicle (trajectory_inference.py:230-233): enc_up, enc_down,
        then the six nin_k convolutions of the two auto-regressive blocks on the MEANS mu (traj_test decodes with mu_app,
        :413-426).  enc_down still draws its two Sampler tensors, (V,128,4,4) and (V,128,8,8), like the reference, although
        z is not used.  Returns [ELU(nin_k(ELU(S2D(mu_n))))] for n = 0, 1 and k = 0..2: six (V,h,w,512) tensors, h = 2 then 4,
        whose rows dec_down(..., enc_gk=...) takes per item."""
        V = x_nchw.shape[0]
        out_e, skips_e = self.enc_up(x_nchw)
        mu, _ = self.enc_down(out_e, skips_e)
        gk = []
        for n, blk in enumerate(("shape_decoder_1", "shape_decoder_2")):
            g = mu[n].aux["s2d_elu"]
            ga = Act(512, g.shape[1], g.shape[2], elu=g)
            gk += [self.nin(f"{blk}.nin_{k}", [ga.slice(128 * k, 128)], V, raw=False).elu for k in range(3)]
        return gk

    def dec_up(self, y_nchw, raw_skips=True):
        """models.py:355-388 -> (outputs [Act], skips [14 Acts]).  raw_skips=False writes only the ELU copies of the NiN
        skips, which is all dec_down reads; the sub-forward API (forward_dec_up) also returns the raw values."""
        B = y_nchw.shape[0]
        yin = self.from_nchw(y_nchw, elu_only=True, cpad=32, cphys=16)
        skips = []
        x, sl = self.init_block("shape_encoder_1", yin, B, last_elu=True)
        skips += [self.nin("shape_skip_1_b", [sl[-2]], B, raw=raw_skips), self.nin("shape_skip_1_c", [sl[-1]], B, raw=raw_skips)]
        for enc, sk in (("shape_encoder_1_a", "shape_skip_1_a"), ("shape_encoder_2", "shape_skip_2"),
                        ("shape_encoder_3", "shape_skip_3"), ("shape_encoder_4", "shape_skip_4"),
                        ("shape_encoder_5", "shape_skip_5"), ("shape_encoder_6", "shape_skip_6")):
            x, sl = self.down_block(enc, x, B, last_elu=True)
            skips += [self.nin(sk + "_b", [sl[-2]], B, raw=raw_skips), self.nin(sk + "_c", [sl[-1]], B, raw=raw_skips)]
        return [x], skips

    def dec_down(self, outputs, skips, enc_g=(), enc_gk=None):
        """models.py:410-459.  skips: list of 14 Acts (consumed from the end, like the reference's pop()).
        enc_g: () or two (B,h/2,w/2,512) ELU(SpaceToDepth(enc_down_mu)) tensors.
        enc_gk: None or, per auto-regressive block, the three ELU(nin_k(g)) tensors encode_vehicles returns (gathered to the
        items); replaces enc_g.  Returns (x_tilde fp32 NCHW tensor, [mu Acts], [z Acts])."""
        torch = self.torch
        skips = list(skips)
        x0 = outputs[-1]
        B = x0.raw.shape[0]
        x = self._act(B, 128, x0.H, x0.W)
        self.conv("shape_bottleneck", [(x0, "raw")], outs=self._plain_outs(x), B=B)
        mus, zs = [], []
        for n, blk in enumerate(("shape_decoder_1", "shape_decoder_2")):
            skip_a, skip_b = skips.pop(), skips.pop()
            if enc_gk is not None:
                x, mu_n, z_n = self.ar_block(blk, x, skip_a, B, gk=enc_gk[n])
            else:
                x, mu_n, z_n = self.ar_block(blk, x, skip_a, B, None if len(enc_g) == 0 else enc_g[n])
            mus.append(mu_n)
            zs.append(z_n)
            x = self.nin(blk + "_n", [x, z_n], B)
            x = self.residual(blk + "_o", x, skip_b, B=B, elu=False)
            x = self.upsample(blk + "_p", x, B)
        for blk in ("shape_decoder_3", "shape_decoder_4", "shape_decoder_5", "shape_decoder_5_a"):
            skip_a, skip_b = skips.pop(), skips.pop()
            x = self.up_block(blk, x, skip_a, skip_b, B)
        skip_a, skip_b = skips.pop(), skips.pop()
        x = self.residual("shape_decoder_6.residual_0", x, skip_a, B=B)
        x = self.residual("shape_decoder_6.residual_1", x, skip_b, B=B, elu=False)
        assert not skips
        x_tilde = self._empty(B, 3, x.H, x.W, dtype=torch.float32)
        self.conv("shape_decoder_6.conv", [(x, "raw")], outs=[OutSpec(layout=1, tensor=x_tilde)], B=B)
        return x_tilde, mus, zs

    def g_from_api(self, t):
        """ELU(SpaceToDepth(enc_down_mu)) (B,h/2,w/2,512) for an API tensor (models.py:60-64)."""
        tag = getattr(t, "_fusg_act", None)
        if tag is not None and tag[1] == t._version and "s2d_elu" in tag[0].aux:
            return tag[0].aux["s2d_elu"]
        # foreign tensor: SpaceToDepth on the NCHW view (block-major, layers.py:197-221), then NHWC + ELU
        t = t.detach().to(self.device()).float()
        b, c, h, w = t.shape
        s2d = t.view(b, c, h // 2, 2, w // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(b, 4 * c, h // 2, w // 2).contiguous()
        return self.from_nchw(s2d, elu_only=True).elu
