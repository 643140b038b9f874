"""Every launch of the VUNet and ICN engines against an fp64 reference of its layer (oracle/launch_oracle.py).

The whole-network tests bound the final image at 1e-2, which a fault confined to one layer -- one image column of a
pair-packed layer, one D2S_BLOCK quadrant, the last partly filled batch tile, one CTA-pair tile -- can stay under.
Here a fixture wraps the engines' launch methods on the instance; each launch

  1. has its output tensors filled with NaN first (a D2S_BLOCK output, shared by four launches, is snapshotted and only
     the launch's own quadrant is filled),
  2. runs and is synchronised,
  3. is compared per element with the fp64 reference of its layer, slot by slot, within the bounds of
     launch_oracle; every element it owns must be finite, and a D2S_BLOCK launch must leave the other quadrants as
     they were,
  4. may only read tensors that were themselves checked when they were written, so no link of the chain goes
     unverified.

Each launch's kernel and tcgen05 tiling plan are recorded; the last test asserts that the product networks, at the
batch sizes they run, reached every plan variant of k_conv_tc.  Run with -s to see the per-launch margin lines
(worst |got - ref| / bound).
"""
import time

import pytest

from oracle import launch_oracle as LO

pytestmark = pytest.mark.gpu

IMPL_NAMES = {1: "tc", 2: "direct", 3: "smallcin"}
NAN_DT = {2: "int16", 4: "int32"}

# plan variants of k_conv_tc (plan_tc) the walks below must reach between them
REQUIRED_VARIANTS = {"smallcin", "pair", "halo k=3", "halo k=5", "halo k=7", "halo+w_resident", "msub2 no halo", "ksplit",
                     "fast_epi=0", "fast_epi=1", "fast_epi=2", "fast_epi=3", "fused under halo"}
WALKS = {"vunet bf16 B=1", "vunet bf16 B=5", "vunet bf16 B=8", "vunet bf16 B=64", "trajectory V=8 B=64",
         "dec_down g_from_api B=2", "vunet fp32 B=2", "icn fp16 B=64 256", "icn fp16 B=3 64", "icn bf16 B=8 256"}
REACHED = {"variants": set(), "walks": set()}


def _cfg():
    from argparse import Namespace
    return Namespace(up_mode='subpixel', w_norm=True, drop_prob=0.2, vunet_256=True)


@pytest.fixture(scope="module")
def vnet(cuda):
    from future_urban_scene_generation_b200.vunet.models import Vunet_fix_res
    from oracle import vunet_oracle as VO
    m = Vunet_fix_res(_cfg())
    m.load_state_dict(VO.make_state_dict(0), strict=True)
    return m.to("cuda").eval()


def _icn(dtype):
    from future_urban_scene_generation_b200.warp_learn.models import G_Resnet
    from oracle import icn_oracle as IO
    m = G_Resnet(21, dtype=dtype)
    m.load_state_dict(IO.make_state_dict(0), strict=True)
    return m.cuda().eval()


def _vunet_inputs(torch, start, B):
    from future_urban_scene_generation_b200 import synth
    x, y = synth.make_vunet_inputs(start, B)
    return torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()


def _icn_inputs(torch, start, B, res):
    from future_urban_scene_generation_b200 import synth
    return torch.from_numpy(synth.make_icn_inputs(start, B, res)).cuda()


def _nchw(t, layout):
    """An output slot's tensor as an NCHW view (layout 0: NHWC activation, 1: NCHW fp32)."""
    return t if layout == 1 else t.permute(0, 3, 1, 2)


def _chunks(B, per_image):
    """Batch ranges whose fp64 reference tensors stay near 2^26 elements (512 MB) each."""
    cb = max(1, (1 << 26) // max(1, per_image))
    return [(b, min(B, b + cb)) for b in range(0, B, cb)]


class Walker:
    """Checks every launch of one engine instance; see the module docstring."""

    def __init__(self, torch, monkeypatch, eng, label, perturb=None):
        from future_urban_scene_generation_b200 import _lib
        self.torch, self.eng, self.label, self.perturb = torch, eng, label, perturb
        self.checked = {}                 # id(tensor) -> weakref: tensors whose values were verified when written
        self.blocks = {}                  # id(tensor) -> quadrants of a D2S_BLOCK output verified so far
        self.lines = []
        self.last = None
        self._wcache = {}
        self.t0 = time.time()
        lib = _lib.lib()
        orig_conv2d = lib.fusg_conv2d

        def fusg_conv2d(dref, stream):
            d = dref._obj
            impl = d.impl if d.impl != 0 else lib.fusg_conv2d_select(dref)
            rc = orig_conv2d(dref, stream)
            plan = _lib.conv_last_plan() if rc == 0 and impl == 1 else None
            self.last = dict(impl=impl, plan=plan, ksize=d.ksize, zero_kblocks=d.zero_kblocks, c0=d.c0, W=d.W)
            return rc
        monkeypatch.setattr(lib, "fusg_conv2d", fusg_conv2d)

        def empty(*shape, dtype=None):    # every tensor the engine allocates starts as NaN
            return torch.full(shape, float("nan"), dtype=dtype or eng.tdtype, device=eng.device())
        monkeypatch.setattr(eng, "_empty", empty)
        for name in (("conv", "from_nchw", "_ensure_elu", "draw_noise") if hasattr(eng, "draw_noise") else ("conv", "norm", "to_padded")):
            orig = getattr(eng, name)
            wrapper = getattr(self, ("vunet_" if hasattr(eng, "draw_noise") else "icn_") + name.lstrip("_"))
            monkeypatch.setattr(eng, name, (lambda o, w: lambda *a, **k: w(o, *a, **k))(orig, wrapper))

    # ------------------------------------------------------------------ bookkeeping
    def mark(self, t):
        import weakref
        self.checked[id(t)] = weakref.ref(t)

    def need(self, t, path, what):
        ref = self.checked.get(id(t))
        assert ref is not None and ref() is t, f"{self.label} {path}: {what} was not checked when it was written"

    def fail_if(self, ratio, idx, finite, got, ref, bound, path, slot):
        shape = tuple(got.shape)
        if finite and ratio <= 1.0:
            return
        import numpy as np
        where = tuple(int(v) for v in np.unravel_index(idx, shape))
        raise AssertionError(f"{self.label} {path} {slot}: worst |got-ref|/bound = {ratio:.3g} at (b,c,y,x)={where} "
                             f"got {float(got.reshape(-1)[idx]):.8g} ref {float(ref.reshape(-1)[idx]):.8g} "
                             f"bound {float(bound.reshape(-1)[idx]):.3g}{'' if finite else ' (non-finite values)'}")

    def record(self, path, ratio, fused=False):
        rec, self.last = self.last, None
        impl, plan = (rec["impl"], rec["plan"]) if rec else (0, None)
        desc = IMPL_NAMES.get(impl, "-")
        if plan:
            desc += " msub=%d pair=%d halo=%d ksplit=%d wres=%d epi=%d" % (plan["msub"], plan["pair"], plan["halo"], plan["ksplit"],
                                                                            plan["w_resident"], plan["fast_epi"])
        self.lines.append((path, desc, ratio))
        v = REACHED["variants"]
        if impl == 3:
            v.add("smallcin")
        if plan:
            if plan["pair"]:
                v.add("pair")
            if plan["halo"]:
                v.add(f"halo k={rec['ksize']}")
                if plan["w_resident"]:
                    v.add("halo+w_resident")
                if fused:
                    v.add("fused under halo")
            elif plan["msub"] == 2:
                v.add("msub2 no halo")
            if plan["ksplit"] > 1:
                v.add("ksplit")
            v.add(f"fast_epi={plan['fast_epi']}")
        return rec

    def report(self):
        worst = max(self.lines, key=lambda l: l[2])
        print(f"\n=== {self.label}: {len(self.lines)} launches checked in {time.time() - self.t0:.1f} s, worst ratio {worst[2]:.3f} ({worst[0]})")
        for path, desc, ratio in self.lines:
            print(f"  {ratio:7.4f}  {path:52s} {desc}")
        REACHED["walks"].add(self.label)

    def weights(self, path):
        """(w, step) of a VUNet layer: fp64 weight_norm fold of the module's parameters, rounded to the engine dtype."""
        if path not in self._wcache:
            conv = self.eng.m.convs[path]
            self._wcache[path] = LO.rounded(LO.fold(conv.weight_v, conv.weight_g), self.eng.tdtype)
        return self._wcache[path]

    # ------------------------------------------------------------------ VUNet
    def vunet_draw_noise(self, orig, *a, **k):
        eps = orig(*a, **k)
        self.mark(eps)                    # a primary input: the Sampler's N(0,1) draw
        return eps

    def vunet_from_nchw(self, orig, t, elu_only=False, cpad=None, cphys=None):
        torch = self.torch
        act = orig(t, elu_only=elu_only, cpad=cpad, cphys=cphys)
        torch.cuda.synchronize()
        src = t.detach().to(self.eng.device()).double()
        Cn = src.shape[1]
        u = LO.unit(self.eng.tdtype)
        for which, elu in (("raw", 0), ("elu", 1)):
            out = getattr(act, which)
            if out is None:
                continue
            got = out.permute(0, 3, 1, 2)
            ref = torch.nn.functional.elu(src) if elu else src
            bound = u * ref.abs() + (LO.ELU_ABS if elu else 0.0)
            self.fail_if(*LO.worst(got[:, :Cn], ref, bound), got[:, :Cn], ref, bound, "from_nchw", which)
            assert bool((got[:, Cn:] == 0).all()), f"{self.label} from_nchw {which}: channel padding is not zero"
            self.mark(out)
        return act

    def vunet_ensure_elu(self, orig, act):
        torch = self.torch
        had = act.elu is not None
        orig(act)
        if not had:
            torch.cuda.synchronize()
            self.need(act.raw, "ensure_elu", "input")
            raw = act.raw.double()
            ref = torch.nn.functional.elu(raw)
            bound = LO.unit(self.eng.tdtype) * ref.abs() + LO.ELU_ABS
            self.fail_if(*LO.worst(act.elu, ref, bound), act.elu, ref, bound, "ensure_elu", "elu")
            self.mark(act.elu)
        return act

    def vunet_conv(self, orig, path, srcs, stride=1, residual=None, noise=None, outs=(), B=None, fused=False):
        torch = self.torch
        from future_urban_scene_generation_b200.vunet.engine import D2S_BLOCK, FUSED_NIN
        for i, (a, which) in enumerate(srcs):
            self.need(getattr(a, which), path, f"input {i} ({which})")
        if residual is not None:
            self.need(residual.raw, path, "residual")
        if noise is not None:
            self.need(noise, path, "noise")
        snaps = {}
        for o in outs:
            if o.mode == D2S_BLOCK:
                if id(o.tensor) not in snaps:
                    snaps[id(o.tensor)] = o.tensor.clone()
                LO.d2s_block(_nchw(o.tensor, o.layout), o.blk).fill_(float("nan"))
            else:
                o.tensor.fill_(float("nan"))
        orig(path, srcs, stride=stride, residual=residual, noise=noise, outs=outs, B=B, fused=fused)
        torch.cuda.synchronize()
        rec = self.record(path, 0.0, fused)
        if self.perturb is not None:
            self.perturb(path, outs, rec)
        # ------------------------------------------------ the reference, chunked over the batch
        eng = self.eng
        acc = LO.ACC32 if eng.dtype == "fp32" else LO.ACC16
        a0 = srcs[0][0]
        Ho, Wo = (a0.H - 1) // stride + 1, (a0.W - 1) // stride + 1
        conv = eng.m.convs[path]
        worst = 0.0
        for b0, b1 in _chunks(B, max(sum(a.C for a, _ in srcs) * a0.H * a0.W, 4 * conv.cout * Ho * Wo)):
            def x_of(a, which):
                t = getattr(a, which)[b0:b1]
                return t[..., a.off:a.off + a.C].permute(0, 3, 1, 2).double()
            if fused:
                w_r, s_r = self.weights(path)
                w_n, s_n = self.weights(FUSED_NIN[0])
                xn = x_of(*srcs[1])[:, :eng.m.convs[FUSED_NIN[0]].cin]
                terms = [(x_of(*srcs[0]), w_r, s_r, 1), (xn, w_n, s_n, 0)]
                extras = [conv.bias.detach().double().view(1, -1, 1, 1), eng.m.convs[FUSED_NIN[0]].bias.detach().double().view(1, -1, 1, 1)]
            else:
                w, s = self.weights(path)
                x = torch.cat([x_of(a, wh) for a, wh in srcs], 1)[:, :conv.cin]
                terms = [(x, w, s, conv.k // 2)]
                extras = [conv.bias.detach().double().view(1, -1, 1, 1)]
            if residual is not None:
                extras.append(residual.raw[b0:b1].permute(0, 3, 1, 2).double())
            y, base = LO.conv_terms(terms, stride, extras, acc)
            del terms
            if noise is not None:
                nz = noise[b0:b1].permute(0, 3, 1, 2).double()
                z, base_z = y + nz, base + acc * nz.abs()
                del nz
            for i, o in enumerate(outs):
                val, bs = (z, base_z) if o.source == 1 else (y, base)
                u = LO.unit(eng.tdtype) if o.layout == 0 else 0.0
                ref, bound = LO.slot_ref(val, bs, o.elu, u)
                ref, bound = LO.place(ref, o.mode), LO.place(bound, o.mode)
                got = _nchw(o.tensor, o.layout)[b0:b1]
                if o.mode == D2S_BLOCK:
                    got = LO.d2s_block(got, o.blk)
                r = LO.worst(got, ref, bound)
                self.fail_if(*r, got, ref, bound, path, f"slot {i} (source={o.source} elu={o.elu} layout={o.layout} mode={o.mode} blk={o.blk})")
                worst = max(worst, r[0])
                del ref, bound, got
        for o in outs:
            if o.mode == D2S_BLOCK:
                snap = snaps[id(o.tensor)]
                isz = o.tensor.element_size()
                now_b = _nchw(o.tensor.view(getattr(torch, NAN_DT[isz])), o.layout)
                was_b = _nchw(snap.view(getattr(torch, NAN_DT[isz])), o.layout)
                owned = torch.zeros(now_b.shape, dtype=torch.bool, device=now_b.device)
                LO.d2s_block(owned, o.blk).fill_(True)
                assert torch.equal(now_b[~owned], was_b[~owned]), \
                    f"{self.label} {path}: D2S_BLOCK launch (blk={o.blk}) changed pixels of other quadrants"
                seen = self.blocks.setdefault(id(o.tensor), set())
                seen.add(o.blk)
                if seen == {0, 1, 2, 3}:
                    self.mark(o.tensor)
            else:
                self.mark(o.tensor)
        self.lines[-1] = (path, self.lines[-1][1], worst)

    # ------------------------------------------------------------------ ICN
    def icn_to_padded(self, orig, x_nchw, border, cpad=None):
        torch = self.torch
        p = orig(x_nchw, border, cpad=cpad)
        torch.cuda.synchronize()
        src = x_nchw.detach().to(self.eng.device()).double()
        Cn = src.shape[1]
        ref = torch.nn.functional.pad(src, (border,) * 4, mode="reflect")
        got = p.t.permute(0, 3, 1, 2)
        bound = LO.unit(self.eng.tdtype) * ref.abs()
        self.fail_if(*LO.worst(got[:, :Cn], ref, bound), got[:, :Cn], ref, bound, "to_padded", "out")
        assert bool((got[:, Cn:] == 0).all()), f"{self.label} to_padded: channel padding is not zero"
        self.mark(p.t)
        return p

    def icn_conv(self, orig, path, x, stride, pad, out=None, tanh_nchw=None):
        torch = self.torch
        self.need(x.t, path, "input")
        if tanh_nchw is not None:
            tanh_nchw.fill_(float("nan"))
        res, Ho, Wo = orig(path, x, stride, pad, out=out, tanh_nchw=tanh_nchw)
        torch.cuda.synchronize()
        rec = self.record(path, 0.0)
        if self.perturb is not None:
            self.perturb(path, [res], rec)
        eng = self.eng
        blk = eng.m.blocks[path]
        w = blk.conv.weight.detach().to(eng.tdtype).double()
        b = blk.conv.bias.detach().double()
        B = x.t.shape[0]
        worst = 0.0
        for b0, b1 in _chunks(B, max(x.t[0].numel(), 4 * w.shape[0] * Ho * Wo)):
            store = x.t[b0:b1].permute(0, 3, 1, 2).double()
            y, base = LO.icn_conv(store, x.border, pad, w, b, stride)
            del store
            if tanh_nchw is not None:
                ref, bound = LO.slot_ref(y, base, 2, 0.0)
                got = tanh_nchw[b0:b1]
            else:
                ref, bound = LO.slot_ref(y, base, 0, LO.unit(eng.tdtype))
                got = res[b0:b1].permute(0, 3, 1, 2)
            r = LO.worst(got, ref, bound)
            self.fail_if(*r, got, ref, bound, path, "tanh NCHW" if tanh_nchw is not None else "raw")
            worst = max(worst, r[0])
        self.mark(tanh_nchw if tanh_nchw is not None else res)
        self.lines[-1] = (path, self.lines[-1][1], worst)
        return res, Ho, Wo

    def icn_norm(self, orig, name, raw, H, W, kind, gamma=None, beta=None, residual=None, relu=True, up=1, border=1):
        torch = self.torch
        self.need(raw, name + ".norm", "input")
        if residual is not None:
            self.need(residual.t, name + ".norm", "residual")
        out = orig(name, raw, H, W, kind, gamma, beta, residual=residual, relu=relu, up=up, border=border)
        torch.cuda.synchronize()
        self.last = None
        u = LO.unit(self.eng.tdtype)
        worst = 0.0
        for b0, b1 in _chunks(raw.shape[0], 2 * out.t[0].numel()):
            r_in = raw[b0:b1].permute(0, 3, 1, 2).double()
            res = None
            if residual is not None:
                rb = residual.border
                res = residual.t[b0:b1, rb:rb + H, rb:rb + W].permute(0, 3, 1, 2).double()
            ref = LO.icn_norm(r_in, kind, gamma, beta, res, relu, up, border)
            bound = u * ref.abs() + LO.NORM_ABS
            got = out.t[b0:b1].permute(0, 3, 1, 2)
            r = LO.worst(got, ref, bound)
            self.fail_if(*r, got, ref, bound, name + ".norm", kind)
            worst = max(worst, r[0])
        self.lines.append((name + ".norm", kind, worst))
        self.mark(out.t)
        return out


@pytest.fixture
def walker(cuda, monkeypatch):
    """attach(engine, label, perturb=None) -> Walker; the wrappers are removed when the test ends."""
    return lambda eng, label, perturb=None: Walker(cuda, monkeypatch, eng, label, perturb)


# --------------------------------------------------------------------------- the walks
@pytest.mark.parametrize("B", [1, 5, 8, 64])
def test_vunet_walk(cuda, vnet, walker, B):
    """m(y, x) on the bf16 product path.  B = 5 leaves partly filled batch tiles at the coarse scales; B = 64 (the
    product batch) also runs the 128^2 layers on CTA pairs."""
    torch = cuda
    vnet.set_compute("bf16", "auto")
    w = walker(vnet.engine(), f"vunet bf16 B={B}")
    x, y = _vunet_inputs(torch, 11, B)
    torch.manual_seed(B)
    vnet(y, x)
    w.report()


def test_vunet_trajectory_walk(cuda, vnet, walker):
    """The trajectory form: encode_vehicles on V = 8 vehicles, then per item (B = 64) dec_up and dec_down(..., enc_gk=)
    with each item's vehicle rows gathered by torch indexing."""
    torch = cuda
    vnet.set_compute("bf16", "auto")
    eng = vnet.engine()
    w = walker(eng, "trajectory V=8 B=64")
    x, y = _vunet_inputs(torch, 3, 64)
    torch.manual_seed(8)
    with torch.no_grad():
        gk = eng.encode_vehicles(x[:8].contiguous())
        idx = (torch.arange(64, device="cuda") * 5) % 8
        gk_b = []
        for t in gk:
            w.need(t, "encode_vehicles", "gk")
            tb = t[idx]
            w.mark(tb)                    # rows of checked tensors, copied by torch
            gk_b.append(tb)
        od, sk = eng.dec_up(y, raw_skips=False)
        eng.dec_down(od, sk, enc_gk=[gk_b[:3], gk_b[3:]])
    w.report()


def test_vunet_g_from_api_walk(cuda, vnet, walker):
    """dec_down with enc_g converted from foreign API tensors (clones carry no engine tag: g_from_api re-derives
    ELU(SpaceToDepth(mu)) through from_nchw)."""
    torch = cuda
    vnet.set_compute("bf16", "auto")
    eng = vnet.engine()
    w = walker(eng, "dec_down g_from_api B=2")
    x, y = _vunet_inputs(torch, 5, 2)
    torch.manual_seed(4)
    oe, se = vnet.forward_enc_up(x)
    mu, _ = vnet.forward_enc_down(oe, se)
    with torch.no_grad():
        enc_g = [eng.g_from_api(t.clone()) for t in mu]
        od, sk = eng.dec_up(y)
        eng.dec_down(od, sk, enc_g)
    w.report()


def test_vunet_fp32_walk(cuda, vnet, walker):
    """The fp32 verification build (direct kernel): every slot within 2^-20 * A."""
    torch = cuda
    vnet.set_compute("fp32", "direct")
    try:
        w = walker(vnet.engine(), "vunet fp32 B=2")
        x, y = _vunet_inputs(torch, 2, 2)
        torch.manual_seed(2)
        vnet(y, x)
        w.report()
    finally:
        vnet.set_compute("bf16", "auto")


@pytest.mark.parametrize("dtype,B,res", [("fp16", 64, 256), ("fp16", 3, 64), ("bf16", 8, 256)])
def test_icn_walk(cuda, walker, dtype, B, res):
    """G_Resnet(21): every convolution and every norm pass (the whole bordered output of each)."""
    torch = cuda
    m = _icn(dtype)
    w = walker(m.engine(), f"icn {dtype} B={B} {res}")
    m(_icn_inputs(torch, 7, B, res))
    w.report()


# --------------------------------------------------------------------------- grid independence
def test_outputs_do_not_depend_on_the_sm_reserve(cuda, vnet):
    """A tile's accumulation order is fixed by the plan, not by the grid: reserve 5 leaves an odd grid for the CTA
    pairs, 141 takes the fallback to all SMs; VUNet and ICN outputs at B = 64 stay bit-identical."""
    torch = cuda
    from future_urban_scene_generation_b200 import _lib
    L = _lib.lib()
    vnet.set_compute("bf16", "auto")
    icn = _icn("fp16")
    x, y = _vunet_inputs(torch, 21, 64)
    xi = _icn_inputs(torch, 9, 64, 256)
    prev = L.fusg_conv2d_set_sm_reserve(-1)
    got = {}
    try:
        for r in (0, 4, 5, 141):
            L.fusg_conv2d_set_sm_reserve(r)
            torch.manual_seed(6)
            img, mu_a, mu_s = vnet(y, x)
            got[r] = [t.clone() for t in [img] + mu_a + mu_s] + [icn(xi).clone()]
            torch.cuda.synchronize()
    finally:
        L.fusg_conv2d_set_sm_reserve(prev)
    for r in (4, 5, 141):
        for i, (a, b) in enumerate(zip(got[0], got[r])):
            assert torch.equal(a, b), f"SM reserve {r}: output {i} differs from reserve 0 (max {(a - b).abs().max().item():.3g})"


# --------------------------------------------------------------------------- the weight folds
def _ulps(torch, a, b):
    """Per-element distance in units in the last place between two bf16 tensors."""
    def key(t):
        i = t.contiguous().view(torch.int16).int()
        return torch.where(i < 0, -(i & 0x7fff), i)
    return (key(a) - key(b)).abs()


def test_weight_folds(cuda, vnet):
    """fusg_fold_weightnorm, fusg_fold_weightnorm_paired (with the pair-shift taps) and the fused NiN + residual block
    against their layouts re-derived in numpy from the fp64 fold: at most 1 ulp per weight, and only where the fp64
    value sits at a rounding midpoint; zero_kblocks marks exactly the all-zero k-blocks."""
    torch = cuda
    from future_urban_scene_generation_b200.vunet.engine import FUSED_NIN
    vnet.set_compute("bf16", "auto")
    eng = vnet.engine()
    n_paired = n_diff = 0
    w64 = {p: LO.fold(c.weight_v, c.weight_g).cpu() for p, c in vnet.convs.items()}

    def compare(name, got, want64):
        nonlocal n_diff
        want = torch.from_numpy(want64).to(torch.bfloat16)
        _, step = LO.rounded(torch.from_numpy(want64), torch.bfloat16)
        d = _ulps(torch, got.cpu(), want)
        assert d.shape == want.shape and int(d.max()) <= 1, f"{name}: {int(d.max())} ulp"
        amb = step > 0 if step is not None else torch.zeros_like(d, dtype=torch.bool)
        assert not bool(((d > 0) & ~amb).any()), f"{name}: a weight away from any rounding midpoint differs"
        n_diff += int((d > 0).sum())

    for path, conv in vnet.convs.items():
        w, bias, cout, cout_pad, cin_pad, k = eng._w[path]
        compare(path, w, LO.pack_plain(w64[path].numpy(), cout_pad, cin_pad))
        assert torch.equal(bias[:cout].cpu(), conv.bias.detach().float().cpu()) and not bool(bias[cout:].any())
        if path in eng._wp:
            wp, bp, cout2, cp2, _, _ = eng._wp[path]
            want, want_b = LO.pack_paired(w64[path].numpy(), conv.bias.detach().double().cpu().numpy(), 32, conv.cin - 32, cp2)
            compare(path + " (paired)", wp, want)
            assert torch.equal(bp.cpu(), torch.from_numpy(want_b).float())
            n_paired += 1
    nin_p, res_p = FUSED_NIN
    wc, bsum, cout, cout_pad, cin_tot, k, zero = eng._wfused[res_p]
    want, want_zero = LO.pack_fused(w64[res_p].numpy(), w64[nin_p].numpy(), eng._w[res_p][4], eng._w[nin_p][4], cout_pad)
    compare(res_p + " (fused)", wc, want)
    assert zero == want_zero == LO.zero_kblocks(wc.float().cpu().numpy())
    assert n_paired >= 10
    print(f"folds: {len(eng._w)} plain, {n_paired} paired, 1 fused; {n_diff} weights 1 ulp off (all at rounding midpoints)")


# --------------------------------------------------------------------------- the checker can fail
def _bump_4ulp(path, outs, rec):
    if path == "shape_encoder_3.residual_0.layers.2":
        import torch
        t = next(o.tensor for o in outs if o.elu == 0 and o.layout == 0)
        i = int(t.float().abs().argmax())           # the largest value: 4 ulp there is far outside u*|ref| + 2^-16*A
        t.view(torch.int16).view(-1)[i] += 4


def _zero_pair_column(path, outs, rec):
    if path == "shape_decoder_6.residual_0.layers.2":
        assert rec["W"] * 2 == outs[0].tensor.shape[2] and rec["c0"] == 64, "expected the pixel-pair packed launch"
        next(o.tensor for o in outs if o.elu == 0)[:, :, 0, :] = 0


def _swap_quadrants(path, outs, rec):
    if path == "shape_decoder_2.sampler_3.conv":
        from future_urban_scene_generation_b200.vunet.engine import D2S_BLOCK
        o = next(o for o in outs if o.mode == D2S_BLOCK and o.elu == 1)
        v = _nchw(o.tensor, o.layout)
        q0, q1 = LO.d2s_block(v, 0).clone(), LO.d2s_block(v, 1).clone()
        LO.d2s_block(v, 0).copy_(q1)
        LO.d2s_block(v, 1).copy_(q0)


@pytest.mark.parametrize("perturb,path", [(_bump_4ulp, "shape_encoder_3.residual_0.layers.2"),
                                          (_zero_pair_column, "shape_decoder_6.residual_0.layers.2"),
                                          (_swap_quadrants, "shape_decoder_2.sampler_3.conv")],
                         ids=["4ulp_mid_network", "pair_column0", "d2s_block_swap"])
def test_checker_catches_injected_faults(cuda, vnet, walker, perturb, path):
    """A fault injected into one launch's output after its kernel ran is reported, naming the layer."""
    torch = cuda
    vnet.set_compute("bf16", "auto")
    walker(vnet.engine(), "perturbed", perturb)
    x, y = _vunet_inputs(torch, 1, 1)
    torch.manual_seed(1)
    with pytest.raises(AssertionError) as ei:
        vnet(y, x)
    print(f"\n{ei.value}")
    assert path in str(ei.value)


# --------------------------------------------------------------------------- coverage
def test_walks_reached_every_plan_variant(cuda):
    """Must run after the walks above (file order).  Variants the product networks did not reach would be named here
    together with the tests/test_vunet_gpu.py CONV_CASES entry that covers them."""
    if not WALKS <= REACHED["walks"]:
        pytest.skip("needs every walk of this file in the same session")
    print(f"\nplan variants reached: {sorted(REACHED['variants'])}")
    missing = REQUIRED_VARIANTS - REACHED["variants"]
    assert not missing, f"not reached by the product networks: {sorted(missing)}"
