"""Drop-in `vunet.models` for the hot path: `Vunet_fix_res` with the reference's constructor,
methods, tensor conventions and checkpoint layout (reference: vunet/models.py:191-484,
run_test.py:82-87), executed by hand-written sm_100a kernels (libfusg.so) instead of torch ops.

Contract kept (SURVEY.md §8b):
  * `Vunet_fix_res(Namespace(up_mode, w_norm, drop_prob, vunet_256))` is an nn.Module; `.to()`,
    `.eval()`, `.load_state_dict(sd, strict=True)` with the reference's 336 keys
    `<path>.conv.{bias,weight_g,weight_v}` in the reference's order, `.state_dict()` round trip;
  * `forward_enc_up / forward_enc_down / forward_dec_up / forward_dec_down / forward` take and
    return NCHW fp32 tensors on the module's device with the reference's list structures
    (`forward_dec_down` pops `skips` empty, like models.py:416-457);
  * Sampler noise is `torch.randn` on the CPU default generator in the reference's order and shapes
    (vunet/layers.py:166), so `torch.manual_seed(s)` reproduces the reference's draw.
Only the configuration the reference ships (`run_test.py:82`: subpixel / w_norm / 256) has
kernels; any other configuration raises NotImplementedError.  There is no CPU path.
"""
import argparse
import math

import torch
import torch.nn as nn

from .engine import VunetEngine


class _WNConv(nn.Module):
    """Parameter holder matching `weight_norm(nn.Conv2d(..., bias=True), dim=0)`:
    registration order bias, weight_g, weight_v (vunet/layers.py:27-31)."""

    def __init__(self, cin, cout, k):
        super().__init__()
        self.cin, self.cout, self.k = cin, cout, k
        bound = 1.0 / math.sqrt(cin * k * k)
        v = (torch.rand(cout, cin, k, k) * 2 - 1) * bound          # nn.Conv2d's default uniform range
        self.bias = nn.Parameter((torch.rand(cout) * 2 - 1) * bound)
        self.weight_g = nn.Parameter(v.flatten(1).norm(dim=1).view(cout, 1, 1, 1).clone())   # weight_norm init: g = ||v||
        self.weight_v = nn.Parameter(v)


class _Scope(nn.Module):
    """Plain container; child names reproduce the reference's attribute paths."""


def _conv_table():
    """[(path, cout, cin, k)] in the reference's parameter registration order
    (vunet/models.py:208-331; AutoRegressiveBlock :27-51)."""
    t = []

    def res(p, cin, cout):
        t.append((p + ".layers.2", cout, cin, 3))

    def nin(p, cin, cout):
        t.append((p + ".layers.1", cout, cin, 1))

    def down(p, cin, cout):
        t.append((p + ".down.down", cout, cin, 3))
        res(p + ".residual_0", cout, cout)
        res(p + ".residual_1", cout, cout)

    def init(p, cin, cout):
        nin(p + ".nin", cin, cout)
        res(p + ".residual_0", cout, cout)
        res(p + ".residual_1", cout, cout)

    def up(p, cin, cmid, cout):
        res(p + ".residual_0", cin, cmid)
        res(p + ".residual_1", cin, cmid)
        t.append((p + ".up.depth4x", 4 * cout, cmid, 3))

    def ar(p):
        res(p + ".residual_init", 256, 128)
        t.append((p + ".sampler_0.conv", 128, 512, 3))
        res(p + ".residual_0", 1024, 512)
        t.append((p + ".sampler_1.conv", 128, 512, 3))
        res(p + ".residual_1", 1024, 512)
        t.append((p + ".sampler_2.conv", 128, 512, 3))
        res(p + ".residual_2", 1024, 512)
        t.append((p + ".sampler_3.conv", 128, 512, 3))
        for k in range(3):
            nin(f"{p}.nin_{k}", 128, 512)
        res(p + ".residual_s2d", 128, 128)

    # appearance encoder / decoder
    init("app_encoder_1", 6, 128)
    for n in ("1_a", "1_b", "1_c", "2", "3", "4"):
        down("app_encoder_" + n, 128, 128)
    nin("app_skip_3_c", 128, 128)
    nin("app_skip_4_c", 128, 128)
    t.append(("app_bottleneck", 128, 128, 1))
    res("app_decoder_1_a", 256, 128)
    t.append(("app_decoder_1_b.conv", 128, 128, 3))
    t.append(("app_decoder_1_c", 128, 256, 1))
    res("app_decoder_1_d", 256, 128)
    t.append(("app_decoder_1_e.depth4x", 512, 128, 3))
    res("app_decoder_2_a", 128, 128)
    t.append(("app_decoder_2_b.conv", 128, 128, 3))
    # shape encoder
    init("shape_encoder_1", 3, 32)
    down("shape_encoder_1_a", 32, 32)
    down("shape_encoder_2", 32, 64)
    down("shape_encoder_3", 64, 128)
    for n in ("4", "5", "6"):
        down("shape_encoder_" + n, 128, 128)
    for n, c in (("1", 32), ("1_a", 32), ("2", 64), ("3", 128), ("4", 128), ("5", 128), ("6", 128)):
        nin(f"shape_skip_{n}_b", c, c)
        nin(f"shape_skip_{n}_c", c, c)
    # shape decoder
    t.append(("shape_bottleneck", 128, 128, 1))
    for n in ("1", "2"):
        ar("shape_decoder_" + n)
        nin(f"shape_decoder_{n}_n", 256, 128)
        res(f"shape_decoder_{n}_o", 256, 128)
        t.append((f"shape_decoder_{n}_p.depth4x", 512, 128, 3))
    up("shape_decoder_3", 256, 128, 128)
    up("shape_decoder_4", 256, 128, 64)
    up("shape_decoder_5", 128, 64, 32)
    up("shape_decoder_5_a", 64, 32, 32)
    res("shape_decoder_6.residual_0", 64, 32)
    res("shape_decoder_6.residual_1", 64, 32)
    t.append(("shape_decoder_6.conv", 3, 32, 3))
    return t


class Vunet_fix_res(nn.Module):
    def __init__(self, args: argparse.Namespace, dtype: str = "bf16", impl: str = "auto"):
        """:param args: Namespace(up_mode, w_norm, drop_prob, vunet_256) as in run_test.py:82-83.
        dtype: 'bf16' (tcgen05 path) or 'fp32' (verification build on CUDA-core kernels)."""
        super().__init__()
        self.args = args
        self.w_norm = args.w_norm
        self.drop_prob = args.drop_prob
        self.up_mode = args.up_mode
        self.vunet_256 = args.vunet_256
        if not (self.up_mode == 'subpixel' and self.w_norm and self.vunet_256):
            raise NotImplementedError(
                "the B200 path implements the shipped configuration only "
                "(up_mode='subpixel', w_norm=True, vunet_256=True; run_test.py:82)")
        self.convs = {}
        for path, cout, cin, k in _conv_table():
            parts = (path + ".conv").split(".")
            scope = self
            for name in parts[:-1]:
                if name not in scope._modules:
                    scope.add_module(name, _Scope())
                scope = scope._modules[name]
            leaf = _WNConv(cin, cout, k)
            scope.add_module(parts[-1], leaf)
            self.convs[path] = leaf
        self._engines = {}
        self._dtype = dtype
        self._impl = impl

    # ------------------------------------------------------------------ engine access
    def engine(self) -> VunetEngine:
        key = (self._dtype, self._impl)
        if key not in self._engines:
            self._engines[key] = VunetEngine(self, self._dtype, self._impl)
        eng = self._engines[key]
        if self.training:
            raise NotImplementedError("Vunet_fix_res (B200): inference only -- call .eval() (Dropout2d must be inactive)")
        eng.prepare_weights()
        return eng

    def set_compute(self, dtype="bf16", impl="auto"):
        self._dtype, self._impl = dtype, impl
        return self

    def _dev_ctx(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            from .._lib import FusgError
            raise FusgError("Vunet_fix_res (B200): parameters are on %s; this path has no CPU fallback -- call .to('cuda')" % dev)
        return torch.cuda.device(dev)

    # ------------------------------------------------------------------ reference API
    def forward_enc_up(self, x):
        with torch.no_grad(), self._dev_ctx():
            e = self.engine()
            outputs, skips = e.enc_up(x)
            return [e.to_nchw(a) for a in outputs], [e.to_nchw(a) for a in skips]

    def forward_dec_up(self, x):
        with torch.no_grad(), self._dev_ctx():
            e = self.engine()
            outputs, skips = e.dec_up(x)
            return [e.to_nchw(a) for a in outputs], [e.to_nchw(a) for a in skips]

    def forward_enc_down(self, enc_up_outputs, skips):
        with torch.no_grad(), self._dev_ctx():
            e = self.engine()
            outs = [e.as_act(t) for t in enc_up_outputs]
            sk = [e.as_act(t, need_raw=False) for t in skips]
            mu, z = e.enc_down(outs, sk)
            return [e.to_nchw(a) for a in mu], [e.to_nchw(a) for a in z]

    def forward_dec_down(self, dec_up_outputs, skips, enc_down_mu=()):
        with torch.no_grad(), self._dev_ctx():
            e = self.engine()
            outs = [e.as_act(t) for t in dec_up_outputs]
            sk = [e.as_act(t, need_raw=False) for t in skips]
            g = [e.g_from_api(t) for t in enc_down_mu]
            x_tilde, mu, z = e.dec_down(outs, sk, g)
            del skips[:]                       # the reference pops the caller's list empty (models.py:416-457)
            return x_tilde, [e.to_nchw(a) for a in mu], [e.to_nchw(a) for a in z]

    def _side_stream(self):
        dev = torch.cuda.current_device()
        if getattr(self, "_side", None) is None or self._side[0] != dev:
            self._side = (dev, torch.cuda.Stream(dev))
        return self._side[1]

    def forward(self, y_tilde, x=None, mean_mode='mean_appearance'):
        if self.vunet_256:
            assert y_tilde.shape[-1] == 256
            if x is not None:
                assert x.shape[-1] == 256
        assert mean_mode in ['mean_appearance', 'mean_shape']
        with torch.no_grad(), self._dev_ctx():
            e = self.engine()
            # raw_skips=False: the fused path consumes the skips pre-activated only
            if mean_mode == 'mean_appearance':
                # the shape encoder (dec_up) does not depend on the appearance branch (enc_up -> enc_down):
                # run it on a forked stream so its layers fill the SMs the narrow appearance layers leave idle
                # (fork_branches = False keeps everything on the current stream, e.g. for per-launch timing)
                if getattr(self, "fork_branches", True):
                    cur = torch.cuda.current_stream()
                    side = self._side_stream()
                    side.wait_stream(cur)
                    with torch.cuda.stream(side):
                        out_d, skips_d = e.dec_up(y_tilde, raw_skips=False)
                    out_e, skips_e = e.enc_up(x)
                    mu_app, z_app = e.enc_down(out_e, skips_e)
                    cur.wait_stream(side)
                    # the shape-encoder activations were allocated on the side stream and are consumed on `cur`:
                    # tell the caching allocator, or another caller stream could be handed their blocks too early
                    for a in list(out_d) + list(skips_d):
                        e.record_stream(a, cur)
                else:
                    out_e, skips_e = e.enc_up(x)
                    mu_app, z_app = e.enc_down(out_e, skips_e)
                    out_d, skips_d = e.dec_up(y_tilde, raw_skips=False)
                x_tilde, mu_shape, _ = e.dec_down(out_d, skips_d, [z.aux["s2d_elu"] for z in z_app])
                return x_tilde, [e.to_nchw(a) for a in mu_app], [e.to_nchw(a) for a in mu_shape]
            out_d, skips_d = e.dec_up(y_tilde, raw_skips=False)
            x_tilde, _, _ = e.dec_down(out_d, skips_d)
            return x_tilde

    def __call__(self, *args, **kwargs):
        return super().__call__(*args, **kwargs)
