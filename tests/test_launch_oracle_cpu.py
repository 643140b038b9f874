"""oracle/launch_oracle.py, the per-launch fp64 reference of tests/test_engine_launches_gpu.py, checked against the
whole-network oracles' layer primitives in fp64: chaining its launch references must reproduce vunet_oracle.residual,
the fused NiN + residual launch, ar_block's D2S_BLOCK placement, icn_oracle.conv_block and the ResBlock / upsample
steps of the ICN; and its packed weight layouts must compute the same convolution as the logical weights."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import icn_oracle as IO
from oracle import launch_oracle as LO
from oracle import vunet_oracle as VO


@pytest.fixture(scope="module")
def vsd():
    return {k: v.double() for k, v in VO.make_state_dict(0).items()}


def _w(sd, path):
    return LO.fold(sd[path + ".conv.weight_v"], sd[path + ".conv.weight_g"])


def _b(sd, path):
    return sd[path + ".conv.bias"].view(1, -1, 1, 1)


def _close(a, b, tol=1e-12):
    assert a.shape == b.shape
    assert (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item())


def test_residual_with_skip(vsd):
    g = torch.Generator().manual_seed(0)
    x, skip = torch.randn(2, 32, 8, 8, generator=g).double(), torch.randn(2, 32, 8, 8, generator=g).double()
    path = "shape_decoder_6.residual_0"
    want = VO.residual(vsd, path, x, skip)
    p = path + ".layers.2"
    y, base = LO.conv_terms([(F.elu(torch.cat([x, skip], 1)), _w(vsd, p), None, 1)], 1, [_b(vsd, p), x], acc=1.0)
    _close(y, want)
    assert bool((base >= y.abs() - 1e-12).all())               # with acc = 1, base is A itself


def test_fused_nin_residual_launch(vsd):
    """The engine's fused launch: conv3x3(ELU(x0)) + conv1x1(ELU(in)) with both biases == residual(NiN(in))."""
    g = torch.Generator().manual_seed(1)
    xin = torch.randn(2, 6, 8, 8, generator=g).double()
    nin_p, res_p = "app_encoder_1.nin.layers.1", "app_encoder_1.residual_0.layers.2"
    x0 = VO.nin(vsd, "app_encoder_1.nin", xin)
    want = VO.residual(vsd, "app_encoder_1.residual_0", x0)
    y, _ = LO.conv_terms([(F.elu(x0), _w(vsd, res_p), None, 1), (F.elu(xin), _w(vsd, nin_p), None, 0)], 1,
                            [_b(vsd, res_p), _b(vsd, nin_p)])
    _close(y, want)


def test_ar_block_placement(vsd):
    """Four Sampler launches, each placed as its D2S_BLOCK quadrant, and the S2D residual output rebuild ar_block."""
    g = torch.Generator().manual_seed(2)
    path = "shape_decoder_1"
    x, skip_a = torch.randn(1, 128, 4, 4, generator=g).double(), torch.randn(1, 128, 4, 4, generator=g).double()
    torch.manual_seed(5)
    want_x, want_mu, want_z = VO.ar_block(vsd, path, x, skip_a)
    # the launches in the engine's order, with the noise drawn in the reference's order
    torch.manual_seed(5)
    p = path + ".residual_init.layers.2"
    xi, _ = LO.conv_terms([(F.elu(torch.cat([x, skip_a], 1)), _w(vsd, p), None, 1)], 1, [_b(vsd, p), x])
    _close(xi, want_x)
    p = path + ".residual_s2d.layers.2"
    xs, _ = LO.conv_terms([(F.elu(xi), _w(vsd, p), None, 1)], 1, [_b(vsd, p), xi])
    x_ = LO.place(xs, LO.S2D)
    mu = torch.full((1, 128, 4, 4), float("nan"), dtype=torch.float64)
    z = mu.clone()
    for k in range(4):
        p = f"{path}.sampler_{k}.conv"
        y, _ = LO.conv_terms([(x_, _w(vsd, p), None, 1)], 1, [_b(vsd, p)])
        eps = torch.randn(*y.shape).double()
        LO.d2s_block(mu, k).copy_(LO.place(y, LO.D2S_BLOCK))
        LO.d2s_block(z, k).copy_(LO.place(y + eps, LO.D2S_BLOCK))
        if k < 3:
            p = f"{path}.nin_{k}.layers.1"
            gk, _ = LO.conv_terms([(F.elu(y + eps), _w(vsd, p), None, 0)], 1, [_b(vsd, p)])
            p = f"{path}.residual_{k}.layers.2"
            x_, _ = LO.conv_terms([(F.elu(torch.cat([x_, gk], 1)), _w(vsd, p), None, 1)], 1, [_b(vsd, p), x_])
    _close(mu, want_mu)
    _close(z, want_z)


def test_upsample_d2s(vsd):
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 128, 4, 4, generator=g).double()
    p = "shape_decoder_3.up.depth4x"
    y, _ = LO.conv_terms([(x, _w(vsd, p), None, 1)], 1, [_b(vsd, p)])
    _close(LO.place(y, LO.D2S), VO.upsample(vsd, "shape_decoder_3.up", x))


def _icn_sd(cout, cin, k, ln, seed):
    g = torch.Generator().manual_seed(seed)
    sd = {"p.conv.weight": (torch.rand(cout, cin, k, k, generator=g) * 2 - 1).double() / (cin * k * k) ** 0.5,
          "p.conv.bias": (torch.rand(cout, generator=g) * 2 - 1).double() * 0.1}
    if ln:
        sd["p.norm.gamma"] = torch.rand(cout, generator=g).double()
        sd["p.norm.beta"] = (torch.rand(cout, generator=g).double() - 0.5) * 0.2
    return sd


@pytest.mark.parametrize("k,stride,pad,border,kind,act", [(7, 1, 3, 3, "inst", "relu"), (4, 2, 1, 1, "inst", "relu"),
                                                          (3, 1, 1, 2, "inst", "none"), (5, 1, 2, 2, "ln", "relu")])
def test_icn_conv_block(k, stride, pad, border, kind, act):
    """Stored reflection border (border >= pad) -> bordered conv -> norm pass == icn_oracle.conv_block."""
    g = torch.Generator().manual_seed(k)
    x = torch.randn(2, 8, 16, 16, generator=g).double()
    sd = _icn_sd(12, 8, k, kind == "ln", k)
    want = IO.conv_block(sd, "p", x, stride, pad, kind, act)
    store = F.pad(x, (border,) * 4, mode="reflect")
    y, _ = LO.icn_conv(store, border, pad, sd["p.conv.weight"], sd["p.conv.bias"], stride)
    got = LO.icn_norm(y, kind, sd.get("p.norm.gamma"), sd.get("p.norm.beta"), relu=act == "relu", up=1, border=0)
    _close(got, want)
    # the output is written with the next layer's border, which is the reflection of the interior
    got_b = LO.icn_norm(y, kind, sd.get("p.norm.gamma"), sd.get("p.norm.beta"), relu=act == "relu", up=1, border=2)
    _close(got_b, F.pad(want, (2,) * 4, mode="reflect"))


def test_icn_resblock_and_upsample():
    """ResBlock: norm(conv(h)) + x with the residual interior; Decoder: upsample folded into the norm pass of the
    previous block, then the 5x5 LayerNorm block."""
    g = torch.Generator().manual_seed(9)
    x = torch.randn(1, 8, 8, 8, generator=g).double()
    s0, s1 = _icn_sd(8, 8, 3, False, 1), _icn_sd(8, 8, 3, False, 2)
    sd = {"r.model.0.model.0" + k[1:]: v for k, v in s0.items()}
    sd.update({"r.model.0.model.1" + k[1:]: v for k, v in s1.items()})
    want = IO.res_blocks(sd, "r", x, n_res=1)
    store = F.pad(x, (1,) * 4, mode="reflect")
    y, _ = LO.icn_conv(store, 1, 1, s0["p.conv.weight"], s0["p.conv.bias"], 1)
    h = LO.icn_norm(y, "inst", relu=True, border=1)
    y, _ = LO.icn_conv(h, 1, 1, s1["p.conv.weight"], s1["p.conv.bias"], 1)
    out = LO.icn_norm(y, "inst", residual=store[:, :, 1:-1, 1:-1], relu=False, up=2, border=2)
    _close(out, F.pad(F.interpolate(want, scale_factor=2, mode="nearest"), (2,) * 4, mode="reflect"))
    s2 = _icn_sd(4, 8, 5, True, 3)
    y, _ = LO.icn_conv(out, 2, 2, s2["p.conv.weight"], s2["p.conv.bias"], 1)
    got = LO.icn_norm(y, "ln", s2["p.norm.gamma"], s2["p.norm.beta"], relu=True, border=0)
    _close(got, IO.conv_block(s2, "p", F.interpolate(want, scale_factor=2, mode="nearest"), 1, 2, "ln", "relu"))


def test_rounded_marks_only_midpoint_weights():
    w = torch.tensor([1.0, 1.0 + 2.0 ** -8, 1.0 + 2.0 ** -8 + 2.0 ** -20, 1.0 + 2.0 ** -9, -(1.0 + 2.0 ** -8)], dtype=torch.float64)
    r, step = LO.rounded(w, torch.bfloat16)
    assert r.tolist()[0] == 1.0 and r.tolist()[3] == 1.0
    assert step.tolist() == [0.0, 2.0 ** -7, 2.0 ** -7, 0.0, 2.0 ** -7]
    assert LO.rounded(w, torch.float32)[1] is None


@pytest.mark.parametrize("cins,cout,k", [((32,), 32, 3), ((32, 32), 32, 3), ((32,), 32, 1), ((32,), 3, 3)])
def test_paired_layout_is_the_same_convolution(cins, cout, k):
    """pack_paired: a conv over W/2 pixel pairs (the NHWC bytes viewed as 2c channels) with the packed weights equals
    the logical conv over W pixels, output channel dx*cout + co being pixel 2X+dx."""
    g = torch.Generator().manual_seed(sum(cins) + cout + k)
    B, H, W = 2, 6, 8
    xs = [torch.randn(B, c, H, W, generator=g).double() for c in cins]
    w = torch.randn(cout, sum(cins), k, k, generator=g).double()
    b = torch.randn(cout, generator=g).double()
    want = F.conv2d(torch.cat(xs, 1), w, b, padding=k // 2)
    cp2 = (2 * cout + 15) // 16 * 16
    wp, bp = LO.pack_paired(w.numpy(), b.numpy(), cins[0], sum(cins) - cins[0], cp2)
    assert not wp[2 * cout:].any() and not bp[2 * cout:].any()

    def pairs(x):          # NCHW [B,c,H,W] -> [B, 2c, H, W/2], channel h*c + ci = pixel 2X+h
        c = x.shape[1]
        return x.view(B, c, H, W // 2, 2).permute(0, 4, 1, 2, 3).reshape(B, 2 * c, H, W // 2)
    wv = torch.from_numpy(LO.pair_view_weight(wp, 2 * cout).copy())
    got = F.conv2d(torch.cat([pairs(x) for x in xs], 1), wv, torch.from_numpy(bp[:2 * cout]), padding=(k // 2, k // 2))
    got = got.view(B, 2, cout, H, W // 2).permute(0, 2, 3, 4, 1).reshape(B, cout, H, W)
    _close(got, want)


def test_fused_layout_and_zero_kblocks():
    g = torch.Generator().manual_seed(4)
    w_res, w_nin = torch.randn(128, 128, 3, 3, generator=g).double(), torch.randn(128, 6, 1, 1, generator=g).double()
    wc, mask = LO.pack_fused(w_res.numpy(), w_nin.numpy(), 128, 64, 128)
    assert wc.shape == (128, 9, 192)
    want = sum(1 << (tap * 3 + 2) for tap in range(9) if tap != 4)
    assert mask == want
    # as a convolution: the packed block over [x | x_nin] is the 3x3 residual plus the 1x1 NiN
    x, xn = torch.randn(1, 128, 5, 5, generator=g).double(), torch.randn(1, 6, 5, 5, generator=g).double()
    xn64 = torch.cat([xn, torch.zeros(1, 58, 5, 5, dtype=torch.float64)], 1)
    wv = torch.from_numpy(wc.reshape(128, 3, 3, 192).transpose(0, 3, 1, 2).copy())
    _close(F.conv2d(torch.cat([x, xn64], 1), wv, padding=1), F.conv2d(x, w_res, padding=1) + F.conv2d(xn, w_nin))
