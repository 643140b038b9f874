"""fp64 reference of ONE engine launch (a VUNet or ICN convolution, an ICN norm pass) -- TEST INFRASTRUCTURE ONLY.

The whole-network oracles (vunet_oracle.py, icn_oracle.py) bound the product path at the final image, where a fault in
one layer can hide below the tolerance after a hundred launches.  This module restates a single launch from the layer's
meaning -- the module's parameters and the stored input values -- so tests/test_engine_launches_gpu.py can check every
launch of a forward on its own, per element:

  * VUNet weights are the weight_norm fold g*v/||v|| in fp64 (vunet_oracle._weight), rounded to the activation dtype;
    ICN weights are the module's, rounded the same way.  Nothing is taken from the engine's packed weights.
  * A launch computes y = sum of convolutions + biases (+ residual); a Sampler slot adds the noise: z = y + noise.
  * Each output slot applies its activation (ELU, tanh) and its placement (PLAIN, D2S, S2D, one D2S_BLOCK quadrant).

Bounds, per element, with y the fp64 pre-rounding value and A the same expression on absolute values:

  16-bit slot   |got - ref| <= u*|ref| + 2^-16*A + E       u = 2^-8 (bf16), 2^-10 (fp16)
  fp32 slot     |got - ref| <= 2^-16*A + E                 (2^-20*A in the fp32 verification build)
  norm pass     |got - ref| <= u*|ref| + 2^-14

2^-16*A covers fp32 accumulation order; it is ~1000x smaller than one missing tap or one missing 64-channel chunk.
E covers the one thing a correct kernel may legitimately do differently from this reference: the kernels fold
weight_norm in fp32, and a weight whose fp64 value lies within 2^-16 (relative) of a rounding midpoint of the 16-bit
type may round to either neighbour.  E = conv(|x|, step) with `step` the size of that rounding step at such weights and
zero elsewhere -- exactly the error one such weight can cause, and nothing more.

ELU slots get two more terms.  The kernels take ELU of the ROUNDED raw value (so the stored ELU copy equals ELU of the
stored raw copy, conv.cu epilogue16), which on the negative branch adds u*|y|*exp(y); and their ELU uses ex2.approx,
~2e-7 absolute (conv.cu elu1), hence ELU_ABS.

Only tests/ may import this module.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import vunet_oracle as VO

PLAIN, D2S, S2D, D2S_BLOCK = 0, 1, 2, 3
ACC16 = 2.0 ** -16          # accumulation-order term of the 16-bit builds
ACC32 = 2.0 ** -20          # ... of the fp32 verification build
NORM_ABS = 2.0 ** -14
ELU_ABS = 2.0 ** -21
AMBIGUOUS = 2.0 ** -16      # relative distance to a rounding midpoint below which an fp32 fold may round either way
ICN_EPS = 1e-5


def unit(dtype):
    """Unit roundoff of a stored slot of `dtype` (0 for fp32: the fp32 terms are carried by the accumulation term)."""
    return {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -10}.get(dtype, 0.0)


# ------------------------------------------------------------------ weights
def fold(weight_v, weight_g):
    """weight_norm(dim=0) in fp64: g * v / ||v|| (vunet_oracle._weight)."""
    return VO._weight({"l.conv.weight_v": weight_v.detach().double(), "l.conv.weight_g": weight_g.detach().double()}, "l")


def rounded(w64, dtype):
    """(w, step): `w64` rounded to `dtype`, back in fp64; `step` [same shape] is |other neighbour - w| where an fp32
    computation of w64 could round to the other neighbour (|w64 - midpoint| <= AMBIGUOUS*|w64|), else 0.  step is None
    when no weight is ambiguous or dtype is fp32."""
    w = w64.to(dtype).double()
    if dtype == torch.float32:
        return w, None
    lo = (w64 * (1 - AMBIGUOUS)).to(dtype).double()
    hi = (w64 * (1 + AMBIGUOUS)).to(dtype).double()
    step = (hi - lo).abs()
    return w, (step if bool(step.any()) else None)


# ------------------------------------------------------------------ one convolution launch
def conv_terms(terms, stride=1, extras=(), acc=ACC16):
    """(y, base): y = sum_i conv(x_i, w_i) + sum extras; base = acc*A + E, the part of every slot's bound that does not
    depend on its activation or dtype (A = the same sum on absolute values, E = sum_i conv(|x_i|, step_i)), computed
    as ONE convolution per term: conv(|x|, acc*|w| + step).
    terms: (x NCHW fp64, w fp64 [cout,cin,k,k], step or None, pad); extras: fp64 tensors broadcastable to y (the bias
    as [1,cout,1,1], the residual)."""
    y = base = None
    for x, w, step, pad in terms:
        wa = acc * w.abs() if step is None else acc * w.abs() + step
        t = F.conv2d(x, w, stride=stride, padding=pad)
        ta = F.conv2d(x.abs(), wa, stride=stride, padding=pad)
        y = t if y is None else y + t
        base = ta if base is None else base + ta
    for e in extras:
        y = y + e
        base = base + acc * e.abs()
    return y, base


def place(t, mode):
    """An NCHW launch value as the output slot stores it (fusg.h FUSG_OUT_*).  D2S_BLOCK returns `t` itself: the
    launch owns the quadrant `d2s_block(full, blk)` of the full [B, C, 2H, 2W] tensor."""
    if mode == D2S:
        return VO.depth_to_space(t)
    if mode == S2D:
        return VO.space_to_depth(t)
    return t


def d2s_block(full, blk):
    """The pixels of quadrant `blk` of a DepthToSpace'd channel concat (vunet/models.py:85-86), as a strided view."""
    return full[:, :, blk // 2::2, blk % 2::2]


def slot_ref(y, base, elu, u):
    """(ref, bound) of one output slot holding act(y): elu 0 raw, 1 ELU, 2 tanh; base from conv_terms; u = unit
    roundoff of the slot's dtype (0 for fp32 slots).  ELU and tanh have slopes <= 1, so base bounds them too."""
    bound = base
    if elu == 1:
        ref = F.elu(y)
        bound = bound + u * ref.abs() + u * y.abs() * torch.exp(torch.clamp(y, max=0.0)) + ELU_ABS
    elif elu == 2:
        ref = torch.tanh(y)
        bound = bound + u * ref.abs()
    else:
        ref = y
        bound = bound + u * ref.abs()
    return ref, bound


def worst(got, ref, bound):
    """(max |got - ref| / bound, flat index of it, all finite?) over matching tensors."""
    got = got.double()
    finite = bool(torch.isfinite(got).all())
    r = (got - ref).abs() / bound.clamp_min(1e-300)
    r = torch.where(torch.isfinite(got), r, torch.full_like(r, float("inf")))
    i = int(torch.argmax(r))
    return float(r.reshape(-1)[i]), i, finite


# ------------------------------------------------------------------ ICN launches
def icn_conv(store, border, pad, w, bias, stride, acc=ACC16):
    """One bordered (pad_mode 1) convolution: `store` NCHW fp64 [B, C, H+2*border, W+2*border] holds the image and its
    reflection border; the convolution reads [border-pad, border+H+pad) of it.  w fp64 [cout,cin,k,k] (cin real
    channels), bias fp64 [cout].  Returns (y, base) as conv_terms."""
    x = store[:, :w.shape[1]]
    if border > pad:
        x = x[:, :, border - pad:x.shape[2] - (border - pad), border - pad:x.shape[3] - (border - pad)]
    return conv_terms([(x, w, None, 0)], stride, [bias.view(1, -1, 1, 1)], acc)


def icn_norm(raw, kind, gamma=None, beta=None, residual=None, relu=True, up=1, border=1):
    """fusg_norm_apply's output from the stored raw conv output `raw` (NCHW fp64): InstanceNorm2d (biased variance,
    no affine) or the reference's LayerNorm (per sample, unbiased std, (x - mean)/(std + eps), then gamma / beta),
    + residual (NCHW fp64, the residual's interior), ReLU, nearest `up`x upsampling, reflection border."""
    if kind == "inst":
        mean = raw.mean(dim=(2, 3), keepdim=True)
        var = raw.var(dim=(2, 3), unbiased=False, keepdim=True)
        y = (raw - mean) / torch.sqrt(var + ICN_EPS)
    else:
        flat = raw.reshape(raw.shape[0], -1)
        mean = flat.mean(1).view(-1, 1, 1, 1)
        std = flat.std(1).view(-1, 1, 1, 1)
        y = (raw - mean) / (std + ICN_EPS)
        y = y * gamma.double().view(1, -1, 1, 1) + beta.double().view(1, -1, 1, 1)
    if residual is not None:
        y = y + residual
    if relu:
        y = F.relu(y)
    if up > 1:
        y = F.interpolate(y, scale_factor=up, mode="nearest")
    if border:
        y = F.pad(y, (border,) * 4, mode="reflect")
    return y


# ------------------------------------------------------------------ packed weight layouts, re-derived in numpy
def pack_plain(w, cout_pad, cin_pad):
    """fusg_fold_weightnorm's layout: [cout,cin,k,k] -> [cout_pad][k*k][cin_pad], zero padded."""
    cout, cin, k, _ = w.shape
    out = np.zeros((cout_pad, k * k, cin_pad), dtype=w.dtype)
    out[:cout, :, :cin] = w.transpose(0, 2, 3, 1).reshape(cout, k * k, cin)
    return out


def pack_paired(w, bias, c0, c1, cout_pad):
    """fusg_fold_weightnorm_paired's layout for a k x k (k = 1 or 3) layer c0(+c1) -> cout run on pixel pairs:
    output channel n' = dx*cout + co is pixel 2X+dx of pair X; K index = tap' * 2*(c0+c1) + [in0: h*c0 + ci |
    in1: 2*c0 + h*c1 + ci] for input half h; a 3x3 tap' = (ky, pair shift s+1) holds the original tap
    kx = 2s + h - dx + 1 when 0 <= kx < 3.  Returns (w [cout_pad][k*k][2*(c0+c1)], bias [cout_pad])."""
    cout, cin, k, _ = w.shape
    assert cin == c0 + c1
    kp = 2 * cin
    out = np.zeros((cout_pad, k * k, kp), dtype=w.dtype)
    bout = np.zeros((cout_pad,), dtype=bias.dtype)
    for dx in range(2):
        bout[dx * cout:(dx + 1) * cout] = bias
        for h in range(2):
            kin = [h * c0 + np.arange(c0)] + ([2 * c0 + h * c1 + np.arange(c1)] if c1 else [])
            kin = np.concatenate(kin)
            rows = slice(dx * cout, (dx + 1) * cout)
            if k == 1:
                if h == dx:
                    out[rows, 0, kin] = w[:, :, 0, 0]
                continue
            for ky in range(3):
                for s in (-1, 0, 1):
                    kx = 2 * s + h - dx + 1
                    if 0 <= kx < 3:
                        out[rows, ky * 3 + s + 1, kin] = w[:, :, ky, kx]
    return out, bout


def pair_view_weight(wp, cout2):
    """A pair-packed weight [cout_pad][k*k][2cin] as a conv2d weight [cout2, 2cin, k, k] over the pair view
    [B, 2cin, H, W/2] of an NCHW activation (channel h*c + ci <-> pixel 2X+h, channel ci)."""
    taps, kp = wp.shape[1], wp.shape[2]
    k = int(round(taps ** 0.5))
    return wp[:cout2].reshape(cout2, k, k, kp).transpose(0, 3, 1, 2)


def pack_fused(w_res, w_nin, cin_res_pad, cin_nin_pad, cout_pad):
    """Weights of the NiN folded into the following residual (vunet/engine.py prepare_weights): the 3x3 residual over
    the first cin_res_pad channels, the 1x1 NiN at the centre tap over the next cin_nin_pad.
    Returns (w [cout_pad][9][cin_res_pad + cin_nin_pad], zero_kblocks bitmask of the all-zero 64-channel k-blocks)."""
    out = np.zeros((cout_pad, 9, cin_res_pad + cin_nin_pad), dtype=w_res.dtype)
    out[:, :, :cin_res_pad] = pack_plain(w_res, cout_pad, cin_res_pad)
    out[:, 4, cin_res_pad:] = pack_plain(w_nin, cout_pad, cin_nin_pad)[:, 0, :]
    return out, zero_kblocks(out)


def zero_kblocks(wpacked, kc=64):
    """fusg_conv_desc.zero_kblocks of a packed weight: bit (tap * chunks + chunk) set iff that k-block is all zero."""
    taps, ktot = wpacked.shape[1], wpacked.shape[2]
    chunks = ktot // kc
    mask = 0
    for tap in range(taps):
        for c in range(chunks):
            if not np.any(wpacked[:, tap, c * kc:(c + 1) * kc]):
                mask |= 1 << (tap * chunks + c)
    return mask
