"""CPU restatement of `torch.randn(b, c, h, w)` on torch's CPU generator, for contiguous fp32 draws whose numel is a
multiple of 16 (test infrastructure: what csrc/noise.cu must reproduce bit for bit).

The pieces, from the headers that ship with torch (torch/include/ATen/...):
  - the generator state: `get_state()` is 5056 bytes; u64 seed at 0, i32 `left` at 8, i32 `seeded` at 12, u64 `next` at
    16, the 624 MT19937 words as u64 from 24, then the cached normal samples (untouched by these draws);
  - core/MT19937RNGEngine.h: each word decrements `left`, twists the whole state when it reaches 0 (left = 624, next = 0),
    then returns state[next++] tempered;
  - core/TransformationHelper.h: one word per uniform, (w & 0xFFFFFF) * 2^-24 in float (exact);
  - native/cpu/DistributionTemplates.h `normal_fill_AVX2`: all uniforms first, then per 16-element chunk Box-Muller on
    elements j and j+8 (u1 = 1 - u[j], u2 = u[j+8]), with log256_ps / sincos256_ps of native/cpu/avx_mathfun.h;
  - libtorch_cpu contracts mul + add pairs of those functions into FMA (GCC's -ffp-contract=fast; DESIGN.md §4.8 lists
    which pairs).  `_fma` below is a correctly rounded fp32 FMA; every other operation is one rounded numpy fp32 op.
"""
import numpy as np

N = 624
M = 397
MATRIX_A = np.uint32(0x9908B0DF)
STATE_BYTES = 5056


# ---------------------------------------------------------------------------------------------------------------- state
def parse_state(state):
    """5056-byte generator state (torch ByteTensor or bytes) -> (words u32[624], left, next)."""
    b = bytes(state.numpy().tobytes() if hasattr(state, "numpy") else state)
    if len(b) != STATE_BYTES:
        raise ValueError(f"generator state is {len(b)} bytes, expected {STATE_BYTES}")
    left, _seeded = np.frombuffer(b, np.int32, 2, 8)
    nxt = int(np.frombuffer(b, np.uint64, 1, 16)[0])
    words = np.frombuffer(b, np.uint64, N, 24).astype(np.uint32)
    return words, int(left), nxt


def build_state(template, words, left, nxt):
    """The state `template` with its MT19937 words and position replaced (seed, `seeded` and the cached normal samples
    kept) -> torch uint8 tensor for Generator.set_state."""
    import torch
    b = bytearray(template.numpy().tobytes() if hasattr(template, "numpy") else template)
    b[8:12] = np.int32(left).tobytes()
    b[16:24] = np.uint64(nxt).tobytes()
    b[24:24 + 8 * N] = np.asarray(words, np.uint32).astype(np.uint64).tobytes()
    return torch.frombuffer(b, dtype=torch.uint8).clone()


# ---------------------------------------------------------------------------------------------------------------- MT19937
def _twist(u, v):
    mix = (u & np.uint32(0x80000000)) | (v & np.uint32(0x7FFFFFFF))
    return (mix >> np.uint32(1)) ^ np.where(v & np.uint32(1), MATRIX_A, np.uint32(0))


def next_state(st):
    """MT19937RNGEngine::next_state, vectorised in the pieces its in-place loop allows."""
    st = np.asarray(st, np.uint32)
    new = st.copy()
    new[:227] = st[M:N] ^ _twist(st[:227], st[1:228])
    new[227:454] = new[0:227] ^ _twist(st[227:454], st[228:455])
    new[454:623] = new[227:396] ^ _twist(st[454:623], st[455:624])
    new[623] = new[396] ^ _twist(st[623:624], new[0:1])[0]
    return new


def raw_words(words, left, nxt, n):
    """The next n untempered words from (words, left, next) and the position after them: (raw u32[n], words, left, next)."""
    if not (0 < left <= N and 0 <= nxt and nxt + left - 1 <= N):
        raise ValueError(f"MT19937 position left={left} next={nxt} is not one torch's generator reaches")
    out = np.empty(n, np.uint32)
    k = min(n, left - 1)
    out[:k] = words[nxt:nxt + k]
    left, nxt = left - k, nxt + k
    while k < n:
        words = next_state(words)
        t = min(N, n - k)
        out[k:k + t] = words[:t]
        k += t
        left, nxt = N - t + 1, t
    return out, np.asarray(words, np.uint32), left, nxt


def advance(words, left, nxt, n):
    """State after n words (twists only): (words, left, next)."""
    return raw_words(words, left, nxt, n)[1:]


def temper(y):
    y = y ^ (y >> np.uint32(11))
    y = y ^ ((y << np.uint32(7)) & np.uint32(0x9D2C5680))
    y = y ^ ((y << np.uint32(15)) & np.uint32(0xEFC60000))
    return y ^ (y >> np.uint32(18))


def uniforms(raw):
    return ((temper(raw) & np.uint32(0xFFFFFF)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------- transform
F = np.float32


def _fma(a, b, c):
    """fp32 a*b + c rounded once.  The product is exact in fp64; the fp64 sum is exact up to `err` (TwoSum), and its
    rounding to fp32 is wrong only when the sum sits exactly halfway between two floats and err is non-zero."""
    a64, b64, c64 = (np.asarray(t, F).astype(np.float64) for t in (a, b, c))
    p = a64 * b64
    s = p + c64
    bb = s - p
    err = (p - (s - bb)) + (c64 - bb)
    r = s.astype(F)
    r64 = r.astype(np.float64)
    toward = np.where(s > r64, F(np.inf), F(-np.inf))
    other = np.nextafter(r, toward)
    tie = (s != r64) & (np.abs(s - r64) == np.abs(other.astype(np.float64) - s))
    fix = tie & (err != 0) & (np.sign(err) == np.sign(s - r64))
    return np.where(fix, other, r).astype(F)


def _bits(x):
    return np.asarray(x, F).view(np.uint32)


def _float(u):
    return np.asarray(u, np.uint32).view(F)


LOG_P = [F(v) for v in (7.0376836292E-2, -1.1514610310E-1, 1.1676998740E-1, -1.2420140846E-1, 1.4249322787E-1,
                        -1.6668057665E-1, 2.0000714765E-1, -2.4999993993E-1, 3.3333331174E-1)]
LOG_Q1, LOG_Q2, SQRTHF = F(-2.12194440e-4), F(0.693359375), F(0.707106781186547524)
DP = [F(-0.78515625), F(-2.4187564849853515625e-4), F(-3.77489497744594108e-8)]
SINCOF = [F(-1.9515295891E-4), F(8.3321608736E-3), F(-1.6666654611E-1)]
COSCOF = [F(2.443315711809948E-005), F(-1.388731625493765E-003), F(4.166664568298827E-002)]
FOPI = F(1.27323954473516)
TWO_PI = F(2.0 * np.pi)           # 2.0f * c10::pi<double>, a double, rounded by _mm256_set1_ps


def log256(x):
    """log256_ps for x in (0, 1] (what 1 - u reaches)."""
    x = np.maximum(np.asarray(x, F), _float(0x00800000))
    e = ((_bits(x) >> np.uint32(23)).astype(np.int32) - 127).astype(F) + F(1)
    x = _float((_bits(x) & np.uint32(~0x7F800000 & 0xFFFFFFFF)) | _bits(F(0.5)))
    mask = x < SQRTHF
    tmp = np.where(mask, x, F(0))
    x = x - F(1)
    e = e - np.where(mask, F(1), F(0))
    x = x + tmp
    z = x * x
    y = np.full_like(x, LOG_P[0])
    for p in LOG_P[1:]:
        y = _fma(y, x, p)
    y = y * x
    y = _fma(y, z, e * LOG_Q1)
    y = _fma(-z, F(0.5), y)
    x = x + y
    return _fma(e, LOG_Q2, x)


def sincos256(x):
    """sincos256_ps for x >= 0 (theta = 2 pi u2): (sin, cos)."""
    x = np.abs(np.asarray(x, F))
    j = (x * FOPI).astype(np.int32)               # cvttps: x >= 0, so truncation
    j = (j + 1) & ~1
    y = j.astype(F)
    swap_sin = ((j & 4) << 29).astype(np.uint32)
    poly = (j & 2) == 0
    for d in DP:
        x = _fma(y, d, x)
    sign_cos = ((~(j - 2) & 4) << 29).astype(np.uint32)
    z = x * x
    c = np.full_like(x, COSCOF[0])
    c = _fma(c, z, COSCOF[1])
    c = _fma(c, z, COSCOF[2])
    c = c * z
    c = _fma(c, z, -(z * F(0.5)))
    c = c + F(1)
    s = np.full_like(x, SINCOF[0])
    s = _fma(s, z, SINCOF[1])
    s = _fma(s, z, SINCOF[2])
    s = s * z
    s = _fma(s, x, x)
    ysin2 = np.where(poly, s, F(0))
    ysin1 = np.where(poly, F(0), c)
    sin = ysin1 + ysin2
    cos = (c - ysin1) + (s - ysin2)
    return _float(_bits(sin) ^ swap_sin), _float(_bits(cos) ^ sign_cos)


def box_muller(u):
    """normal_fill_16_AVX2 over a flat fp32 array of uniforms (length a multiple of 16), mean 0 and std 1."""
    u = np.asarray(u, F).reshape(-1, 2, 8)
    u1, u2 = F(1) - u[:, 0], u[:, 1]
    radius = np.sqrt(log256(u1) * F(-2))
    sin, cos = sincos256(TWO_PI * u2)
    out = np.empty_like(u)
    out[:, 0] = radius * cos + F(0)                # _mm256_fmadd_ps(n, 1, 0): n + 0, so -0 becomes +0
    out[:, 1] = radius * sin + F(0)
    return out.reshape(-1)


# ---------------------------------------------------------------------------------------------------------------- draws
def check_shapes(shapes):
    shapes = [tuple(int(d) for d in s) for s in shapes]
    for s in shapes:
        n = int(np.prod(s)) if s else 1
        if n < 16 or n % 16:
            raise ValueError(f"draw of shape {s}: numel {n} is not a positive multiple of 16 (torch takes another path)")
    return shapes


def randn(shapes, state):
    """torch.randn(*shape) for each shape in turn, on a generator in `state` -> (list of fp32 NCHW arrays, new state)."""
    shapes = check_shapes(shapes)
    words, left, nxt = parse_state(state)
    outs = []
    for s in shapes:
        n = int(np.prod(s))
        raw, words, left, nxt = raw_words(words, left, nxt, n)
        outs.append(box_muller(uniforms(raw)).reshape(s))
    return outs, build_state(state, words, left, nxt)
